"""The kNN partition building blocks, the statistics and the outlier threshold against the plain reference of
tests/knn_reference.py, bit for bit.

These entry points are what a partitioned outlier removal is made of (csrc/slab.cpp, cwipc_util_b200/slab.py): the
queries of one part against its points and halo, the open queries, the lists other parts answer them with, the merge,
the all-reduced sums and the threshold.  Every distance here is exact float32 arithmetic and every sum has a fixed
order, so the results are compared exactly, and the keep decisions against the threshold of the exact sums, within the
rounding error those fixed-order sums can have (about 1e-13 relative).
"""
import gc
import os
import sys

import numpy as np
import pytest

from cwipc_util_b200 import synthetic

import knn_reference as ref

pytestmark = pytest.mark.gpu

DT = synthetic.cwipc_point_numpy_dtype
TESTS = os.path.dirname(os.path.abspath(__file__))
REPO = os.path.dirname(TESTS)

QUERY_KS = [1, 7, 30, 63, 64, 200, 511]
LIST_KS = [31, 32, 63, 64, 127, 128, 255, 256, 511]   # both sides of each list width of knn_list_kernel (1/2/4/8/16 per lane)


@pytest.fixture(autouse=True)
def no_leaks(cw):
    gc.collect()
    base = cw.cwipc_dangling_allocations(False)
    yield
    gc.collect()
    assert cw.cwipc_dangling_allocations(False) == base


def shuffled(pts, seed):
    """Random order: the queries (the first nquery points) and the halo (the rest) are mixed in space."""
    return pts[np.random.default_rng(seed).permutation(len(pts))]


def shifted(pts, by):
    out = pts.copy()
    for a in "xyz":
        out[a] = (pts[a].astype(np.float64) + by).astype(np.float32)
    return out


def volume_cloud():
    """A random volume with 200 copies of one point and three far outliers."""
    rng = np.random.default_rng(8)
    n = 30000
    pts = np.zeros(n, DT)
    for a in "xyz":
        pts[a] = rng.uniform(-0.3, 0.3, n).astype(np.float32)
    pts["tile"] = rng.choice(np.array([1, 2, 4, 8], np.uint8), n)
    pts[:200] = pts[0]
    pts["x"][-1], pts["y"][-2], pts["z"][-3] = 55.0, -70.0, 1000.0
    return shuffled(pts, 8)


CLOUDS = ["camera", "volume", "shifted", "ds_tf"]


def make_cloud(cw, name):
    """(device cloud, its points) for one of CLOUDS."""
    if name == "camera":
        pts = shuffled(synthetic.camera_cloud(40000, seed=41), 41)
    elif name == "volume":
        pts = volume_cloud()
    elif name == "shifted":
        pts = shuffled(shifted(synthetic.camera_cloud(20000, seed=43), 3e3), 43)
    else:   # downsample -> tilefilter: the result keeps the bounding box of the whole cloud, which the kNN grid is built on
        raw = cw.cwipc_from_numpy_array(synthetic.camera_cloud(90000, seed=44), 1)
        raw._set_cellsize(synthetic.cellsize_of(90000))
        ds = cw.cwipc_downsample(raw, 0.006)
        pc = cw.cwipc_tilefilter(ds, 1)
        raw.free()
        ds.free()
        return pc, pc.get_numpy_array().copy()
    return cw.cwipc_from_numpy_array(pts, 1), pts


def nqueries(n):
    return sorted({1, 31, 32, 33, n // 3, n - 1, n})


_WHOLE = {}


def whole_cloud_ref(name, pts, k):
    """(mean, kth2) of every point of the cloud against the whole cloud (cached: the same for every nquery)."""
    key = (name, k)
    if key not in _WHOLE:
        lists = ref.ref_lists(pts, pts, k)
        _WHOLE[key] = ref.ref_mean(lists, k), ref.ref_kth2(lists, k).copy()
    return _WHOLE[key]


# ---- cwipc_cuda_knn_query ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", CLOUDS)
def test_knn_query_equals_the_reference(cw, name):
    """cwipc_cuda_knn_query: knn_tile_kernel (k <= 63) or knn_queue_all_kernel (k >= 64), knn_second_kernel and
    knn_far_kernel with d_kth set and nquery < n.  mean and kth2 of the first nquery points against ALL points must be the
    reference's, bit for bit: a halo point missed, a query skipped or a wrong (k+1)-th element shows."""
    pc, pts = make_cloud(cw, name)
    assert len(pts) > 512
    for k in QUERY_KS:
        want_mean, want_kth2 = whole_cloud_ref(name, pts, k)
        for nq in nqueries(len(pts)):
            mean, kth2 = cw.util.knn_query(pc, k, nq)
            assert np.array_equal(mean, want_mean[:nq]), (name, k, nq, np.flatnonzero(mean != want_mean[:nq])[:5])
            assert np.array_equal(kth2, want_kth2[:nq]), (name, k, nq, np.flatnonzero(kth2 != want_kth2[:nq])[:5])
    pc.free()


ENV_KS = [1, 30, 63, 200]


def dump_queries(path):
    """Child process of test_knn_query_passes_honour_nquery: knn_query of every cloud, k in ENV_KS, every nquery."""
    import cwipc_util_b200 as cw
    out = {}
    for name in CLOUDS:
        pc, pts = make_cloud(cw, name)
        out[f"{name}/pts"] = pts
        for k in ENV_KS:
            for nq in nqueries(len(pts)):
                out[f"{name}/{k}/{nq}/mean"], out[f"{name}/{k}/{nq}/kth2"] = cw.util.knn_query(pc, k, nq)
        pc.free()
    np.savez(path, **out)


# the settings of test_gpu_parity.py::test_knn_passes_split_the_work_not_the_result
@pytest.mark.parametrize("env", [
    {"CWIPC_CUDA_KNN_SECOND_FROM_N": "0"},
    {"CWIPC_CUDA_KNN_SECOND_FROM_N": "0", "CWIPC_CUDA_KNN_RC_FAR": "3.5", "CWIPC_CUDA_KNN_SECOND_MAX": "100000", "CWIPC_CUDA_KNN_SECOND_MIN": "1"},
    {"CWIPC_CUDA_KNN_RC_FAR": "0"},
    {"CWIPC_CUDA_KNN_SECOND_FROM_N": "0", "CWIPC_CUDA_KNN_PITCH": "0.6"},
    {"CWIPC_CUDA_KNN_RC_FAR": "0", "CWIPC_CUDA_KNN_PITCH": "0.4"},
    {"CWIPC_CUDA_KNN_RC_FAR": "0", "CWIPC_CUDA_KNN_PITCH": "0.4", "CWIPC_CUDA_KNN_FAR_START": "0"},
])
def test_knn_query_passes_honour_nquery(cw, env, tmp_path):
    """The tunables move queries between the main pass, the second scan (knn_second_kernel) and the tree search
    (knn_far_kernel); each of them must stop at nquery and still see the halo.  They are read once per process, so a child
    process runs with them set, and its mean and kth2 must be the reference's, bit for bit."""
    import subprocess
    path = str(tmp_path / "queries.npz")
    code = f"import sys; sys.path[:0] = [{REPO!r}, {TESTS!r}]; import test_gpu_knn_blocks as t; t.dump_queries({path!r})"
    subprocess.run([sys.executable, "-c", code], env=dict(os.environ, **env), check=True, timeout=900)
    got = np.load(path)
    for name in CLOUDS:
        pts = got[f"{name}/pts"]
        for k in ENV_KS:
            want_mean, want_kth2 = whole_cloud_ref(name, pts, k)
            for nq in nqueries(len(pts)):
                assert np.array_equal(got[f"{name}/{k}/{nq}/mean"], want_mean[:nq]), (name, k, nq)
                assert np.array_equal(got[f"{name}/{k}/{nq}/kth2"], want_kth2[:nq]), (name, k, nq)


# ---- cwipc_cuda_knn_query_open and the cwipc_cuda_distances_* calls ---------------------------------------------------------
def float32_beside(b):
    """The largest float32 below and the smallest above the float64 b."""
    f = np.float32(b)
    below = f if float(f) < b else np.nextafter(f, np.float32(-np.inf))
    above = f if float(f) > b else np.nextafter(f, np.float32(np.inf))
    return float(below), float(above)


def open_set(cw, pc, k, nq, x_lo, x_hi):
    h = cw.util.cuda_distances(pc, k, nq, x_lo, x_hi)
    idx, pts, kth2 = h.open_queries()
    assert len(idx) == h.nopen
    order = np.argsort(idx)   # a set: warps append the open queries in whatever order they finish
    return h, idx, idx[order], pts[order], kth2[order]


def test_open_queries_equal_the_reference(cw):
    """mark_open_kernel (float64 predicate), gather_points_kernel and gather_floats_kernel of cwipc_cuda_knn_query_open /
    cwipc_cuda_distances_open: the open set, the points and their kth2, at x_lo / x_hi one float32 on each side of chosen
    queries' boundaries, at (-inf, inf) (none open) and at x_lo > x_hi (all open)."""
    k = 30
    pc, pts = make_cloud(cw, "camera")
    nq = len(pts) // 2
    mean, kth2 = whole_cloud_ref("camera", pts, k)
    x = pts["x"][:nq].astype(np.float64)
    rk = np.sqrt(kth2[:nq].astype(np.float64)) * (1.0 + 1e-6)
    cases = [(-np.inf, np.inf), (1.0, -1.0), (-0.1, 0.1)]
    for i in (0, 17, nq // 2, nq - 1):
        lo_below, lo_above = float32_beside(x[i] - rk[i])
        hi_below, hi_above = float32_beside(x[i] + rk[i])
        cases += [(lo_below, np.inf), (lo_above, np.inf), (-np.inf, hi_below), (-np.inf, hi_above)]
    for x_lo, x_hi in cases:
        want = ref.ref_open(pts["x"], kth2, nq, x_lo, x_hi)
        h, raw, idx, opts, okth2 = open_set(cw, pc, k, nq, x_lo, x_hi)
        h.free()
        assert np.array_equal(idx, want), (x_lo, x_hi, len(idx), len(want))
        assert opts.tobytes() == pts[idx].tobytes()
        assert np.array_equal(okth2, kth2[idx])
        assert len(np.unique(raw)) == len(raw)
    assert open_set(cw, pc, k, nq, -np.inf, np.inf)[1].size == 0
    assert open_set(cw, pc, k, nq, 1.0, -1.0)[1].size == nq
    for i in (0, 17):   # the chosen queries flip exactly at their boundaries
        lo_below, lo_above = float32_beside(x[i] - rk[i])
        assert i not in ref.ref_open(pts["x"], kth2, nq, lo_below, np.inf) and i in ref.ref_open(pts["x"], kth2, nq, lo_above, np.inf)
    pc.free()


def test_open_queries_of_a_cloud_of_at_most_k_points(cw):
    """Fewer points than neighbours: every query is open and its kth2 is 0x7f7f7f7f (a huge finite float), whatever the
    interval."""
    for n in (1, 20, 30):
        pts = shuffled(synthetic.camera_cloud(400, seed=n), n)[:n]
        pc = cw.cwipc_from_numpy_array(pts, 1)
        for nq, x_lo, x_hi in ((n, -np.inf, np.inf), (max(1, n // 2), -1.0, 1.0)):
            h, _, idx, opts, okth2 = open_set(cw, pc, 30, nq, x_lo, x_hi)
            assert np.array_equal(idx, np.arange(nq, dtype=np.uint32))
            assert opts.tobytes() == pts[:nq].tobytes()
            assert np.all(okth2.view(np.uint32) == 0x7F7F7F7F)
            h.free()
        pc.free()


def test_patch_stats_and_filter_of_the_device_distances(cw):
    """scatter_floats_kernel (patch), stats_kernel on the device-resident distances, compact_kernel (filter): the stats
    before the patch are distance_stats of the reference means, after it of the patched host array (same kernel, same
    order: same bits), within sum_bound of the exact sums; the filter is filter_by_distance of the patched array."""
    k = 30
    pc, pts = make_cloud(cw, "camera")
    nq = len(pts) // 3
    mean, kth2 = whole_cloud_ref("camera", pts, k)
    local = cw.cwipc_from_numpy_array(pts[:nq].copy(), 1)
    for x_lo, x_hi in ((-0.05, 0.05), (1.0, -1.0)):
        h, raw, idx, _, _ = open_set(cw, pc, k, nq, x_lo, x_hi)
        assert h.stats() == cw.util.distance_stats(mean[:nq])
        values = np.random.default_rng(len(raw)).gamma(3.0, 0.01, len(raw)).astype(np.float32)
        values[:3] = [np.float32(0.0), mean[raw[3 % len(raw)]], np.float32(1.0)]
        h.patch(values)
        patched = mean[:nq].copy()
        patched[raw] = values
        got = h.stats()
        assert got == cw.util.distance_stats(patched)
        exact, bound = ref.exact_sums(patched), ref.sum_bound(nq, patched)
        assert abs(got[0] - exact[0]) <= bound[0] and abs(got[1] - exact[1]) <= bound[1]
        thr = cw.util.outlier_threshold(got[0], got[1], float(nq), 1.0)
        a = h.filter(local, thr)
        b = cw.util.filter_by_distance(local, patched, thr)
        assert a.get_numpy_array().tobytes() == b.get_numpy_array().tobytes()
        assert a.get_numpy_array().tobytes() == pts[:nq][~(patched.astype(np.float64) > thr)].tobytes()
        a.free()
        b.free()
        h.free()
    local.free()
    pc.free()


# ---- cwipc_cuda_knn_lists -----------------------------------------------------------------------------------------------
def list_queries(pts, seed):
    """Cloud points (distance 0, duplicates among them), midpoints of nearby pairs, points 0.5 m and 100 m outside the
    bounding box."""
    rng = np.random.default_rng(seed)
    n = len(pts)
    on = pts[rng.choice(n, 200, replace=False)]
    order = np.argsort(pts["x"], kind="stable")
    i = rng.choice(n - 1, 150, replace=False)
    a, b = pts[order[i]], pts[order[i + 1]]
    mid = a.copy()
    for c in "xyz":
        mid[c] = ((a[c].astype(np.float64) + b[c]) / 2).astype(np.float32)
    out = []
    for off in (0.5, 100.0):
        q = pts[rng.choice(n, 25, replace=False)].copy()
        axis = rng.choice(list("xyz"), 25)
        for j, c in enumerate(axis):
            side = rng.integers(0, 2)
            q[c][j] = np.float32(pts[c].max() + off) if side else np.float32(pts[c].min() - off)
        out.append(q)
    return np.concatenate([on, pts[:2], mid] + out)


def limit_cases(full, k, seed):
    """(name, limits, j): None, +inf, 0, negative, NaN, exactly element j, the float below element j."""
    nq = len(full)
    j = int(np.random.default_rng(seed).integers(0, k + 1))
    exact = full[:, j].copy()
    return [("none", None), ("inf", np.full(nq, np.inf, np.float32)), ("zero", np.zeros(nq, np.float32)),
            ("negative", np.full(nq, -1e-3, np.float32)), ("nan", np.full(nq, np.nan, np.float32)),
            (f"element {j}", exact), (f"below element {j}", np.nextafter(exact, np.float32(-np.inf)))]


@pytest.mark.parametrize("name", ["camera", "shifted"])
def test_knn_lists_equal_the_reference(cw, name):
    """knn_list_kernel -> dfs_knn from the root, with and without limits: the k+1 smallest d² <= limit of external
    queries, ascending, +inf padded, bit for bit.  A limit equal to a list element must report it (d² <= limit), the
    float below it must not; k on both sides of every list width; cellsize hints 0, 1e-5 and 1."""
    pc, pts = make_cloud(cw, name)
    pc.free()
    pts[1] = pts[0]   # a duplicate, asked for below
    queries = list_queries(pts, seed=len(name))
    fulls = {k: ref.ref_lists(pts, queries, k) for k in LIST_KS}
    for cellsize in (0.0, 1e-5, 1.0):
        pc = cw.cwipc_from_numpy_array(pts, 1)
        pc._set_cellsize(cellsize)
        for k, full in fulls.items():
            for what, limits in limit_cases(full, k, seed=k):
                got = cw.util.knn_lists(pc, queries, k, limits)
                want = full if limits is None else ref.with_limits(full, limits)
                assert np.array_equal(got, want), (name, cellsize, k, what, np.argwhere(got != want)[:5])
        pc.free()


def test_knn_lists_of_empty_and_small_clouds(cw):
    """n = 0: every list is +inf.  0 < n < k+1: the n distances, then +inf padding."""
    queries = list_queries(synthetic.camera_cloud(400, seed=3), seed=3)[:64]
    empty = cw.cwipc_from_points([], 0)
    for k in (1, 31, 64, 511):
        assert np.all(cw.util.knn_lists(empty, queries, k) == np.inf)
    empty.free()
    for n in (1, 5, 31, 32, 33, 100):
        cloud = shuffled(synthetic.camera_cloud(400, seed=n), n)[:n]
        pc = cw.cwipc_from_numpy_array(cloud, 1)
        for k in (31, 32, 63, 127, 511):
            got = cw.util.knn_lists(pc, queries, k)
            assert np.array_equal(got, ref.ref_lists(cloud, queries, k)), (n, k)
            if n < k + 1:
                assert np.all(got[:, n:] == np.inf) and np.all(np.isfinite(got[:, :n]))
        pc.free()


# ---- cwipc_cuda_knn_merge_lists ------------------------------------------------------------------------------------------
def splits(pts, G, seed):
    """(how, parts): random, x-slabs, and one part left empty."""
    rng = np.random.default_rng(seed)
    n = len(pts)
    owner = rng.integers(0, G, n)
    yield "random", [pts[owner == g] for g in range(G)]
    edges = np.quantile(pts["x"], np.linspace(0, 1, G + 1))
    slab = np.clip(np.searchsorted(edges, pts["x"], side="right") - 1, 0, G - 1)
    yield "x-slabs", [pts[slab == g] for g in range(G)]
    if G > 1:
        owner = rng.integers(0, G - 1, n)
        owner[owner >= G // 2] += 1   # part G // 2 holds nothing
        yield "one empty", [pts[owner == g] for g in range(G)]


@pytest.mark.parametrize("G", [1, 2, 3, 16])
def test_merged_lists_equal_the_whole_cloud(cw, G):
    """knn_merge_lists_kernel over lists from knn_list_kernel: each part answers the same queries with limits = the
    whole cloud's kth2 and with no limit; the merged mean and kth2 are the whole cloud's, bit for bit."""
    pc, pts = make_cloud(cw, "camera")
    pc.free()
    pts = pts[:20000]
    queries = pts[:1500]
    for k in (7, 30, 200):
        mean, kth2 = whole_cloud_ref("camera20k", pts, k)
        mean, kth2 = mean[:1500], kth2[:1500]
        for how, parts in splits(pts, G, seed=G + k):
            for limits in (kth2, None):
                lists = []
                for part in parts:
                    pc = cw.cwipc_from_numpy_array(part, 1)
                    lists.append(cw.util.knn_lists(pc, queries, k, limits))
                    pc.free()
                got_mean, got_kth2 = cw.util.knn_merge_lists(np.stack(lists), k)
                assert np.array_equal(got_mean, mean), (k, how, limits is None)
                assert np.array_equal(got_kth2, kth2), (k, how, limits is None)


def merged_ref(lists, k):
    merged = np.sort(np.concatenate(list(lists), axis=1), axis=1)[:, :k + 1]
    return ref.ref_mean(merged, k), ref.ref_kth2(merged, k)


def test_merge_lists_written_by_hand(cw, lib):
    """knn_merge_lists_kernel on lists that no search produces: equal values in different lists (each counted once per
    list it is in), all-+inf lists, and fewer than k+1 finite entries in total (mean +inf); 17 lists are refused."""
    rng = np.random.default_rng(12)
    k = 9
    for nlists in (2, 3, 16):
        lists = np.sort(rng.choice(np.array([0.0, 0.25, 1.0, 2.0, 4.0, 9.0], np.float32), (nlists, 64, k + 1)), axis=2)
        lists[:, :8] = np.sort(rng.uniform(0, 1, (nlists, 8, k + 1)).astype(np.float32), axis=2)
        lists[0, 8:16] = np.inf                              # one list all +inf
        lists[-1, 16:24] = lists[0, 16:24]                   # the same list twice
        lists[:, 24:32, 1:] = np.inf                         # one finite entry per list
        lists[:, 32:40, :] = np.inf                          # nothing at all
        lists[-1, 40:48] = 0.0                               # the smallest entries in the last list
        mean, kth2 = cw.util.knn_merge_lists(lists, k)
        want_mean, want_kth2 = merged_ref(lists, k)
        assert np.array_equal(mean, want_mean) and np.array_equal(kth2, want_kth2), nlists
        if nlists <= k:
            assert np.all(mean[24:40] == np.inf)
        assert np.all(mean[32:40] == np.inf) and np.all(kth2[32:40] == np.inf)
    seen = []
    cw.cwipc_log_configure(cw.CWIPC_LOG_LEVEL_WARNING, lambda level, msg: seen.append((level, msg.decode())))
    try:
        lists = np.zeros((17, 4, k + 1), np.float32)
        mean, kth2 = np.zeros(4, np.float32), np.zeros(4, np.float32)
        assert lib.cwipc_cuda_knn_merge_lists(lists.ctypes.data, 17, 4, k, mean.ctypes.data, kth2.ctypes.data) == -1
    finally:
        cw.cwipc_log_configure(cw.CWIPC_LOG_LEVEL_WARNING, None)
    errors = [m for level, m in seen if level == cw.CWIPC_LOG_LEVEL_ERROR]
    assert len(errors) == 1 and errors[0].startswith("cwipc_cuda_knn_merge_lists: "), seen


# ---- statistics and threshold --------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n", [0, 1, 255, 65535, 65536, 65537, 2 ** 20 + 3])
def test_distance_stats_within_the_bound_of_the_exact_sums(cw, n):
    """stats_kernel + the host's 256 serial adds: sum d and sum float32(d*d) in double, in a fixed order.  Within
    sum_bound of the exact sums (a square taken in double, or a sum in float, is far outside it), the same bits twice."""
    d = np.random.default_rng(n).gamma(3.0, 0.01, n).astype(np.float32)
    got = cw.util.distance_stats(d)
    assert cw.util.distance_stats(d) == got
    exact, bound = ref.exact_sums(d), ref.sum_bound(n, d)
    assert abs(got[0] - exact[0]) <= bound[0], (got[0] - exact[0], bound[0])
    assert abs(got[1] - exact[1]) <= bound[1], (got[1] - exact[1], bound[1])
    if n == 0:
        assert got == (0.0, 0.0)


def same_double(a, b):
    return (np.isnan(a) and np.isnan(b)) or np.float64(a).view(np.uint64) == np.float64(b).view(np.uint64)


def test_outlier_threshold_is_the_float64_formula(cw):
    """outlier_threshold: mean + mul * sqrt((sq - sum*sum/n) / (n - 1)) in double, in this order, bit for bit; n = 1
    gives NaN (0/0) or +inf (x/0)."""
    rng = np.random.default_rng(4)
    for _ in range(200):
        n = float(rng.integers(2, 10 ** 7))
        d = rng.gamma(3.0, 0.01, 64)
        s = float(d.sum() * n / 64)
        sq = float((d * d).sum() * n / 64 * rng.uniform(1.0, 1.5))
        mul = float(rng.choice([0.5, 1.0, 1.5, 2.5, 3.3]))
        assert same_double(cw.util.outlier_threshold(s, sq, n, mul), ref.threshold_formula(s, sq, n, mul)), (s, sq, n, mul)
    for s, sq in ((0.5, 0.25), (0.5, 0.3), (0.1, 0.1 * 0.1), (3.0, 9.0)):
        got = cw.util.outlier_threshold(s, sq, 1.0, 1.0)
        assert same_double(got, ref.threshold_formula(s, sq, 1.0, 1.0)), (s, sq, got)
    assert np.isnan(cw.util.outlier_threshold(0.5, 0.25, 1.0, 1.0)) and cw.util.outlier_threshold(0.5, 0.3, 1.0, 1.0) == np.inf


@pytest.mark.parametrize("n,k,mul", [(6400, 30, 1.0), (90000, 30, 1.0), (200000, 8, 2.5), (50000, 63, 0.5)])
def test_remove_outliers_is_its_building_blocks(cw, orc, n, k, mul):
    """stats_threshold_kernel (sums and threshold on the device) against the building blocks: cwipc_remove_outliers must
    be byte-identical to filter_by_distance(d, outlier_threshold(*distance_stats(d), n, mul)) with d the kNN mean
    distances, and must keep exactly the points at or under the threshold of the exact sums (exact_keep_check)."""
    pts = synthetic.camera_cloud(n, seed=n % 97 + k)
    pc = cw.cwipc_from_numpy_array(pts, 1)
    d = cw.util.knn_mean_distances(pc, k)
    thr = cw.util.outlier_threshold(*cw.util.distance_stats(d), float(len(pts)), mul)
    got = cw.cwipc_remove_outliers(pc, k, mul, False).get_numpy_array().copy()
    assert got.tobytes() == cw.util.filter_by_distance(pc, d, thr).get_numpy_array().tobytes()
    ref.exact_keep_check(pts, got, orc.knn_mean_distances(pts, k), mul)
    assert 0 < len(got) < len(pts)
    pc.free()


def test_per_tile_keep_decisions_at_the_exact_threshold(cw, orc):
    """stats_threshold_tile_kernel + compact_tile_group_chained: group by group (first-appearance order of the tile
    value), the kept points are those at or under the group's threshold of the exact sums.  Groups of k+1 and k+2 points
    have statistics; a group of at most k is kept whole."""
    k, mul = 30, 1.0
    pts = synthetic.camera_cloud(60000, seed=23)
    rng = np.random.default_rng(23)
    where = rng.choice(len(pts), 3 * k + 3, replace=False)
    pts["tile"][where[:k + 1]] = 16
    pts["tile"][where[k + 1:2 * k + 3]] = 32
    pts["tile"][where[2 * k + 3:]] = 64   # k points
    pc = cw.cwipc_from_numpy_array(pts, 1)
    got = cw.cwipc_remove_outliers(pc, k, mul, True).get_numpy_array().copy()
    pc.free()
    _, first = np.unique(pts["tile"], return_index=True)
    pos = 0
    for t in pts["tile"][np.sort(first)]:
        grp = pts[pts["tile"] == t]
        if len(grp) <= k:
            assert got[pos:pos + len(grp)].tobytes() == grp.tobytes()
            pos += len(grp)
        else:
            pos += ref.exact_keep_check(grp, got[pos:], orc.knn_mean_distances(grp, k), mul, whole=False)
    assert pos == len(got)


def test_slab_protocol_sharing_one_gpu_at_the_exact_threshold(cw, orc, tmp_path):
    """slab.py's protocol with the library's building blocks on one shared GPU (gloo): open queries, lists, merge,
    device distances, all-reduced sums.  The survivors, in rank order, must be exactly those at or under the threshold of
    the exact sums of the whole cloud's distances."""
    import _slab_runner as runner
    from test_slab_cpu import make_parts
    parts = make_parts(40000, 3, seed=61)
    _, sorn, _ = runner.launch(3, "cuda-shared", parts, str(tmp_path), voxelsize=0.01, k=30, mul=1.0, cellsize=0.002, port=29761)
    whole = np.concatenate(parts)
    ref.exact_keep_check(whole, np.concatenate(sorn), orc.knn_mean_distances(whole, 30), 1.0)


# ---- cwipc_cuda_filter_by_distance ---------------------------------------------------------------------------------------
def test_filter_by_distance_compares_in_double(cw, lib):
    """compact_kernel with DistPred: keep point i iff !((double)dist[i] > threshold), order kept.  A threshold one double
    below 1.0 drops a distance of 1.0f (a comparison in float would keep it); NaN thresholds and NaN distances keep."""
    pts = shuffled(synthetic.camera_cloud(10000, seed=5), 5)
    n = len(pts)
    pc = cw.cwipc_from_numpy_array(pts, 1)
    rng = np.random.default_rng(5)
    d = rng.gamma(3.0, 0.01, n).astype(np.float32)
    d[::7] = 1.0
    d[3::11] = np.nan
    d[5::13] = np.inf

    def kept(dist, thr):
        return cw.util.filter_by_distance(pc, dist, thr).get_numpy_array().tobytes()

    below_one = float(np.nextafter(1.0, 0.0))
    for thr in (below_one, 1.0, float(np.nextafter(1.0, 2.0)), 0.03, float(np.float32(0.03)), np.inf, -np.inf, np.nan, 0.0):
        with np.errstate(invalid="ignore"):
            want = pts[~(d.astype(np.float64) > thr)]
        assert kept(d, thr) == want.tobytes(), thr
    ones = np.ones(n, np.float32)
    assert kept(ones, below_one) == b""
    assert kept(ones, 1.0) == pts.tobytes()
    assert kept(np.full(n, np.nan, np.float32), -np.inf) == pts.tobytes()
    assert kept(d, np.nan) == pts.tobytes()
    seen = []
    cw.cwipc_log_configure(cw.CWIPC_LOG_LEVEL_WARNING, lambda level, msg: seen.append((level, msg.decode())))
    try:
        assert not lib.cwipc_cuda_filter_by_distance(pc.as_cwipc_p(), d.ctypes.data, n - 1, 1.0)
    finally:
        cw.cwipc_log_configure(cw.CWIPC_LOG_LEVEL_WARNING, None)
    errors = [m for level, m in seen if level == cw.CWIPC_LOG_LEVEL_ERROR]
    assert len(errors) == 1 and errors[0].startswith("cwipc_cuda_filter_by_distance: "), seen
    pc.free()
