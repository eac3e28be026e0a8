"""GPU parity tests: the CUDA path, called through the C ABI (ctypes mirror of python/cwipc/util.py),
against the CPU oracle on identical input buffers, against the committed golden fixtures, and -- at
BASELINE.json's full sizes -- through size-independent properties.

Bars (BASELINE.json north_star): tilefilter output, voxel keys, point counts and tile masks bit-exact;
centroids within 1e-5 relative (scale = max(|coordinate|, voxel size)); colours within +-1 LSB;
outlier keep-masks identical except for points within 1e-6 (relative) of the threshold.
"""
import ctypes
import os

import numpy as np
import pytest
import sys

from cwipc_util_b200 import synthetic

pytestmark = pytest.mark.gpu

DT = synthetic.cwipc_point_numpy_dtype
REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "golden_small.npz")


def random_cloud(n, seed=0, extent=1.0, tiles=(1, 2, 4, 8)):
    rng = np.random.default_rng(seed)
    pts = np.zeros(n, DT)
    pts["x"] = rng.uniform(-extent, extent, n).astype(np.float32)
    pts["y"] = rng.uniform(0, 2 * extent, n).astype(np.float32)
    pts["z"] = rng.uniform(-extent, extent, n).astype(np.float32)
    for c in "rgb":
        pts[c] = rng.integers(0, 256, n).astype(np.uint8)
    pts["tile"] = rng.choice(np.array(tiles, np.uint8), n)
    return pts


def upload(cw, pts, timestamp=1234, cellsize=None):
    pc = cw.cwipc_from_numpy_array(pts, timestamp)
    if cellsize is not None:
        pc._set_cellsize(cellsize)
    return pc


def download(pc):
    return pc.get_numpy_array().copy()


def assert_points_close(got, want, cs):
    """xyz within 1e-5 relative, colours within 1 LSB, tiles exact, same order."""
    assert len(got) == len(want)
    for a in "xyz":
        scale = np.maximum(np.abs(want[a].astype(np.float64)), cs)
        err = np.abs(got[a].astype(np.float64) - want[a].astype(np.float64)) / scale
        assert err.max(initial=0.0) <= 1e-5, f"{a}: max rel err {err.max()}"
    for c in "rgb":
        assert np.abs(got[c].astype(np.int32) - want[c].astype(np.int32)).max(initial=0) <= 1
    assert np.array_equal(got["tile"], want["tile"])


# ======================================================================================================
# object model (ref: python/test_cwipc_util.py:80-104, 182-223, 252-288)
# ======================================================================================================
def test_from_points_roundtrip_and_empty(cw):
    pc = cw.cwipc_from_points([], 0)
    assert pc.count() == 0 and pc.get_uncompressed_size() == 0 and len(pc.get_points()) == 0
    points = cw.cwipc_point_array(values=[(1, 2, 3, 0x10, 0x20, 0x30, 1), (4, 5, 6, 0x40, 0x50, 0x60, 2)])
    pc = cw.cwipc_from_points(points, 0)
    assert pc.count() == 2
    new = pc.get_points()
    assert all(points[i] == new[i] for i in range(2))
    big = random_cloud(300001, seed=1)
    assert np.array_equal(download(upload(cw, big)), big)


def test_pageable_copies_through_the_staging_ring(cw):
    """cwipc_from_points / copy_uncompressed with ordinary (pageable) caller memory travel through the calling thread's
    page-locked ring in 2 MB chunks (csrc/runtime.cu: copy_from_host / copy_to_host): sizes around the 1 MB threshold and
    the chunk edges, more chunks than ring slots, back-to-back calls reusing slots in flight, and four threads at once."""
    import threading
    sizes = [65535, 65536, 65537, 131071, 131072, 131073, 4 * 131072, 4 * 131072 + 1, 1000003, 2500000]
    clouds = {n: random_cloud(n, seed=n % 97) for n in sizes}
    pcs = [(n, upload(cw, clouds[n])) for n in sizes]          # uploads back to back: ring slots still in flight
    for n, pc in pcs:
        assert pc.count() == n
        assert np.array_equal(download(pc), clouds[n]), n
        pc.free()
    errors = []

    def worker(seed):
        try:
            cw.cuda_set_device(0)
            for rep in range(3):
                pts = random_cloud(700001 + 4099 * seed, seed=seed * 10 + rep)
                pc = upload(cw, pts)
                d = cw.cwipc_tilefilter(pc, 2)
                assert np.array_equal(download(pc), pts)
                assert np.array_equal(download(d), pts[pts["tile"] == 2])
                d.free()
                pc.free()
        except Exception as e:  # pragma: no cover
            errors.append(e)

    threads = [threading.Thread(target=worker, args=(i,)) for i in range(4)]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    assert not errors, errors
    # short-lived threads, one after the other (a host that starts a thread per frame): each adopts the ring its predecessor
    # left behind instead of pinning another 8 MB
    for i in range(6):
        t = threading.Thread(target=worker, args=(10 + i,))
        t.start()
        t.join()
    assert not errors, errors


def test_from_points_size_mismatch_raises(cw, lib):
    cw.cwipc_log_configure(cw.CWIPC_LOG_LEVEL_NONE, lambda level, msg: None)
    try:
        pts = random_cloud(4)
        err = ctypes.c_char_p()
        rv = lib.cwipc_from_points(pts.ctypes.data, 4 * 16 - 1, 4, 0, ctypes.byref(err), cw.CWIPC_API_VERSION)
        assert not rv and err.value
    finally:
        cw.cwipc_log_configure(cw.CWIPC_LOG_LEVEL_WARNING, None)


def test_timestamp_cellsize(cw, orc):
    timestamp = 0x11223344556677
    pc = cw.cwipc_from_points([(0, 0, 0, 0, 0, 0, 1), (1, 0, 0, 0, 0, 0, 1), (2, 0, 0, 0, 0, 0, 1), (3, 0, 0, 0, 0, 0, 1)], timestamp)
    assert pc.timestamp() == timestamp
    pc._set_timestamp(timestamp + 1)
    assert pc.timestamp() == timestamp + 1
    assert pc.cellsize() == 0
    pc._set_cellsize(0.1)
    assert pc.cellsize() == pytest.approx(0.1)
    pc._set_cellsize(-1)
    assert pc.cellsize() == 1.0
    pts = random_cloud(100000, seed=2)
    pc = upload(cw, pts)
    pc._set_cellsize(-1)
    assert pc.cellsize() == np.float32(orc.min_distance_to_first(pts))


def test_dangling_allocations_and_clone(cw):
    old = cw.cwipc_dangling_allocations(False)
    pc = upload(cw, random_cloud(1000))
    assert cw.cwipc_dangling_allocations(False) == old + 1
    clone = pc.clone()
    assert cw.cwipc_dangling_allocations(False) == old + 2
    assert clone.count() == pc.count() and clone.timestamp() == pc.timestamp()
    pc.free()
    assert np.array_equal(download(clone), random_cloud(1000))  # the clone keeps the shared storage alive
    clone.free()
    assert cw.cwipc_dangling_allocations(False) == old


def test_packet_and_debugdump_roundtrip(cw, tmp_path):
    pts = random_cloud(5000, seed=3)
    pc = upload(cw, pts, timestamp=987654321, cellsize=0.25)
    packet = pc.get_packet()
    assert len(packet) == 32 + 16 * len(pts)
    pc2 = cw.cwipc_from_packet(packet)
    assert pc2.timestamp() == 987654321 and pc2.cellsize() == 0.25
    assert np.array_equal(download(pc2), pts)
    assert pc2.get_packet() == packet
    fn = str(tmp_path / "a.cwipcdump")
    assert cw.cwipc_write_debugdump(fn, pc) == 0
    pc3 = cw.cwipc_read_debugdump(fn)
    assert pc3.timestamp() == 987654321 and pc3.cellsize() == 0.25 and np.array_equal(download(pc3), pts)
    for flags in (0, cw.CWIPC_FLAGS_BINARY):
        ply = str(tmp_path / f"a{flags}.ply")
        assert cw.cwipc_write(ply, pc, flags) == 0
        pc4 = cw.cwipc_read(ply, 77)
        assert pc4.timestamp() == 77 and np.array_equal(download(pc4), pts)


def test_copy_uncompressed_buffer_too_small(cw, lib):
    cw.cwipc_log_configure(cw.CWIPC_LOG_LEVEL_NONE, lambda level, msg: None)
    try:
        pc = upload(cw, random_cloud(10))
        buf = (ctypes.c_byte * 100)()
        assert lib.cwipc_pointcloud_copy_uncompressed(pc.as_cwipc_p(), ctypes.addressof(buf), 100) == -1
        assert lib.cwipc_pointcloud_copy_packet(pc.as_cwipc_p(), ctypes.addressof(buf), 100) == 0
    finally:
        cw.cwipc_log_configure(cw.CWIPC_LOG_LEVEL_WARNING, None)


def test_synthetic_source(cw):
    gen = cw.cwipc_synthetic()
    assert gen.start()
    pc = gen.get()
    assert pc.count() == 160000 and pc.cellsize() == pytest.approx(2.0 / 400)
    pts = download(pc)
    assert set(np.unique(pts["tile"]).tolist()) == {1, 2}
    gen.stop()
    gen.free()


# ======================================================================================================
# tilefilter and the other per-point filters: bit-exact, order preserved
# ======================================================================================================
@pytest.mark.parametrize("n", [0, 1, 31, 2047, 2048, 2049, 70001, 1000000])
def test_tilefilter_bit_exact(cw, orc, n):
    pts = random_cloud(n, seed=n, tiles=(0, 1, 2, 5))
    pc = upload(cw, pts, timestamp=42, cellsize=0.5)
    for tile in (0, 1, 2, 5, 6, 300):
        out = cw.cwipc_tilefilter(pc, tile)
        assert out.timestamp() == 42 and out.cellsize() == 0.5
        assert np.array_equal(download(out), orc.tilefilter(pts, tile)), f"n={n} tile={tile}"


def test_tilefilter_reference_properties(cw):
    """python/test_cwipc_util.py:428-450"""
    gen = cw.cwipc_synthetic()
    gen.start()
    pc = gen.get()
    n = len(pc.get_points())
    assert len(cw.cwipc_tilefilter(pc, 0).get_points()) == n
    f1, f2 = cw.cwipc_tilefilter(pc, 1), cw.cwipc_tilefilter(pc, 2)
    assert len(f1.get_points()) + len(f2.get_points()) == n
    assert f1.timestamp() == pc.timestamp() == f2.timestamp()
    empty = cw.cwipc_from_points([], 0)
    assert len(cw.cwipc_tilefilter(empty, 0).get_points()) == 0
    gen.free()


def test_tilefilter_masked_crop_tilemap_colormap_join(cw):
    pts = random_cloud(50000, seed=7, tiles=(1, 2, 4, 8, 3))
    pc = upload(cw, pts, timestamp=5, cellsize=0.125)
    assert np.array_equal(download(cw.cwipc_tilefilter_masked(pc, 3)), pts[(pts["tile"] & 3) != 0])
    box = [-0.25, 0.5, 0.1, 1.0, -2, 0.0]
    keep = (box[0] <= pts["x"]) & (pts["x"] < box[1]) & (box[2] <= pts["y"]) & (pts["y"] < box[3]) & (box[4] <= pts["z"]) & (pts["z"] < box[5])
    assert np.array_equal(download(cw.cwipc_crop(pc, box)), pts[keep])
    mapped = download(cw.cwipc_tilemap(pc, {1: 5, 2: 6}))
    want = pts.copy()
    table = np.zeros(256, np.uint8)
    table[1], table[2] = 5, 6
    want["tile"] = table[pts["tile"]]
    assert np.array_equal(mapped, want)
    col = download(cw.cwipc_colormap(pc, 0xFFFFFFFF, 0x010203))
    assert np.array_equal(col["x"], pts["x"]) and set(col["r"]) == {1} and set(col["g"]) == {2} and set(col["b"]) == {3} and set(col["tile"]) == {0}
    col2 = download(cw.cwipc_colormap(pc, 0x00FF0000, 0x02000000))  # clear red, OR 2 into tile
    assert np.all(col2["r"] == 0) and np.array_equal(col2["g"], pts["g"]) and np.array_equal(col2["tile"], pts["tile"] | 2)
    other = upload(cw, pts[:777], timestamp=3, cellsize=0.5)
    joined = cw.cwipc_join(pc, other)
    assert joined.timestamp() == 3 and joined.cellsize() == 0.125
    assert np.array_equal(download(joined), np.concatenate([pts, pts[:777]]))


# ======================================================================================================
# downsample
# ======================================================================================================
def canonical_ranks(keys6):
    """rank of every point's (leaf, voxel) group in the reference output order"""
    depth = 21
    l = keys6[:, :3].astype(np.int64)
    m = np.zeros(len(l), np.int64)
    for b in range(depth):
        m |= ((l[:, 0] >> b) & 1) << (3 * b + 2)
        m |= ((l[:, 1] >> b) & 1) << (3 * b + 1)
        m |= ((l[:, 2] >> b) & 1) << (3 * b)
    v = keys6[:, 3:].astype(np.int64)
    order = np.lexsort((v[:, 0], v[:, 1], v[:, 2], m))
    full = np.concatenate([m[:, None], v[:, ::-1]], axis=1)[order]
    heads = np.ones(len(full), bool)
    heads[1:] = np.any(full[1:] != full[:-1], axis=1)
    ranks = np.empty(len(full), np.int64)
    ranks[order] = np.cumsum(heads) - 1
    return ranks


@pytest.mark.parametrize("n,voxel,pc_cellsize", [(6400, 0.06, 0.0), (40000, 0.01, 0.0), (40000, -0.01, 0.0), (250000, 0.004, 0.0), (250000, -0.03, 0.0),
                                                 (160000, 0.002, 0.005), (90000, 0.3, 0.0), (90000, -0.3, 0.0), (1000000, 0.01, 0.002)])
def test_downsample_matches_oracle(cw, orc, n, voxel, pc_cellsize):
    pts = synthetic.camera_cloud(n, seed=n % 97)
    want, cs, keys6, counts = orc.downsample(pts, voxel, pc_cellsize, want_keys=True)
    pc = upload(cw, pts, timestamp=99, cellsize=pc_cellsize)
    out = cw.cwipc_downsample(pc, voxel)
    assert out.timestamp() == 99
    assert out.cellsize() == np.float32(cs)
    got = download(out)
    assert len(got) == len(want)                       # surviving voxel count, bit-exact
    assert_points_close(got, want, cs)                 # same order, centroids / colours / tile masks
    # voxel keys: the GPU sort key must induce exactly the oracle's grouping and output order
    gkeys = cw.util.downsample_keys(pc, voxel)
    _, inverse = np.unique(gkeys, return_inverse=True)
    assert np.array_equal(inverse, canonical_ranks(keys6))
    # per-voxel point counts
    assert np.array_equal(np.bincount(inverse, minlength=len(want)), counts)


def test_downsample_random_volume_and_unordered_input(cw, orc):
    pts = random_cloud(300000, seed=5, extent=0.4)
    for voxel in (0.05, -0.05, 0.013):
        want, cs, _, _ = orc.downsample(pts, voxel, 0.0)
        got = download(cw.cwipc_downsample(upload(cw, pts), voxel))
        assert_points_close(got, want, cs)


def test_downsample_long_runs_and_tile_boundaries(cw, orc):
    """Everything in a handful of voxels: runs span many reduce tiles; colours stay within 1 LSB."""
    pts = synthetic.camera_cloud(500000, seed=1)
    for voxel in (2.5, -2.5, 0.7):
        want, cs, _, counts = orc.downsample(pts, voxel, 0.0)
        got = download(cw.cwipc_downsample(upload(cw, pts), voxel))
        assert len(got) == len(want) <= 64
        assert counts.max() > 10000
        for a in "xyz":  # the oracle's float running sum is itself only ~1e-4 accurate on such runs
            assert np.allclose(got[a], want[a], rtol=2e-4, atol=2e-4)
        exact = {a: np.array([pts[a].astype(np.float64).mean()]) for a in "xyz"}
        if len(got) == 1:
            for a in "xyz":
                assert got[a][0] == np.float32(exact[a][0])  # fixed-point sums: correctly rounded mean
        for c in "rgb":
            assert np.abs(got[c].astype(int) - want[c].astype(int)).max() <= 1
        assert np.array_equal(got["tile"], want["tile"])


def test_downsample_edge_cases(cw, orc):
    cw.cwipc_log_configure(cw.CWIPC_LOG_LEVEL_NONE, lambda level, msg: None)
    try:
        empty = cw.cwipc_from_points([], 7)
        out = cw.cwipc_downsample(empty, 1.0)            # python/test_cwipc_util.py:589-594
        assert out.count() == 0 and out.timestamp() == 7
        assert not cw.util.cwipc_util_dll_load().cwipc_downsample(empty.as_cwipc_p(), -1.0)  # reference: ERROR + NULL
        assert not cw.util.cwipc_util_dll_load().cwipc_downsample(None, 1.0)
        one = upload(cw, random_cloud(1))
        assert cw.cwipc_downsample(one, 0.1).count() == 1 and cw.cwipc_downsample(one, -0.1).count() == 1
        # index overflow in single-grid mode -> NULL like the reference
        wide = random_cloud(1000, extent=100.0)
        assert orc.downsample(wide, -0.001)[0] is None
        assert not cw.util.cwipc_util_dll_load().cwipc_downsample(upload(cw, wide).as_cwipc_p(), -0.001)
        # the voxel cut by a leaf face (SURVEY.md finding 2)
        pts = np.zeros(3, DT)
        pts["x"] = [0.5, 0.25, 0.75]
        pts["tile"] = [1, 2, 4]
        assert cw.cwipc_downsample(upload(cw, pts), -1.0).count() == 1
        assert cw.cwipc_downsample(upload(cw, pts), 1.0).count() == 2
    finally:
        cw.cwipc_log_configure(cw.CWIPC_LOG_LEVEL_WARNING, None)


@pytest.mark.parametrize("sign", [1, -1])
def test_downsample_reference_doubling_property(cw, sign):
    """python/test_cwipc_util.py:543-587"""
    gen = cw.cwipc_synthetic()
    gen.start()
    pc = gen.get()
    count_orig = len(pc.get_points())
    count = count_orig
    cellsize = pc.cellsize() / 2
    while cellsize < 16:
        out = cw.cwipc_downsample(pc, sign * cellsize)
        count = len(out.get_points())
        assert 1 <= count <= count_orig
        assert out.timestamp() == pc.timestamp()
        if count < 2:
            break
        cellsize *= 2
    assert count <= 8
    gen.free()


# ======================================================================================================
# outlier removal
# ======================================================================================================
@pytest.mark.parametrize("n,k,cellsize", [(6400, 30, 0.0), (40000, 30, 0.01), (40000, 5, 0.0), (100000, 30, 0.0063), (100000, 63, 0.0), (30000, 10, 1.0), (30000, 10, 1e-5)])
def test_knn_mean_distances_bit_exact(cw, orc, n, k, cellsize):
    """Exact kNN: identical float distances, identical summation order -> identical floats, whatever the grid pitch."""
    pts = synthetic.camera_cloud(n, seed=n % 89 + k)
    want = orc.knn_mean_distances(pts, k)
    got = cw.util.knn_mean_distances(upload(cw, pts, cellsize=cellsize), k)
    assert np.array_equal(got, want)


def test_knn_random_volume_duplicates_and_far_outliers(cw, orc):
    pts = random_cloud(60000, seed=8, extent=0.3)
    pts["x"][:200] = pts["x"][0]
    pts["y"][:200] = pts["y"][0]
    pts["z"][:200] = pts["z"][0]
    pts["x"][-1], pts["y"][-2], pts["z"][-3] = 55.0, -70.0, 1000.0
    for k in (1, 30):
        assert np.array_equal(cw.util.knn_mean_distances(upload(cw, pts), k), orc.knn_mean_distances(pts, k))


@pytest.mark.parametrize("k", [1, 7, 8, 15, 16, 31, 32, 40, 63])
def test_knn_every_list_width(cw, orc, k):
    """k+1 on both sides of every register-list width (8/16/32/64) and of the 32-lane far list."""
    pts = synthetic.add_outliers(synthetic.camera_cloud(20000, seed=k), 0.02, seed=k)
    assert np.array_equal(cw.util.knn_mean_distances(upload(cw, pts, cellsize=0.004), k), orc.knn_mean_distances(pts, k))


def test_knn_mostly_far_queries_and_dense_cells(cw, orc):
    """A pitch far too small (every query goes through the octree search), one far too large (a handful of
    cells, thousands of candidates per stage ring), and clumps denser than one TMA stage."""
    rng = np.random.default_rng(5)
    pts = random_cloud(30000, seed=11, extent=0.5)
    clump = rng.integers(0, 30000, 40)
    for j, c in enumerate(clump):          # 40 clumps of 150 near-identical points
        sl = slice(j * 150, (j + 1) * 150)
        for a in "xyz":
            pts[a][sl] = pts[a][c] + rng.normal(0, 1e-4, 150).astype(np.float32)
    want = orc.knn_mean_distances(pts, 30)
    for cellsize in (1e-4, 0.0, 0.2):
        assert np.array_equal(cw.util.knn_mean_distances(upload(cw, pts, cellsize=cellsize), 30), want), cellsize


@pytest.mark.parametrize("k", [64, 65, 100, 127, 128, 200, 255, 256, 400, 511])
def test_knn_long_lists(cw, orc, k):
    """kNeighbors above 63 (the reference has no limit on meanK): no main pass, one tree search per query with the k+1
    distances in 4 / 8 / 16 registers per lane -- the same exact distances, the same summation order."""
    pts = synthetic.add_outliers(synthetic.camera_cloud(6000, seed=k), 0.02, seed=k)
    assert np.array_equal(cw.util.knn_mean_distances(upload(cw, pts, cellsize=0.008), k), orc.knn_mean_distances(pts, k))


def test_remove_outliers_long_lists(cw, orc):
    from parity_helpers import per_tile_check
    pts = synthetic.camera_cloud(30000, seed=17)
    for k in (100, 300):
        want, _ = orc.remove_outliers(pts, k, 1.0, False)
        got = download(cw.cwipc_remove_outliers(upload(cw, pts), k, 1.0, False))
        if not np.array_equal(got, want):
            keepmask_check(pts, got, orc.knn_mean_distances(pts, k), k, 1.0)
    per_tile_check(orc, pts, download(cw.cwipc_remove_outliers(upload(cw, pts), 100, 1.0, True)), 100, 1.0)
    cw.cwipc_log_configure(cw.CWIPC_LOG_LEVEL_NONE, lambda level, msg: None)
    try:   # beyond the longest list the call is refused, loudly
        assert not cw.util.cwipc_util_dll_load().cwipc_remove_outliers(upload(cw, pts).as_cwipc_p(), 512, 1.0, False)
    finally:
        cw.cwipc_log_configure(cw.CWIPC_LOG_LEVEL_WARNING, None)


@pytest.mark.parametrize("n", [2, 3, 31, 32, 33, 64, 65, 1000])
def test_knn_tiny_clouds(cw, orc, n):
    pts = random_cloud(n, seed=n, extent=0.1)
    k = min(30, n - 1)
    assert np.array_equal(cw.util.knn_mean_distances(upload(cw, pts), k), orc.knn_mean_distances(pts, k))


def keepmask_check(pts, got, want_d, k, mul):
    """got must equal pts[keep] with keep decided by the oracle's distances, except within 1e-6 of the threshold."""
    d = want_d.astype(np.float64)
    n = len(d)
    s, sq = d.sum(), (want_d * want_d).astype(np.float64).sum()
    thr = s / n + mul * np.sqrt((sq - s * s / n) / (n - 1))
    sure_keep = d <= thr * (1 - 1e-6)
    sure_drop = d > thr * (1 + 1e-6)
    # walk both arrays: every sure_keep point must appear, no sure_drop point may
    gi = 0
    for i in range(n):
        if gi < len(got) and got[gi] == pts[i] and not sure_drop[i]:
            gi += 1
        else:
            assert not sure_keep[i], f"point {i} (d={d[i]}, thr={thr}) was dropped"
    assert gi == len(got)


@pytest.mark.parametrize("n,k,mul", [(6400, 30, 1.0), (50000, 30, 1.0), (50000, 8, 2.5), (200000, 30, 0.5)])
def test_remove_outliers_matches_oracle(cw, orc, n, k, mul):
    pts = synthetic.camera_cloud(n, seed=n % 71)
    want, thr = orc.remove_outliers(pts, k, mul, False)
    out = cw.cwipc_remove_outliers(upload(cw, pts, timestamp=11, cellsize=0.003), k, mul, False)
    assert out.timestamp() == 11 and out.cellsize() == np.float32(0.003)
    got = download(out)
    if not np.array_equal(got, want):  # only threshold ties may differ
        keepmask_check(pts, got, orc.knn_mean_distances(pts, k), k, mul)
    assert 0 < len(got) < n


def test_remove_outliers_per_tile_matches_oracle(cw, orc):
    from parity_helpers import per_tile_check
    pts = synthetic.camera_cloud(80000, seed=13)
    got = download(cw.cwipc_remove_outliers(upload(cw, pts), 30, 1.0, True))
    per_tile_check(orc, pts, got, 30, 1.0)
    # tile 0 present: the whole cloud is processed again as its own group (SURVEY.md finding 3)
    pts["tile"][5] = 0
    got = download(cw.cwipc_remove_outliers(upload(cw, pts), 30, 1.0, True))
    assert len(got) > len(pts)
    per_tile_check(orc, pts, got, 30, 1.0)


def test_remove_outliers_edge_cases(cw):
    cw.cwipc_log_configure(cw.CWIPC_LOG_LEVEL_NONE, lambda level, msg: None)
    try:
        assert cw.cwipc_remove_outliers(cw.cwipc_from_points([], 0), 30, 1.0, True).count() == 0
        assert cw.cwipc_remove_outliers(cw.cwipc_from_points([], 0), 30, 1.0, False).count() == 0
        few = random_cloud(20)
        assert np.array_equal(download(cw.cwipc_remove_outliers(upload(cw, few), 30, 1.0, False)), few)  # n <= k: keep all
        assert not cw.util.cwipc_util_dll_load().cwipc_remove_outliers(None, 30, 1.0, False)
        same = np.zeros(500, DT)  # all points identical: every distance 0, nothing exceeds the threshold
        assert cw.cwipc_remove_outliers(upload(cw, same), 30, 1.0, False).count() == 500
    finally:
        cw.cwipc_log_configure(cw.CWIPC_LOG_LEVEL_WARNING, None)


def test_remove_outliers_reference_property(cw):
    """python/test_cwipc_util.py:528-541"""
    gen = cw.cwipc_synthetic()
    gen.start()
    pc = gen.get()
    n = len(pc.get_points())
    m = len(cw.cwipc_remove_outliers(pc, 30, 1.0, True).get_points())
    assert 0 < m < n
    gen.free()


# ======================================================================================================
# chain, golden fixtures, full-size properties
# ======================================================================================================
def test_chain_config3_matches_oracle(cw, orc):
    """BASELINE config 3: tilefilter(1) -> downsample(0.005) -> remove_outliers(30, 1.0, False), device-resident."""
    n = 1414 * 1414
    pts = synthetic.camera_cloud(n, seed=3)
    pc = upload(cw, pts, cellsize=synthetic.cellsize_of(n))
    a = cw.cwipc_tilefilter(pc, 1)
    b = cw.cwipc_downsample(a, 0.005)
    c = cw.cwipc_remove_outliers(b, 30, 1.0, False)
    oa = orc.tilefilter(pts, 1)
    ob, cs, _, _ = orc.downsample(oa, 0.005, synthetic.cellsize_of(n))
    assert np.array_equal(download(a), oa)
    gb = download(b)
    assert_points_close(gb, ob, cs)
    # the outlier stage sees the GPU's own centroids: compare against the oracle run on the same buffer
    oc, _ = orc.remove_outliers(gb, 30, 1.0, False)
    gc = download(c)
    if not np.array_equal(gc, oc):
        keepmask_check(gb, gc, orc.knn_mean_distances(gb, 30), 30, 1.0)
    assert c.cellsize() == np.float32(cs)


def test_golden_fixtures(cw):
    g = np.load(GOLDEN)
    view = lambda name: g[name].view(DT).reshape(-1)
    pts = view("points")
    pc = upload(cw, pts)
    assert np.array_equal(download(cw.cwipc_tilefilter(pc, 4)), view("tilefilter_4"))
    assert_points_close(download(cw.cwipc_downsample(pc, 0.06)), view("ds_pos"), 0.06)
    assert_points_close(download(cw.cwipc_downsample(pc, -0.06)), view("ds_neg"), 0.06)
    assert np.array_equal(cw.util.knn_mean_distances(pc, 30), g["knn30"])
    assert np.array_equal(download(cw.cwipc_remove_outliers(pc, 30, 1.0, False)), view("sor_all"))
    assert np.array_equal(download(cw.cwipc_remove_outliers(pc, 30, 1.0, True)), view("sor_pertile"))


def test_full_size_properties_8m(cw):
    """BASELINE config 4 size (2828^2 points): checks that need no oracle."""
    n = 2828 * 2828
    pts = synthetic.camera_cloud(n, seed=4, noise=0.0005)
    pc = upload(cw, pts, cellsize=synthetic.cellsize_of(n))
    # tilefilter partitions the cloud
    total = sum(cw.cwipc_tilefilter(pc, t).count() for t in (1, 2, 4, 8))
    assert total == n
    for voxel in (0.002, 0.05):
        out = cw.cwipc_downsample(pc, -voxel)
        got = download(out)
        inv = np.float32(1.0) / np.float32(voxel)
        vox = np.stack([np.floor(pts[a] * inv) for a in "xyz"], axis=1).astype(np.int64)
        uniq = np.unique(vox, axis=0)
        assert len(got) == len(uniq)                              # one output per occupied voxel
        gv = np.stack([np.floor(got[a].astype(np.float64) / voxel) for a in "xyz"], axis=1).astype(np.int64)
        lin = (gv[:, 2] * 1000003 + gv[:, 1]) * 1000003 + gv[:, 0]
        assert np.all(np.diff(lin) > 0) or np.mean(np.diff(lin) > 0) > 0.999  # sorted by (z, y, x) (centroids on a face may round across)
        assert np.bitwise_or.reduce(got["tile"]) == 15
        # downsampling again at the same size is the identity on the voxel set (idempotence)
        again = cw.cwipc_downsample(out, -voxel)
        assert abs(again.count() - out.count()) <= out.count() * 1e-3
        # octree-split mode emits at least as many points, all voxels still covered
        split = cw.cwipc_downsample(pc, voxel)
        assert split.count() >= out.count()
    # outlier removal on the 0.002 voxelisation: keeps most, drops some, preserves order (subsequence)
    ds = cw.cwipc_downsample(pc, 0.002)
    sor = cw.cwipc_remove_outliers(ds, 30, 1.0, False)
    a, b = download(ds), download(sor)
    assert 0.5 * len(a) < len(b) < len(a)
    va = a.view(np.dtype((np.void, 16)))
    vb = b.view(np.dtype((np.void, 16)))
    pos = np.flatnonzero(np.isin(va, vb))
    assert len(pos) >= len(b)


# ======================================================================================================
# building blocks: radix sort (both paths), workspace hygiene, concurrent callers
# ======================================================================================================
@pytest.mark.parametrize("n,begin,end", [(1, 3, 20), (2, 0, 1), (4096, 20, 45), (4097, 20, 38), (100000, 17, 42), (500000, 21, 30), (606209, 24, 51),
                                          (700000, 20, 45), (3000000, 22, 49), (3000000, 0, 64), (50000, 16, 25), (50000, 16, 34),
                                          (32768, 16, 41), (32769, 16, 41), (98304, 17, 35), (98305, 17, 35), (12289, 0, 9), (70001, 30, 31)])
def test_radix_sort_is_a_stable_sort_on_the_bit_range(cw, n, begin, end):
    """<= 98304 words: one thread-block cluster, keys in distributed shared memory; <= 148 tiles of 4096 words: the one-launch
    cooperative kernel; larger inputs: onesweep."""
    rng = np.random.default_rng(n + begin)
    words = rng.integers(0, 2**63, n, dtype=np.uint64) * np.uint64(2) + rng.integers(0, 2, n, dtype=np.uint64)
    if n > 10:
        words[: n // 3] &= np.uint64(0xFFFFFFFFFF)          # clustered high digits, as spatial keys are
    got = cw.util.sort_u64(words, begin, end)
    width = end - begin
    field = (words >> np.uint64(begin)) & np.uint64((1 << width) - 1 if width < 64 else 0xFFFFFFFFFFFFFFFF)
    want = words[np.argsort(field, kind="stable")]
    assert np.array_equal(got, want)


def test_downsample_heavy_voxels_and_contended_atomics(cw, orc):
    """Hundreds of thousands of unordered points per voxel: every atomic of a warp lands on a handful of slots."""
    pts = random_cloud(1500000, seed=3, extent=0.06)
    for voxel in (0.05, -0.05):
        d = cw.cwipc_downsample(upload(cw, pts), voxel)
        want, cs, _, counts = orc.downsample(pts, voxel, 0.0, want_keys=False) if False else orc.downsample(pts, voxel, 0.0)
        assert_points_close(download(d), want, cs)
    assert d.count() <= 64


def test_downsample_recovers_after_a_failed_call(cw, orc):
    """A call that fails half way (coordinate out of range) must not leave the thread's hash workspace dirty."""
    pts = synthetic.camera_cloud(50000, seed=4)
    good, cs, _, _ = orc.downsample(pts, 0.01, 0.0)
    assert_points_close(download(cw.cwipc_downsample(upload(cw, pts), 0.01)), good, cs)
    bad = pts.copy()
    bad["x"][1234] = 3.0e7
    lib = cw.util.cwipc_util_dll_load()
    assert not lib.cwipc_downsample(upload(cw, bad).as_cwipc_p(), 0.01)      # NULL + ERROR log
    for _ in range(2):
        assert_points_close(download(cw.cwipc_downsample(upload(cw, pts), 0.01)), good, cs)


def test_concurrent_callers_get_the_sequential_results(cw):
    """ctypes drops the GIL: 8 threads drive the GPU at once, each on its own stream and workspace."""
    import threading
    clouds = [synthetic.camera_cloud(60000 + 997 * i, seed=40 + i) for i in range(8)]

    def chain(p):
        pc = upload(cw, p, cellsize=0.002)
        return download(cw.cwipc_remove_outliers(cw.cwipc_downsample(pc, 0.008), 20, 1.0, False))

    want = [chain(p) for p in clouds]
    got = [None] * len(clouds)
    errors = []

    def worker(i):
        try:
            for _ in range(3):
                got[i] = chain(clouds[i])
        except Exception as e:  # pragma: no cover
            errors.append(e)

    threads = [threading.Thread(target=worker, args=(i,)) for i in range(len(clouds))]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    assert not errors
    for g, w in zip(got, want):
        assert np.array_equal(g, w)


def test_two_devices_in_one_process(cw):
    """One process, one thread per GPU (DESIGN.md section 7): clouds are created, filtered and freed on device 0 and
    device 1 alternately, so that events and pooled memory released on one device are never reused on the other
    (ADVICE r01: the event pool used to be process-global)."""
    import threading
    if cw.cuda_device_count() < 2:
        pytest.skip("needs two GPUs")
    clouds = [synthetic.camera_cloud(50000 + 1000 * i, seed=60 + i) for i in range(4)]

    def chain(p):
        pc = upload(cw, p, cellsize=0.002)
        return download(cw.cwipc_remove_outliers(cw.cwipc_downsample(pc, 0.008), 20, 1.0, False))

    cw.cuda_set_device(0)
    want = [chain(p) for p in clouds]
    errors, got = [], {}

    def worker(dev):
        try:
            cw.cuda_set_device(dev)
            for rep in range(6):
                for i, p in enumerate(clouds):
                    got[(dev, i)] = chain(p)
        except Exception as e:  # pragma: no cover
            errors.append(e)

    threads = [threading.Thread(target=worker, args=(d,)) for d in (0, 1)]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    assert not errors, errors
    for (dev, i), g in got.items():
        assert np.array_equal(g, want[i]), (dev, i)
    # a cloud of device 1 joined to one of device 0 (peer copy), then freed from the other thread's device
    cw.cuda_set_device(1)
    b = upload(cw, clouds[1])
    cw.cuda_set_device(0)
    a = upload(cw, clouds[0])
    j = cw.cwipc_join(a, b)
    assert np.array_equal(download(j), np.concatenate([clouds[0], clouds[1]]))
    b.free()
    a.free()
    assert cw.util.cwipc_util_dll_load().cwipc_cuda_trim() == 0


@pytest.mark.parametrize("path", ["twopass", "generic", "smalltable"])
def test_downsample_every_internal_path_matches_oracle(cw, orc, path):
    """The fused single pass is the default; the two-pass path (leaf tables of the final octree box), the generic path
    (double arithmetic per run, used when a cloud spans more than 32 leaves per axis) and the table-overflow retry are
    forced here through CWIPC_CUDA_DS_PATH and must give the same results."""
    clouds = [(synthetic.camera_cloud(250000, seed=3), 0.004, 0.0), (synthetic.synthetic_cloud(160000), 0.005, 0.005), (random_cloud(120000, seed=9, extent=0.4), 0.013, 0.0)]
    os.environ["CWIPC_CUDA_DS_PATH"] = path
    try:
        for pts, voxel, pc_cellsize in clouds:
            for v in (voxel, -voxel):
                want, cs, keys6, counts = orc.downsample(pts, v, pc_cellsize, want_keys=True)
                got = download(cw.cwipc_downsample(upload(cw, pts, cellsize=pc_cellsize), v))
                assert_points_close(got, want, cs)
    finally:
        del os.environ["CWIPC_CUDA_DS_PATH"]


def test_downsample_far_outlier_and_wide_clouds(cw, orc):
    """One distant noise point on a fine grid (the octree grows deep, most points lie outside the leaf tables of the first
    point), and a cloud more than 32 leaves wide: both stay correct (ADVICE r01: the sort word used to overflow here)."""
    pts = synthetic.camera_cloud(100000, seed=21)
    pts["x"][777], pts["y"][777], pts["z"][777] = 9.0, -7.5, 3.25
    for voxel in (0.002, 0.004):
        want, cs, _, _ = orc.downsample(pts, voxel, 0.0)
        assert_points_close(download(cw.cwipc_downsample(upload(cw, pts), voxel)), want, cs)
    wide = random_cloud(200000, seed=12, extent=3.0)
    want, cs, _, _ = orc.downsample(wide, 0.002, 0.0)       # 6 m / (64 * 2 mm) = 47 leaves per axis
    assert_points_close(download(cw.cwipc_downsample(upload(cw, wide), 0.002)), want, cs)


def test_downsample_first_point_on_coordinate_planes(cw, orc):
    """The octree is anchored on the first point: with p0 = (0, 0, z) leaf faces lie exactly on the planes x = 0 and y = 0,
    where whole rings of the clean synthetic cloud sit, and floats next to zero vanish in (double)x - min.  Includes
    denormal and 1e-20-sized coordinates, which the single-pass path must hand to the two-pass path."""
    pts = synthetic.simulate_cameras(synthetic.synthetic_cloud(250000), 4)
    for voxel in (0.005, 0.01, 0.05):
        want, cs, _, counts = orc.downsample(pts, voxel, 0.0)
        assert_points_close(download(cw.cwipc_downsample(upload(cw, pts), voxel)), want, cs)
    tiny = pts.copy()
    tiny["x"][1000:1010] = [1e-20, -1e-20, 1e-30, -1e-38, 1e-44, -1e-45, 3e-17, -3e-17, 1e-12, -1e-12]
    tiny["y"][2000:2004] = [1e-20, 1e-41, -1e-20, 2e-17]
    for voxel in (0.005, 0.02):
        want, cs, _, counts = orc.downsample(tiny, voxel, 0.0)
        assert_points_close(download(cw.cwipc_downsample(upload(cw, tiny), voxel)), want, cs)


@pytest.mark.parametrize("npoints,angle", [(160000, 0.0), (160000, 1.7), (250000, 0.33), (1000000, 12.5), (7, 0.1)])
def test_synthetic_source_generates_on_the_device(cw, npoints, angle):
    """ref: src/cwipc_synthetic.cpp:182-222.  The source makes its points in HBM from 3 * sqrt(N) host-computed libm values
    (no host-to-device copy of points); the bytes equal the host generator's, which stays reachable as the checker."""
    gen = cw.cwipc_synthetic(0, npoints)
    assert gen.start()
    side = int(np.sqrt(npoints))
    want = gen.host_generate(angle, side * side)
    pc = gen.get()
    assert pc.count() == side * side and pc.cellsize() == np.float32(2.0 / side)
    got = download(pc)
    for a in "xyz":   # geometry: bit-identical by construction (the host's own sin / cos / pow values, expanded on the device)
        assert np.array_equal(got[a].view(np.uint32), want[a].view(np.uint32)), a
    assert np.array_equal(got["tile"], want["tile"])
    for c in "rgb":   # colours use the device's double-precision sin (2 ulp): equal except, at worst, an LSB once in ~1e7 values
        diff = np.abs(got[c].astype(int) - want[c].astype(int))
        assert diff.max(initial=0) <= 1 and np.count_nonzero(diff) <= 1
    gen.free()

@pytest.mark.parametrize("env", [
    {"CWIPC_CUDA_KNN_SECOND_FROM_N": "0"},                                                                   # the second scan on small clouds too
    {"CWIPC_CUDA_KNN_SECOND_FROM_N": "0", "CWIPC_CUDA_KNN_RC_FAR": "3.5", "CWIPC_CUDA_KNN_SECOND_MAX": "100000", "CWIPC_CUDA_KNN_SECOND_MIN": "1"},  # every open query, boxes larger than the range list
    {"CWIPC_CUDA_KNN_RC_FAR": "0"},                                                                          # never
    {"CWIPC_CUDA_KNN_SECOND_FROM_N": "0", "CWIPC_CUDA_KNN_PITCH": "0.6"},                                     # small pitch: most queries open
    {"CWIPC_CUDA_KNN_RC_FAR": "0", "CWIPC_CUDA_KNN_PITCH": "0.4"},                                            # ... all of them through the tree search, started near the query
    {"CWIPC_CUDA_KNN_RC_FAR": "0", "CWIPC_CUDA_KNN_PITCH": "0.4", "CWIPC_CUDA_KNN_FAR_START": "0"},           # ... and started at the root
])
def test_knn_passes_split_the_work_not_the_result(cw, orc, env):
    """Main pass, second scan (knn_second_kernel) and tree search (knn_far_kernel) are three ways to the same exact
    k+1 smallest distances; the tunables only move queries between them.  A child process runs with the tunables forced
    (they are read once per process) and must reproduce the oracle's distances bit for bit, whole cloud and per tile."""
    import subprocess
    code = ("import sys, numpy as np; sys.path.insert(0, %r); import cwipc_util_b200 as cw; from cwipc_util_b200 import synthetic\n"
            "out = []\n"
            "for n, seed in ((90000, 31), (200000, 32)):\n"
            "    pts = synthetic.camera_cloud(n, seed=seed, noise=0.004)\n"
            "    pc = cw.cwipc_from_numpy_array(pts, 1); pc._set_cellsize(synthetic.cellsize_of(n))\n"
            "    out.append(cw.util.knn_mean_distances(pc, 30).astype(np.float32).tobytes())\n"
            "    out.append(cw.cwipc_remove_outliers(pc, 12, 1.5, True).get_numpy_array().tobytes())\n"
            "sys.stdout.buffer.write(b''.join(out))" % REPO)
    raw = subprocess.run([sys.executable, "-c", code], env=dict(os.environ, **env), capture_output=True, check=True, timeout=900).stdout
    pos = 0
    for n, seed in ((90000, 31), (200000, 32)):
        pts = synthetic.camera_cloud(n, seed=seed, noise=0.004)
        d = np.frombuffer(raw[pos:pos + 4 * len(pts)], np.float32)   # (the generator rounds n to a square)
        pos += 4 * len(pts)
        assert np.array_equal(d, orc.knn_mean_distances(pts, 30))
        want = download(cw.cwipc_remove_outliers(upload(cw, pts, cellsize=synthetic.cellsize_of(n)), 12, 1.5, True))
        got = np.frombuffer(raw[pos:pos + want.nbytes], DT)
        pos += want.nbytes
        assert np.array_equal(got, want)
    assert pos == len(raw)
