"""cwipc_cuda_estimate_normals and cwipc_cuda_icp_point_to_plane on the device, against tests/icp_plane_reference.py.

Neighbourhoods are chosen by exact float32 keys on both sides, so the points with a zero normal must be the reference's
exactly; the normals themselves come from differently ordered double sums and a different eigen-solver, so they are compared
where the smallest eigenvalue is well separated.  The first evaluation of a call is cwipc_icp's, bit for bit; later steps are
compared within tolerances, as in tests/test_gpu_icp.py.
"""
import ctypes
import json
import threading

import numpy as np
import pytest
from scipy.spatial.transform import Rotation

import icp_plane_reference as pref
from cwipc_util_b200 import synthetic

DT = synthetic.cwipc_point_numpy_dtype
pytestmark = pytest.mark.gpu


def pose(seed, degrees, metres, centre=(0.0, 0.0, 0.0)):
    """A seeded rigid motion: a rotation of `degrees` about an axis through `centre`, then a translation of `metres`."""
    rng = np.random.default_rng(seed)
    axis = rng.normal(size=3)
    R = Rotation.from_rotvec(np.radians(degrees) * axis / np.linalg.norm(axis)).as_matrix()
    t = rng.normal(size=3)
    c = np.asarray(centre, np.float64)
    T = np.eye(4)
    T[:3, :3] = R
    T[:3, 3] = c - R @ c + metres * t / np.linalg.norm(t)
    return T


def from_xyz(xyz, tile=1):
    pts = np.zeros(len(xyz), DT)
    for i, a in enumerate("xyz"):
        pts[a] = xyz[:, i]
    pts["tile"] = tile
    return pts


def xyz(pc):
    return pref.xyz32(pc.get_numpy_array().copy())


def camera_pair(cw, n=1000000, seed=1, offset=0.0):
    """Camera 1 of the jittered 4-camera cloud, and cameras 2|4|8 of it, as registration pairs them."""
    pts = synthetic.camera_cloud(n, seed=seed)
    if offset:
        for a in "xyz":
            pts[a] = (pts[a].astype(np.float64) + offset).astype(np.float32)
    pc = cw.cwipc_from_numpy_array(pts, 1)
    return pc, cw.cwipc_tilefilter(pc, 1), cw.cwipc_tilefilter_masked(pc, ~1 & 0xff)


def sheet(n, seed, offset=0.0):
    """A wavy 2 m x 2 m sheet: no motion slides it along itself, so ICP can recover every degree of freedom."""
    rng = np.random.default_rng(seed)
    u, v = rng.uniform(-1, 1, n), rng.uniform(-1, 1, n)
    return (np.stack([u, 0.3 * np.sin(3 * u) * np.cos(2 * v) + 0.1 * u * v, v], 1) + offset).astype(np.float32)


SPACING = 2.0 ** -6  # every lattice coordinate and every difference of two of them is exact in float32


def lattice(n, seed, spacing=SPACING):
    rng = np.random.default_rng(seed)
    g = np.stack(np.meshgrid(np.arange(n), np.arange(n), np.arange(n), indexing="ij"), -1).reshape(-1, 3)
    return (g[rng.permutation(len(g))] * spacing).astype(np.float32)


def lattice_pair(cw, seed, n=24):
    """A shuffled lattice as the target and lattice points moved half a spacing along x as the source: every source point
    has two nearest target points at the same float32 d2, and every target neighbourhood has ties at its edge."""
    rng = np.random.default_rng(seed)
    target = lattice(n, seed)
    g = np.round(target / np.float32(SPACING)).astype(np.int64)
    src = g[g[:, 0] < n - 1][rng.permutation(int((g[:, 0] < n - 1).sum()))[:4000]]
    source = (src * SPACING).astype(np.float32)
    source[:, 0] = ((src[:, 0] + 0.5) * SPACING).astype(np.float32)
    return cw.cwipc_from_numpy_array(from_xyz(source), 1), cw.cwipc_from_numpy_array(from_xyz(target), 1), source, target


def rot_angle(R):
    return float(np.arccos(np.clip((np.trace(R) - 1.0) / 2.0, -1.0, 1.0)))


def assert_normals_match(got, want):
    zero_got = np.all(got == 0.0, axis=1)
    zero_want = np.all(want.normals == 0.0, axis=1)
    assert np.array_equal(zero_got, zero_want), (int(zero_got.sum()), int(zero_want.sum()))
    assert np.all(np.abs(np.linalg.norm(got[~zero_got].astype(np.float64), axis=1) - 1.0) < 1e-6)
    w = want.eigvals
    clear = ~zero_want & (w[:, 1] - w[:, 0] > 1e-3 * w[:, 2])
    dot = np.abs(np.einsum("na,na->n", got.astype(np.float64), want.normals.astype(np.float64)))
    assert clear.sum() > 0.5 * (~zero_want).sum()
    assert dot[clear].min() >= 1 - 1e-6, dot[clear].min()


# ---- 1. normals ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("offset", [0.0, 1e4])
def test_normals_are_the_reference(cw, offset):
    pts = synthetic.camera_cloud(1000000, seed=1)
    if offset:
        for a in "xyz":
            pts[a] = (pts[a].astype(np.float64) + offset).astype(np.float32)
    raw = cw.cwipc_from_numpy_array(pts, 1)
    for pc, radius in ((raw, 0.01), (cw.cwipc_downsample_pertile(raw, 0.005), 0.02)):
        P = xyz(pc)
        tree = pref.cKDTree(P.astype(np.float64))
        for max_nn in ((3, 8, 30, 32) if offset == 0.0 else (30,)):
            got = cw.cwipc_estimate_normals(pc, radius, max_nn)
            assert got.shape == (len(P), 3) and got.dtype == np.float32
            want = pref.estimate_normals(P, radius, max_nn, tree)
            assert_normals_match(got, want)
            assert np.array_equal(cw.cwipc_estimate_normals(pc, radius, max_nn), got)   # bit-identical on a second run


@pytest.mark.parametrize("max_nn", [3, 8, 30, 32])
def test_normals_on_lattices_with_ties(cw, max_nn):
    """A shuffled square lattice whose points are lifted by 0..3 units of 2^-12 at random: every d2 is exact in float32,
    neighbourhoods end in ties that only the index settles, and which points join changes the normal."""
    for seed, radius in ((1, 1.0 * SPACING), (2, 1.5 * SPACING), (3, 2.0 * SPACING)):
        rng = np.random.default_rng(seed)
        g = np.stack(np.meshgrid(np.arange(60), np.arange(60), indexing="ij"), -1).reshape(-1, 2)
        g = g[rng.permutation(len(g))]
        T = np.c_[g * SPACING, rng.integers(0, 4, len(g)) * 2.0 ** -12].astype(np.float32)
        pc = cw.cwipc_from_numpy_array(from_xyz(T), 1)
        got = cw.cwipc_estimate_normals(pc, radius, max_nn)
        assert_normals_match(got, pref.estimate_normals(T, radius, max_nn))


# ---- 2. evaluation only ----------------------------------------------------------------------------------------------------------
def test_evaluation_only_is_cwipc_icp_bit_for_bit(cw):
    pc, s, t = camera_pair(cw, n=400000, seed=2)
    for seed, d in ((1, 0.05), (2, 0.01), (3, 0.2)):
        init = pose(seed, 3.0, 0.03, centre=xyz(s).mean(0))
        a = cw.cwipc_icp(s, t, d, init=init, max_iterations=0)
        b = cw.cwipc_icp_point_to_plane(s, t, d, 0.01, init=init, max_iterations=0)
        assert b.correspondences == a.correspondences > 0
        assert (b.fitness, b.inlier_rmse, b.iterations) == (a.fitness, a.inlier_rmse, 0)
        assert np.array_equal(b.matrix, init)
    for seed in (1, 2):
        sp, tp, S, T = lattice_pair(cw, seed)
        for d in (SPACING / 2, SPACING * 0.51, 2 * SPACING):
            a = cw.cwipc_icp(sp, tp, d, max_iterations=0)
            b = cw.cwipc_icp_point_to_plane(sp, tp, d, 1.5 * SPACING, max_iterations=0)
            assert (b.correspondences, b.fitness, b.inlier_rmse) == (a.correspondences, a.fitness, a.inlier_rmse)


# ---- 3. one iteration ----------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("max_nn", [8, 30])
def test_one_iteration_matrix_is_the_reference(cw, max_nn):
    pc, s, t = camera_pair(cw, n=400000, seed=2)
    S, T = xyz(s), xyz(t)
    tp = cw.cwipc_from_numpy_array(from_xyz(T), 1)   # a cloud without a stored box: the library's origin is T's box centre
    init = pose(4, 3.0, 0.02, centre=S.mean(0))
    r = cw.cwipc_icp_point_to_plane(s, tp, 0.05, 0.01, init=init, max_iterations=1, relative_fitness=0.0, relative_rmse=0.0, normal_max_nn=max_nn)
    want = pref.icp_point_to_plane(S, T, 0.05, 0.01, init=init, max_iterations=1, relative_fitness=0.0, relative_rmse=0.0, normal_max_nn=max_nn)
    assert r.iterations == want.iterations == 1
    assert np.abs(r.matrix - want.matrix).max() < 1e-10, np.abs(r.matrix - want.matrix).max()


# ---- 4. full runs ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("offset", [0.0, 1e4])
def test_recovers_a_seeded_camera_pose(cw, offset):
    T = sheet(200000, 1, offset)
    camera = T[T[:, 0] < np.float32(offset + 0.3)]
    centre = camera.astype(np.float64).mean(0)
    P = pose(5, 4.0, 0.04, centre=centre)
    tp = cw.cwipc_from_numpy_array(from_xyz(T), 1)
    moved = cw.cwipc_transform(cw.cwipc_from_numpy_array(from_xyz(camera), 1), P)
    r = cw.cwipc_icp_point_to_plane(moved, tp, 0.2, 0.03, max_iterations=60)
    p2p = cw.cwipc_icp(moved, tp, 0.2, max_iterations=60)
    print(f"offset {offset}: point-to-plane {r.iterations} iterations, point-to-point {p2p.iterations}")
    err = r.matrix @ P
    assert rot_angle(err[:3, :3]) < (1e-6 if offset == 0.0 else 1e-5)
    d = r.matrix - np.linalg.inv(P)
    assert np.abs(d[:3, :3] @ centre + d[:3, 3]).max() < 1e-5


# ---- 5. a flat plane --------------------------------------------------------------------------------------------------------------
def test_flat_plane_moves_only_along_its_normal(cw):
    rng = np.random.default_rng(7)
    T = np.c_[rng.uniform(-1, 1, (100000, 2)), np.zeros(100000)].astype(np.float32)
    S = (T[:20000] + np.float32([0.01, -0.02, 0.003])).astype(np.float32)   # slid along the plane and lifted off it
    tp, sp = cw.cwipc_from_numpy_array(from_xyz(T), 1), cw.cwipc_from_numpy_array(from_xyz(S), 1)
    normals = cw.cwipc_estimate_normals(tp, 0.03, 30)
    assert np.all(normals[:, :2] == 0.0) and np.all(np.abs(normals[:, 2]) == 1.0)
    r = cw.cwipc_icp_point_to_plane(sp, tp, 0.05, 0.03)
    M = r.matrix
    assert np.all(np.isfinite(M))
    assert abs(M[2, 3] + 0.003) < 1e-6
    assert max(abs(M[0, 1]), abs(M[1, 0]), abs(M[0, 3]), abs(M[1, 3])) < 1e-12, M


# ---- 6. consistency with cwipc_cuda_transform ---------------------------------------------------------------------------------------
def test_result_is_the_evaluation_of_the_moved_source(cw):
    pc, s, t = camera_pair(cw, n=400000, seed=4)
    init = pose(6, 2.0, 0.02, centre=xyz(s).mean(0))
    r = cw.cwipc_icp_point_to_plane(s, t, 0.05, 0.01, init=init)
    assert r.iterations > 1
    again = cw.cwipc_icp_point_to_plane(cw.cwipc_transform(s, r.matrix), t, 0.05, 0.01, max_iterations=0)
    assert (again.correspondences, again.fitness, again.inlier_rmse) == (r.correspondences, r.fitness, r.inlier_rmse)


# ---- 7. determinism and concurrency -------------------------------------------------------------------------------------------------
def test_repeatable_bit_for_bit_also_from_four_threads(cw):
    pc, s, t = camera_pair(cw, n=400000, seed=5)
    init = pose(7, 3.0, 0.03, centre=xyz(s).mean(0))
    call = lambda: cw.cwipc_icp_point_to_plane(s, t, 0.05, 0.01, init=init)
    key = lambda r: (r.matrix.tobytes(), r.fitness, r.inlier_rmse, r.iterations, r.correspondences)
    first = key(call())
    normals = cw.cwipc_estimate_normals(t, 0.01).tobytes()
    got, failures = [], []

    def worker():
        try:
            for _ in range(3):
                got.append((key(call()), cw.cwipc_estimate_normals(t, 0.01).tobytes()))
        except Exception as e:  # pragma: no cover
            failures.append(e)

    threads = [threading.Thread(target=worker) for _ in range(4)]
    for th in threads:
        th.start()
    for th in threads:
        th.join()
    assert not failures, failures
    assert len(got) == 12 and all(g == (first, normals) for g in got)


# ---- 8. edge cases and errors -------------------------------------------------------------------------------------------------------
def test_edge_cases(cw):
    pc, s, t = camera_pair(cw, n=100000, seed=6)
    empty = cw.cwipc_tilefilter(pc, 200)
    assert empty.count() == 0
    init = pose(8, 1.0, 0.01)
    for a, b in ((empty, t), (s, empty), (empty, empty)):
        r = cw.cwipc_icp_point_to_plane(a, b, 0.05, 0.01, init=init)
        assert (r.correspondences, r.fitness, r.inlier_rmse, r.iterations) == (0, 0.0, 0.0, 0)
        assert np.array_equal(r.matrix, init)
    assert cw.cwipc_estimate_normals(empty, 0.01).shape == (0, 3)
    # a target of fewer than 3 points has only zero normals: every step is the identity and T stays init
    two = cw.cwipc_from_numpy_array(from_xyz(np.float32([[0, 0, 0], [0.001, 0, 0]])), 1)
    assert np.all(cw.cwipc_estimate_normals(two, 0.01) == 0.0)
    near = cw.cwipc_from_numpy_array(from_xyz(np.float32([[0, 0, 0.001], [0.001, 0, 0.001], [0.0005, 0.001, 0.001], [0, 0.002, 0]])), 1)
    r = cw.cwipc_icp_point_to_plane(near, two, 0.05, 0.01, init=init)
    assert r.correspondences == 4 and r.iterations == 1 and np.array_equal(r.matrix, init)
    r = cw.cwipc_icp_point_to_plane(s, s, 0.05, 0.01)
    assert r.fitness == 1.0 and r.inlier_rmse == 0.0 and r.correspondences == s.count()
    assert np.abs(r.matrix - np.eye(4)).max() < 1e-12


def test_invalid_arguments_fail_once_and_leave_the_inputs_usable(cw):
    lib = cw.util.cwipc_util_dll_load()
    base = cw.cwipc_dangling_allocations(False)
    rng = np.random.default_rng(9)
    good = from_xyz(rng.uniform(-1, 1, (20000, 3)).astype(np.float32))
    with_nan, with_inf = good.copy(), good.copy()
    with_nan["y"][123] = np.nan
    with_inf["z"][7] = np.inf
    s = cw.cwipc_from_numpy_array(good, 1)
    t = cw.cwipc_from_numpy_array(good[::2].copy(), 1)
    sn, ti = cw.cwipc_from_numpy_array(with_nan, 1), cw.cwipc_from_numpy_array(with_inf, 1)
    want = cw.cwipc_icp_point_to_plane(s, t, 0.2, 0.2)
    want_n = cw.cwipc_estimate_normals(t, 0.2)
    eye = np.eye(4)
    nan_init, w_init = eye.copy(), eye.copy()
    nan_init[1, 2] = np.nan
    w_init[3, 3] = 2.0
    res = cw.util.cwipc_cuda_icp_result()
    cases = [  # (what, source, target, init, d, iterations, rf, rr, radius, max_nn, result)
        ("d = 0", s, t, None, 0.0, 30, 1e-6, 1e-6, 0.2, 30, True),
        ("d NaN", s, t, None, np.nan, 30, 1e-6, 1e-6, 0.2, 30, True),
        ("iterations < 0", s, t, None, 0.2, -1, 1e-6, 1e-6, 0.2, 30, True),
        ("fitness < 0", s, t, None, 0.2, 30, -1e-6, 1e-6, 0.2, 30, True),
        ("rmse inf", s, t, None, 0.2, 30, 1e-6, np.inf, 0.2, 30, True),
        ("init NaN", s, t, nan_init, 0.2, 30, 1e-6, 1e-6, 0.2, 30, True),
        ("init last row", s, t, w_init, 0.2, 30, 1e-6, 1e-6, 0.2, 30, True),
        ("result NULL", s, t, None, 0.2, 30, 1e-6, 1e-6, 0.2, 30, False),
        ("radius 0", s, t, None, 0.2, 30, 1e-6, 1e-6, 0.0, 30, True),
        ("radius < 0", s, t, None, 0.2, 30, 1e-6, 1e-6, -0.1, 30, True),
        ("radius NaN", s, t, None, 0.2, 30, 1e-6, 1e-6, np.nan, 30, True),
        ("radius inf", s, t, None, 0.2, 30, 1e-6, 1e-6, np.inf, 30, True),
        ("max_nn 2", s, t, None, 0.2, 30, 1e-6, 1e-6, 0.2, 2, True),
        ("max_nn 33", s, t, None, 0.2, 30, 1e-6, 1e-6, 0.2, 33, True),
        ("NaN in the source", sn, t, None, 0.2, 30, 1e-6, 1e-6, 0.2, 30, True),
        ("inf in the target", s, ti, None, 0.2, 30, 1e-6, 1e-6, 0.2, 30, True),
        ("NaN in the target", s, sn, None, 0.2, 30, 1e-6, 1e-6, 0.2, 30, True),
    ]
    out = np.zeros((20000, 3), np.float32)
    ncases = [  # (what, cloud, radius, max_nn, buffer, nfloats)
        ("radius 0", t, 0.0, 30, out.ctypes.data, out.size),
        ("radius NaN", t, np.nan, 30, out.ctypes.data, out.size),
        ("radius inf", t, np.inf, 30, out.ctypes.data, out.size),
        ("max_nn 2", t, 0.2, 2, out.ctypes.data, out.size),
        ("max_nn 33", t, 0.2, 33, out.ctypes.data, out.size),
        ("NULL buffer", t, 0.2, 30, None, out.size),
        ("short buffer", t, 0.2, 30, out.ctypes.data, 3 * t.count() - 1),
        ("NaN in the cloud", sn, 0.2, 30, out.ctypes.data, out.size),
        ("inf in the cloud", ti, 0.2, 30, out.ctypes.data, out.size),
    ]
    seen = []
    cw.cwipc_log_configure(cw.CWIPC_LOG_LEVEL_WARNING, lambda level, msg: seen.append((level, msg.decode())))
    try:
        for what, a, b, init, d, n, rf, rr, radius, max_nn, has_result in cases:
            seen.clear()
            m = None if init is None else np.ascontiguousarray(init)
            rv = lib.cwipc_cuda_icp_point_to_plane(a.as_cwipc_p(), b.as_cwipc_p(), None if m is None else m.ctypes.data, d, n, rf, rr, radius, max_nn,
                                                   ctypes.byref(res) if has_result else None)
            assert rv == -1, what
            assert len(seen) == 1 and seen[0][0] == cw.CWIPC_LOG_LEVEL_ERROR and seen[0][1].startswith("cwipc_cuda_icp_point_to_plane: "), (what, seen)
        for what, pc, radius, max_nn, buf, nfloats in ncases:
            seen.clear()
            rv = lib.cwipc_cuda_estimate_normals(pc.as_cwipc_p(), radius, max_nn, buf, nfloats)
            assert rv == -1, what
            assert len(seen) == 1 and seen[0][0] == cw.CWIPC_LOG_LEVEL_ERROR and seen[0][1].startswith("cwipc_cuda_estimate_normals: "), (what, seen)
        for a, b in ((None, t), (s, None), (None, None)):
            seen.clear()
            rv = lib.cwipc_cuda_icp_point_to_plane(a.as_cwipc_p() if a else None, b.as_cwipc_p() if b else None, None, -1.0, -1, -1.0, -1.0, -1.0, 0, None)
            assert rv == -1 and not seen
        seen.clear()
        assert lib.cwipc_cuda_estimate_normals(None, -1.0, 0, None, 0) == -1 and not seen
    finally:
        cw.cwipc_log_configure(cw.CWIPC_LOG_LEVEL_WARNING, None)
    with pytest.raises(cw.CwipcError):
        cw.cwipc_icp_point_to_plane(s, t, 0.2, -1.0)
    with pytest.raises(cw.CwipcError):
        cw.cwipc_estimate_normals(t, 0.2, max_nn=40)
    for pc, pts in ((s, good), (t, good[::2]), (sn, with_nan), (ti, with_inf)):
        assert pc.get_numpy_array().tobytes() == pts.tobytes()
    again = cw.cwipc_icp_point_to_plane(s, t, 0.2, 0.2)
    assert (again.matrix.tobytes(), again.fitness, again.inlier_rmse, again.correspondences) == (want.matrix.tobytes(), want.fitness, want.inlier_rmse, want.correspondences)
    assert np.array_equal(cw.cwipc_estimate_normals(t, 0.2), want_n)
    for pc in (s, t, sn, ti):
        pc.free()
    assert cw.cwipc_dangling_allocations(False) == base


def test_clouds_on_two_devices(cw):
    if cw.cuda_device_count() < 2:
        pytest.skip("needs two GPUs")
    pts = from_xyz(np.random.default_rng(10).uniform(-1, 1, (5000, 3)).astype(np.float32))
    s = cw.cwipc_from_numpy_array(pts, 1)
    cw.cuda_set_device(1)
    try:
        t = cw.cwipc_from_numpy_array(pts, 1)
    finally:
        cw.cuda_set_device(0)
    seen = []
    cw.cwipc_log_configure(cw.CWIPC_LOG_LEVEL_WARNING, lambda level, msg: seen.append((level, msg.decode())))
    try:
        res = cw.util.cwipc_cuda_icp_result()
        rv = cw.util.cwipc_util_dll_load().cwipc_cuda_icp_point_to_plane(s.as_cwipc_p(), t.as_cwipc_p(), None, 0.05, 30, 1e-6, 1e-6, 0.1, 30, ctypes.byref(res))
    finally:
        cw.cwipc_log_configure(cw.CWIPC_LOG_LEVEL_WARNING, None)
    assert rv == -1
    assert len(seen) == 1 and seen[0][0] == cw.CWIPC_LOG_LEVEL_ERROR and seen[0][1].startswith("cwipc_cuda_icp_point_to_plane: "), seen
    assert cw.cwipc_icp_point_to_plane(s, s, 0.05, 0.1).fitness == 1.0 and cw.cwipc_icp_point_to_plane(t, t, 0.05, 0.1).fitness == 1.0
    assert np.array_equal(cw.cwipc_estimate_normals(s, 0.1), cw.cwipc_estimate_normals(t, 0.1))


# ---- 9. launches and leaks ----------------------------------------------------------------------------------------------------------
def test_index_and_normals_are_built_once_per_call_and_nothing_leaks(cw):
    lib = cw.util.cwipc_util_dll_load()
    base = cw.cwipc_dangling_allocations(False)
    pc, s, t = camera_pair(cw, n=200000, seed=11)
    init = pose(12, 3.0, 0.03, centre=xyz(s).mean(0))
    launches = []
    for n in (0, 1, 2, 5):
        lib.cwipc_cuda_profile_reset()
        lib.cwipc_cuda_profile_enable(1)
        before = cw.cuda_kernel_launches()
        r = cw.cwipc_icp_point_to_plane(s, t, 0.05, 0.01, init=init, max_iterations=n, relative_fitness=0.0, relative_rmse=0.0)
        launches.append(cw.cuda_kernel_launches() - before)
        lib.cwipc_cuda_profile_enable(0)
        need = lib.cwipc_cuda_profile_report(None, 0)
        buf = ctypes.create_string_buffer(need)
        lib.cwipc_cuda_profile_report(buf, need)
        prof = json.loads(buf.value.decode())
        assert r.iterations == n
        assert prof["knn_keygen_kernel"]["launches"] == 1 and prof["knn_layout_kernel"]["launches"] == 1
        assert prof["icp_normals_kernel"]["launches"] == 1
        assert prof["icp_plane_match_kernel"]["launches"] == prof["icp_plane_reduce_kernel"]["launches"] == n + 1
        assert "icp_match_kernel" not in prof
    per = launches[1] - launches[0]
    assert per == 2 and launches[2] - launches[0] == 2 * per and launches[3] - launches[0] == 5 * per, launches
    for c in (pc, s, t):
        c.free()
    assert cw.cwipc_dangling_allocations(False) == base
