"""cwipc_cuda_icp: point-to-point ICP on the device, against the numpy/cKDTree loop of tests/icp_reference.py.

The first evaluation of a call moves the source by the same double `init` on both sides with the same arithmetic, so its
correspondences must be the reference's exactly.  Later evaluations move the source by a matrix that the library solved
from fixed-order double sums and the reference from an SVD: the two matrices differ in the last bits, a moved point can
then round to the neighbouring float, and those iterations are compared within tolerances.
"""
import ctypes
import threading

import numpy as np
import pytest
from scipy.spatial.transform import Rotation

import icp_reference as ref
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


def records(pc):
    return pc.get_numpy_array().copy()


def from_xyz(xyz, tile=1):
    pts = np.zeros(len(xyz), DT)
    for i, a in enumerate("xyz"):
        pts[a] = xyz[:, i]
    pts["tile"] = tile
    return pts


def camera_pair(cw, n=1000000, seed=1, offset=0.0):
    """Camera 1 of the jittered 4-camera cloud, and cameras 2|4|8 of it, as registration pairs them."""
    pts = synthetic.camera_cloud(n, seed=seed)
    if offset:
        for a in "xyz":
            pts[a] = (pts[a].astype(np.float64) + offset).astype(np.float32)
    pc = cw.cwipc_from_numpy_array(pts, 1)
    return pc, cw.cwipc_tilefilter(pc, 1), cw.cwipc_tilefilter_masked(pc, ~1 & 0xff)


SPACING = 2.0 ** -6  # every lattice coordinate and every difference of two of them is exact in float32


def lattice_pair(cw, seed, n=24, spacing=SPACING):
    """A shuffled lattice as the target and, as the source, a sample of lattice points moved half a spacing along x: every
    source point has two nearest target points at exactly the same float32 d2, and the lower index decides which one."""
    rng = np.random.default_rng(seed)
    g = np.stack(np.meshgrid(np.arange(n), np.arange(n), np.arange(n), indexing="ij"), -1).reshape(-1, 3)
    target = (g[rng.permutation(len(g))] * spacing).astype(np.float32)
    src = g[g[:, 0] < n - 1][rng.permutation(len(g) - n * n)[: 4000]]
    source = (src * spacing).astype(np.float32)
    source[:, 0] = ((src[:, 0] + 0.5) * spacing).astype(np.float32)
    tp = cw.cwipc_from_numpy_array(from_xyz(target), 1)
    sp = cw.cwipc_from_numpy_array(from_xyz(source), 1)
    # the x neighbours of every source point really are equally far in float32
    m = ref.Matcher(target)
    idx, d2 = m.nearest(source, ref.limit32(spacing))
    assert np.all(idx >= 0)
    return sp, tp, source, target


def xyz(pc):
    return ref.xyz32(records(pc))


def rot_angle(R):
    return float(np.arccos(np.clip((np.trace(R) - 1.0) / 2.0, -1.0, 1.0)))


# ---- 1. evaluation only -------------------------------------------------------------------------------------------------
def test_evaluation_only_is_the_reference_exactly(cw):
    pc, s, t = camera_pair(cw)
    S, T = xyz(s), xyz(t)
    m = ref.Matcher(T)
    for seed, d in ((1, 0.05), (2, 0.01), (3, 0.2)):
        init = pose(seed, 3.0, 0.03, centre=S.mean(0))
        r = cw.cwipc_icp(s, t, d, init=init, max_iterations=0)
        e = ref.evaluate(S, m, init, d)
        assert r.iterations == 0 and np.array_equal(r.matrix, init)
        assert r.correspondences == e.correspondences > 0
        assert r.fitness == e.fitness
        assert abs(r.inlier_rmse - e.inlier_rmse) <= 1e-12 * e.inlier_rmse


@pytest.mark.parametrize("seed", [1, 2])
def test_evaluation_only_with_ties(cw, seed):
    sp, tp, S, T = lattice_pair(cw, seed)
    m = ref.Matcher(T)
    for d in (SPACING / 2, SPACING * 0.51, 2 * SPACING):
        r = cw.cwipc_icp(sp, tp, d, max_iterations=0)
        e = ref.evaluate(S, m, np.eye(4), d)
        assert r.correspondences == e.correspondences
        assert r.fitness == e.fitness
        assert abs(r.inlier_rmse - e.inlier_rmse) <= 1e-12 * e.inlier_rmse


# ---- 2. one iteration ---------------------------------------------------------------------------------------------------
def test_one_iteration_matrix_is_the_reference(cw):
    pc, s, t = camera_pair(cw, n=400000, seed=2)
    S, T = xyz(s), xyz(t)
    init = pose(4, 3.0, 0.02, centre=S.mean(0))
    r = cw.cwipc_icp(s, t, 0.05, init=init, max_iterations=1, relative_fitness=0.0, relative_rmse=0.0)
    want = ref.icp(S, T, 0.05, init=init, max_iterations=1, relative_fitness=0.0, relative_rmse=0.0)
    assert r.iterations == want.iterations == 1
    assert np.abs(r.matrix - want.matrix).max() < 1e-10


def test_one_iteration_follows_the_tie_rule(cw):
    sp, tp, S, T = lattice_pair(cw, 3)
    r = cw.cwipc_icp(sp, tp, SPACING / 2, max_iterations=1, relative_fitness=0.0, relative_rmse=0.0)
    want = ref.icp(S, T, SPACING / 2, max_iterations=1, relative_fitness=0.0, relative_rmse=0.0)
    assert np.abs(r.matrix - want.matrix).max() < 1e-10
    # the other choice of every tie (the higher index) moves the result far more than that
    m = ref.Matcher(T)
    e = ref.evaluate(S, m, np.eye(4), SPACING / 2)
    assert e.correspondences == len(S)
    other = e.dst.copy()
    other[:, 0] = np.where(e.dst[:, 0] > e.src[:, 0], e.dst[:, 0] - np.float32(SPACING), e.dst[:, 0] + np.float32(SPACING))
    assert np.abs(ref.kabsch(e.src, other) - want.matrix).max() > 1e-4


# ---- 3. full runs -------------------------------------------------------------------------------------------------------
def sheet(n, seed, offset=0.0):
    """A wavy 2 m x 2 m sheet: unlike the synthetic capture (a surface of revolution), no motion slides it along itself, so
    ICP can recover every degree of freedom."""
    rng = np.random.default_rng(seed)
    u, v = rng.uniform(-1, 1, n), rng.uniform(-1, 1, n)
    return (np.stack([u, 0.3 * np.sin(3 * u) * np.cos(2 * v) + 0.1 * u * v, v], 1) + offset).astype(np.float32)


@pytest.mark.parametrize("offset", [0.0, 1e4])
def test_recovers_a_seeded_camera_pose(cw, offset):
    T = sheet(200000, 1, offset)
    camera = T[T[:, 0] < np.float32(offset + 0.3)]   # one camera sees part of the scene; the target is all of it
    centre = camera.astype(np.float64).mean(0)
    P = pose(5, 4.0, 0.04, centre=centre)
    tp = cw.cwipc_from_numpy_array(from_xyz(T), 1)
    moved = cw.cwipc_transform(cw.cwipc_from_numpy_array(from_xyz(camera), 1), P)
    S = xyz(moved)
    r = cw.cwipc_icp(moved, tp, 0.2, max_iterations=60)
    err = r.matrix @ P
    # 1e4 m from the origin float32 coordinates are multiples of 2^-10 m, which limits the rotation the points can show
    assert rot_angle(err[:3, :3]) < (1e-6 if offset == 0.0 else 1e-5)
    d = r.matrix - np.linalg.inv(P)
    assert np.abs(d[:3, :3] @ centre + d[:3, 3]).max() < 1e-5      # displacement at the camera's centre
    want = ref.icp(S, T, 0.2, max_iterations=60)
    assert np.abs(r.matrix[:3, :3] - want.matrix[:3, :3]).max() < 1e-7
    assert np.abs((r.matrix - want.matrix)[:3, :3] @ centre + (r.matrix - want.matrix)[:3, 3]).max() < 1e-7
    assert abs(r.correspondences - want.correspondences) <= 5


# ---- 4. consistency with cwipc_cuda_transform ------------------------------------------------------------------------------
def test_result_is_the_evaluation_of_the_moved_source(cw):
    pc, s, t = camera_pair(cw, n=400000, seed=4)
    init = pose(6, 2.0, 0.02, centre=xyz(s).mean(0))
    r = cw.cwipc_icp(s, t, 0.05, init=init)
    assert r.iterations > 1
    again = cw.cwipc_icp(cw.cwipc_transform(s, r.matrix), t, 0.05, max_iterations=0)
    assert (again.correspondences, again.fitness, again.inlier_rmse) == (r.correspondences, r.fitness, r.inlier_rmse)


# ---- 5. determinism and concurrency -----------------------------------------------------------------------------------------
def test_repeatable_bit_for_bit_also_from_four_threads(cw):
    pc, s, t = camera_pair(cw, n=400000, seed=5)
    init = pose(7, 3.0, 0.03, centre=xyz(s).mean(0))
    first = cw.cwipc_icp(s, t, 0.05, init=init)
    key = lambda r: (r.matrix.tobytes(), r.fitness, r.inlier_rmse, r.iterations, r.correspondences)
    for _ in range(2):
        assert key(cw.cwipc_icp(s, t, 0.05, init=init)) == key(first)
    got, failures = [], []

    def worker():
        try:
            for _ in range(3):
                got.append(key(cw.cwipc_icp(s, t, 0.05, init=init)))
        except Exception as e:  # pragma: no cover
            failures.append(e)

    threads = [threading.Thread(target=worker) for _ in range(4)]
    for th in threads:
        th.start()
    for th in threads:
        th.join()
    assert not failures, failures
    assert len(got) == 12 and all(g == key(first) for g in got)


# ---- 6. edge cases -----------------------------------------------------------------------------------------------------------
def test_edge_cases(cw):
    pc, s, t = camera_pair(cw, n=100000, seed=6)
    empty = cw.cwipc_tilefilter(pc, 200)
    assert empty.count() == 0
    init = pose(8, 1.0, 0.01)
    for a, b in ((empty, t), (s, empty), (empty, empty)):
        r = cw.cwipc_icp(a, b, 0.05, init=init)
        assert (r.correspondences, r.fitness, r.inlier_rmse, r.iterations) == (0, 0.0, 0.0, 0)
        assert np.array_equal(r.matrix, init)
    r = cw.cwipc_icp(s, s, 0.05)
    assert r.fitness == 1.0 and r.inlier_rmse == 0.0 and r.correspondences == s.count()
    assert np.abs(r.matrix - np.eye(4)).max() < 1e-12
    far = np.eye(4)
    far[0, 3] = 10.0
    r = cw.cwipc_icp(s, t, 0.05, init=far)
    assert (r.correspondences, r.fitness, r.inlier_rmse, r.iterations) == (0, 0.0, 0.0, 0)
    assert np.array_equal(r.matrix, far)


# ---- 7. errors ----------------------------------------------------------------------------------------------------------------
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
    want = cw.cwipc_icp(s, t, 0.05)
    eye = np.eye(4)
    nan_init, w_init = eye.copy(), eye.copy()
    nan_init[1, 2] = np.nan
    w_init[3, 3] = 2.0
    res = cw.util.cwipc_cuda_icp_result()
    cases = [  # (what, source, target, init, d, iterations, rf, rr, result)
        ("d = 0", s, t, None, 0.0, 30, 1e-6, 1e-6, True),
        ("d < 0", s, t, None, -1.0, 30, 1e-6, 1e-6, True),
        ("d NaN", s, t, None, np.nan, 30, 1e-6, 1e-6, True),
        ("d inf", s, t, None, np.inf, 30, 1e-6, 1e-6, True),
        ("iterations < 0", s, t, None, 0.05, -1, 1e-6, 1e-6, True),
        ("fitness < 0", s, t, None, 0.05, 30, -1e-6, 1e-6, True),
        ("fitness NaN", s, t, None, 0.05, 30, np.nan, 1e-6, True),
        ("rmse inf", s, t, None, 0.05, 30, 1e-6, np.inf, True),
        ("init NaN", s, t, nan_init, 0.05, 30, 1e-6, 1e-6, True),
        ("init last row", s, t, w_init, 0.05, 30, 1e-6, 1e-6, True),
        ("result NULL", s, t, None, 0.05, 30, 1e-6, 1e-6, False),
        ("NaN in the source", sn, t, None, 0.05, 30, 1e-6, 1e-6, True),
        ("inf in the target", s, ti, None, 0.05, 30, 1e-6, 1e-6, True),
        ("NaN in the target", s, sn, None, 0.05, 30, 1e-6, 1e-6, True),
    ]
    seen = []
    cw.cwipc_log_configure(cw.CWIPC_LOG_LEVEL_WARNING, lambda level, msg: seen.append((level, msg.decode())))
    try:
        for what, a, b, init, d, n, rf, rr, has_result in cases:
            seen.clear()
            m = None if init is None else np.ascontiguousarray(init)
            rv = lib.cwipc_cuda_icp(a.as_cwipc_p(), b.as_cwipc_p(), None if m is None else m.ctypes.data, d, n, rf, rr, ctypes.byref(res) if has_result else None)
            assert rv == -1, what
            assert len(seen) == 1 and seen[0][0] == cw.CWIPC_LOG_LEVEL_ERROR and seen[0][1].startswith("cwipc_cuda_icp: "), (what, seen)
        for a, b in ((None, t), (s, None), (None, None)):
            seen.clear()
            rv = lib.cwipc_cuda_icp(a.as_cwipc_p() if a else None, b.as_cwipc_p() if b else None, None, -1.0, -1, -1.0, -1.0, None)
            assert rv == -1 and not seen
    finally:
        cw.cwipc_log_configure(cw.CWIPC_LOG_LEVEL_WARNING, None)
    with pytest.raises(cw.CwipcError):
        cw.cwipc_icp(s, t, -1.0)
    for pc, pts in ((s, good), (t, good[::2]), (sn, with_nan), (ti, with_inf)):
        assert records(pc).tobytes() == pts.tobytes()
    again = cw.cwipc_icp(s, t, 0.05)
    assert (again.matrix.tobytes(), again.fitness, again.inlier_rmse, again.correspondences) == (want.matrix.tobytes(), want.fitness, want.inlier_rmse, want.correspondences)
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
        rv = cw.util.cwipc_util_dll_load().cwipc_cuda_icp(s.as_cwipc_p(), t.as_cwipc_p(), None, 0.05, 30, 1e-6, 1e-6, ctypes.byref(res))
    finally:
        cw.cwipc_log_configure(cw.CWIPC_LOG_LEVEL_WARNING, None)
    assert rv == -1
    assert len(seen) == 1 and seen[0][0] == cw.CWIPC_LOG_LEVEL_ERROR and seen[0][1].startswith("cwipc_cuda_icp: "), seen
    assert cw.cwipc_icp(s, s, 0.05).fitness == 1.0 and cw.cwipc_icp(t, t, 0.05).fitness == 1.0


# ---- 8. launches and leaks ----------------------------------------------------------------------------------------------------
def test_index_is_built_once_per_call_and_nothing_leaks(cw):
    base = cw.cwipc_dangling_allocations(False)
    pc, s, t = camera_pair(cw, n=200000, seed=11)
    init = pose(12, 3.0, 0.03, centre=xyz(s).mean(0))
    launches = []
    for n in (0, 1, 2, 5):
        before = cw.cuda_kernel_launches()
        r = cw.cwipc_icp(s, t, 0.05, init=init, max_iterations=n, relative_fitness=0.0, relative_rmse=0.0)
        launches.append(cw.cuda_kernel_launches() - before)
        assert r.iterations == n
    per = launches[1] - launches[0]
    assert per > 0 and launches[2] - launches[0] == 2 * per and launches[3] - launches[0] == 5 * per, launches
    for c in (pc, s, t):
        c.free()
    assert cw.cwipc_dangling_allocations(False) == base
