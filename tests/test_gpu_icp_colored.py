"""cwipc_cuda_estimate_color_gradients and cwipc_cuda_icp_colored on the device, against tests/icp_colored_reference.py.

The gradients are compared with the reference fed the library's own normals (which are checked on their own in
tests/test_gpu_icp_plane.py): what is left is differently ordered double sums and a different eigen-solver.  On an exact
colour ramp both round to the same float32, bit for bit.  The first evaluation of a call is cwipc_icp's, and lambda = 1 is
cwipc_icp_point_to_plane's, bit for bit; later steps are compared with the reference within tolerances.
"""
import ctypes
import json
import threading

import numpy as np
import pytest

import icp_colored_reference as cref
import icp_plane_reference as pref
from cwipc_util_b200 import synthetic
from icp_colored_reference import RAMP_COLOURS, RAMP_SPACING, ramp, revolution_pair
from test_gpu_icp_plane import camera_pair, pose, xyz

pytestmark = pytest.mark.gpu


def rot_deg(T):
    R = np.asarray(T)[:3, :3]
    return float(np.degrees(np.arccos(np.clip((np.trace(R) - 1.0) / 2.0, -1.0, 1.0))))


def assert_gradients_match(got, want):
    assert got.shape == want.shape and got.dtype == np.float32
    err = np.linalg.norm(got.astype(np.float64) - want, axis=1)
    scale = np.linalg.norm(want.astype(np.float64), axis=1) + 1e-3
    rel = err / scale
    print(f"gradients: {len(got)} points, {int(np.all(want == 0, axis=1).sum())} zero, relative error median {np.median(rel):.2e} "
          f"99.9% {np.quantile(rel, 0.999):.2e} max {rel.max():.2e}")
    assert np.quantile(rel, 0.999) <= 1e-5
    assert rel.max() <= 1e-2


# ---- 1. gradients ----------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("offset", [0.0, 1e4])
def test_gradients_are_the_reference(cw, offset):
    pts = synthetic.camera_cloud(1000000, seed=1)
    if offset:
        for a in "xyz":
            pts[a] = (pts[a].astype(np.float64) + offset).astype(np.float32)
    raw = cw.cwipc_from_numpy_array(pts, 1)
    for pc, normal_radius in ((raw, 0.01), (cw.cwipc_downsample_pertile(raw, 0.005), 0.02)):
        P = xyz(pc)
        inten = cref.intensity(pc.get_numpy_array())
        tree = pref.cKDTree(P.astype(np.float64))
        nrm = cw.cwipc_estimate_normals(pc, normal_radius, 30)
        for max_nn in ((4, 30, 32) if offset == 0.0 and pc is not raw else (30,)):
            got = cw.cwipc_estimate_color_gradients(pc, normal_radius, 0.1, max_nn=max_nn)
            want = cref.color_gradients(P, inten, nrm, 0.1, max_nn, tree)
            # fewer than 4 neighbours or a zero normal: exactly 0 on both sides
            count = (pref.neighbourhoods(P, 0.1, max_nn, tree) >= 0).sum(1)
            none = (count < 4) | np.all(nrm == 0, axis=1)
            assert np.all(got[none] == 0.0)
            assert_gradients_match(got, want)
            assert np.array_equal(cw.cwipc_estimate_color_gradients(pc, normal_radius, 0.1, max_nn=max_nn), got)   # bit-identical on a second run


def test_gradients_of_an_exact_ramp_are_the_reference_bit_for_bit(cw):
    for colour in RAMP_COLOURS:
        pts, true = ramp(colour=colour)
        pc = cw.cwipc_from_numpy_array(pts, 1)
        nrm = cw.cwipc_estimate_normals(pc, 3 * RAMP_SPACING, 30)
        assert np.all(nrm[:, :2] == 0.0) and np.all(np.abs(nrm[:, 2]) == 1.0)
        got = cw.cwipc_estimate_color_gradients(pc, 3 * RAMP_SPACING, 3 * RAMP_SPACING)
        want = cref.color_gradients(pref.xyz32(pts), cref.intensity(pts), nrm, 3 * RAMP_SPACING, 30)
        assert np.array_equal(want, np.tile(true.astype(np.float32), (len(pts), 1)))
        assert np.array_equal(got, want), (colour, np.abs(got - want).max())


# ---- 2. evaluation only and lambda = 1 -----------------------------------------------------------------------------------------
def test_evaluation_only_is_cwipc_icp_bit_for_bit(cw):
    pc, s, t = camera_pair(cw, n=400000, seed=2)
    for seed, d in ((1, 0.05), (2, 0.01), (3, 0.2)):
        init = pose(seed, 3.0, 0.03, centre=xyz(s).mean(0))
        a = cw.cwipc_icp(s, t, d, init=init, max_iterations=0)
        b = cw.cwipc_icp_colored(s, t, d, 0.01, init=init, max_iterations=0)
        assert b.correspondences == a.correspondences > 0
        assert (b.fitness, b.inlier_rmse, b.iterations) == (a.fitness, a.inlier_rmse, 0)
        assert np.array_equal(b.matrix, init)


def test_lambda_one_is_point_to_plane_bit_for_bit(cw):
    pc, s, t = camera_pair(cw, n=400000, seed=3)
    key = lambda r: (r.matrix.tobytes(), r.fitness, r.inlier_rmse, r.iterations, r.correspondences)
    for seed in (1, 2):
        init = pose(seed, 3.0, 0.03, centre=xyz(s).mean(0))
        a = cw.cwipc_icp_point_to_plane(s, t, 0.05, 0.01, init=init)
        b = cw.cwipc_icp_colored(s, t, 0.05, 0.01, init=init, lambda_geometric=1.0)
        assert a.iterations > 1 and key(b) == key(a)


# ---- 3. one iteration ----------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("lam", [0.968, 0.5, 0.0])
def test_one_iteration_matrix_is_the_reference(cw, lam):
    pc, s, t = camera_pair(cw, n=400000, seed=2)
    S, Tp = s.get_numpy_array().copy(), t.get_numpy_array().copy()
    tp = cw.cwipc_from_numpy_array(Tp, 1)   # a cloud without a stored box: the library's origin is its box centre
    init = pose(4, 3.0, 0.02, centre=xyz(s).mean(0))
    nrm = cw.cwipc_estimate_normals(tp, 0.01, 30)
    grad = cw.cwipc_estimate_color_gradients(tp, 0.01, 0.1)
    r = cw.cwipc_icp_colored(s, tp, 0.05, 0.01, init=init, max_iterations=1, relative_fitness=0.0, relative_rmse=0.0, lambda_geometric=lam)
    want = cref.icp_colored(S, Tp, 0.05, 0.01, init=init, max_iterations=1, relative_fitness=0.0, relative_rmse=0.0, lambda_geometric=lam, normals=nrm, gradients=grad)
    assert r.iterations == want.iterations == 1
    assert np.abs(r.matrix - want.matrix).max() < 1e-10, np.abs(r.matrix - want.matrix).max()


# ---- 4. pose recovery on the surface of revolution -----------------------------------------------------------------------------
@pytest.mark.parametrize("y_degrees", [3.0, 6.0])
def test_recovers_the_turn_about_the_axis_of_revolution(cw, y_degrees):
    source, target, P = revolution_pair(y_degrees)
    sp, tp = cw.cwipc_from_numpy_array(source, 1), cw.cwipc_from_numpy_array(target, 1)
    r = cw.cwipc_icp_colored(sp, tp, 0.05, 0.04)
    plane = cw.cwipc_icp_point_to_plane(sp, tp, 0.05, 0.04)
    centre = pref.move(pref.xyz32(source), np.linalg.inv(P)).astype(np.float64).mean(0)
    E = r.matrix @ P
    residual_m = float(np.linalg.norm(E[:3, :3] @ centre + E[:3, 3] - centre))
    print(f"{y_degrees} deg: colored {r.iterations} iterations, {rot_deg(E):.4f} deg, {residual_m * 1e3:.3f} mm; "
          f"point-to-plane {plane.iterations} iterations, {rot_deg(plane.matrix @ P):.3f} deg")
    assert rot_deg(E) < 0.1 and residual_m < 1e-3 and r.fitness > 0.99
    assert rot_deg(plane.matrix @ P) > 3.0
    want = cref.icp_colored(source, target, 0.05, 0.04, normals=cw.cwipc_estimate_normals(tp, 0.04),
                            gradients=cw.cwipc_estimate_color_gradients(tp, 0.04, 0.1))
    d = r.matrix - want.matrix
    assert np.abs(d[:3, :3]).max() < 1e-6 and np.abs(d[:3, :3] @ centre + d[:3, 3]).max() < 1e-5, (r.iterations, want.iterations, np.abs(d).max())


# ---- 5. determinism and concurrency -------------------------------------------------------------------------------------------------
def test_repeatable_bit_for_bit_also_from_four_threads(cw):
    pc, s, t = camera_pair(cw, n=400000, seed=5)
    init = pose(7, 3.0, 0.03, centre=xyz(s).mean(0))
    call = lambda: cw.cwipc_icp_colored(s, t, 0.05, 0.01, init=init)
    key = lambda r: (r.matrix.tobytes(), r.fitness, r.inlier_rmse, r.iterations, r.correspondences)
    first = key(call())
    grads = cw.cwipc_estimate_color_gradients(t, 0.01, 0.1).tobytes()
    got, failures = [], []

    def worker():
        try:
            for _ in range(3):
                got.append((key(call()), cw.cwipc_estimate_color_gradients(t, 0.01, 0.1).tobytes()))
        except Exception as e:  # pragma: no cover
            failures.append(e)

    threads = [threading.Thread(target=worker) for _ in range(4)]
    for th in threads:
        th.start()
    for th in threads:
        th.join()
    assert not failures, failures
    assert len(got) == 12 and all(g == (first, grads) for g in got)


# ---- 6. edge cases and errors -------------------------------------------------------------------------------------------------------
def test_edge_cases(cw):
    pc, s, t = camera_pair(cw, n=100000, seed=6)
    empty = cw.cwipc_tilefilter(pc, 200)
    assert empty.count() == 0
    init = pose(8, 1.0, 0.01)
    for a, b in ((empty, t), (s, empty), (empty, empty)):
        r = cw.cwipc_icp_colored(a, b, 0.05, 0.01, init=init)
        assert (r.correspondences, r.fitness, r.inlier_rmse, r.iterations) == (0, 0.0, 0.0, 0)
        assert np.array_equal(r.matrix, init)
    assert cw.cwipc_estimate_color_gradients(empty, 0.01, 0.1).shape == (0, 3)
    # lambda = 0: the photometric term alone still gives a finite motion
    init = pose(9, 2.0, 0.01, centre=xyz(s).mean(0))
    r = cw.cwipc_icp_colored(s, t, 0.05, 0.01, init=init, lambda_geometric=0.0)
    assert r.iterations >= 1 and np.all(np.isfinite(r.matrix)) and r.correspondences > 0
    # one colour everywhere: every gradient is 0 and I_s = I_0, so both sums are lambda times point-to-plane's
    S, T = s.get_numpy_array().copy(), t.get_numpy_array().copy()
    for a in (S, T):
        a["r"], a["g"], a["b"] = 90, 140, 30
    su, tu = cw.cwipc_from_numpy_array(S, 1), cw.cwipc_from_numpy_array(T, 1)
    assert np.all(cw.cwipc_estimate_color_gradients(tu, 0.01, 0.1) == 0.0)
    c = cw.cwipc_icp_colored(su, tu, 0.05, 0.01, init=init, max_iterations=1)
    p = cw.cwipc_icp_point_to_plane(su, tu, 0.05, 0.01, init=init, max_iterations=1)
    assert c.correspondences == p.correspondences and np.abs(c.matrix - p.matrix).max() < 1e-12, np.abs(c.matrix - p.matrix).max()


def test_invalid_arguments_fail_once_and_leave_the_inputs_usable(cw):
    lib = cw.util.cwipc_util_dll_load()
    base = cw.cwipc_dangling_allocations(False)
    rng = np.random.default_rng(9)
    good = rng.uniform(-1, 1, (20000, 3)).astype(np.float32)
    pts = np.zeros(len(good), synthetic.cwipc_point_numpy_dtype)
    for i, a in enumerate("xyz"):
        pts[a] = good[:, i]
    pts["r"], pts["g"], pts["b"] = rng.integers(0, 256, (3, len(pts)))
    with_nan, with_inf = pts.copy(), pts.copy()
    with_nan["y"][123] = np.nan
    with_inf["z"][7] = np.inf
    s = cw.cwipc_from_numpy_array(pts, 1)
    t = cw.cwipc_from_numpy_array(pts[::2].copy(), 1)
    sn, ti = cw.cwipc_from_numpy_array(with_nan, 1), cw.cwipc_from_numpy_array(with_inf, 1)
    want = cw.cwipc_icp_colored(s, t, 0.2, 0.2)
    want_g = cw.cwipc_estimate_color_gradients(t, 0.2, 0.2)
    eye = np.eye(4)
    nan_init, w_init = eye.copy(), eye.copy()
    nan_init[1, 2] = np.nan
    w_init[3, 3] = 2.0
    res = cw.util.cwipc_cuda_icp_result()
    cases = [  # (what, source, target, init, d, iterations, rf, rr, radius, max_nn, lambda, result)
        ("d = 0", s, t, None, 0.0, 30, 1e-6, 1e-6, 0.2, 30, 0.968, True),
        ("d NaN", s, t, None, np.nan, 30, 1e-6, 1e-6, 0.2, 30, 0.968, True),
        ("iterations < 0", s, t, None, 0.2, -1, 1e-6, 1e-6, 0.2, 30, 0.968, True),
        ("fitness < 0", s, t, None, 0.2, 30, -1e-6, 1e-6, 0.2, 30, 0.968, True),
        ("rmse inf", s, t, None, 0.2, 30, 1e-6, np.inf, 0.2, 30, 0.968, True),
        ("init NaN", s, t, nan_init, 0.2, 30, 1e-6, 1e-6, 0.2, 30, 0.968, True),
        ("init last row", s, t, w_init, 0.2, 30, 1e-6, 1e-6, 0.2, 30, 0.968, True),
        ("result NULL", s, t, None, 0.2, 30, 1e-6, 1e-6, 0.2, 30, 0.968, False),
        ("radius 0", s, t, None, 0.2, 30, 1e-6, 1e-6, 0.0, 30, 0.968, True),
        ("radius NaN", s, t, None, 0.2, 30, 1e-6, 1e-6, np.nan, 30, 0.968, True),
        ("max_nn 2", s, t, None, 0.2, 30, 1e-6, 1e-6, 0.2, 2, 0.968, True),
        ("max_nn 33", s, t, None, 0.2, 30, 1e-6, 1e-6, 0.2, 33, 0.968, True),
        ("lambda < 0", s, t, None, 0.2, 30, 1e-6, 1e-6, 0.2, 30, -0.01, True),
        ("lambda > 1", s, t, None, 0.2, 30, 1e-6, 1e-6, 0.2, 30, 1.01, True),
        ("lambda NaN", s, t, None, 0.2, 30, 1e-6, 1e-6, 0.2, 30, np.nan, True),
        ("lambda inf", s, t, None, 0.2, 30, 1e-6, 1e-6, 0.2, 30, np.inf, True),
        ("NaN in the source", sn, t, None, 0.2, 30, 1e-6, 1e-6, 0.2, 30, 0.968, True),
        ("inf in the target", s, ti, None, 0.2, 30, 1e-6, 1e-6, 0.2, 30, 0.968, True),
    ]
    out = np.zeros((20000, 3), np.float32)
    gcases = [  # (what, cloud, normal radius, normal max_nn, radius, max_nn, buffer, nfloats)
        ("normal radius 0", t, 0.0, 30, 0.2, 30, out.ctypes.data, out.size),
        ("normal max_nn 2", t, 0.2, 2, 0.2, 30, out.ctypes.data, out.size),
        ("radius 0", t, 0.2, 30, 0.0, 30, out.ctypes.data, out.size),
        ("radius < 0", t, 0.2, 30, -0.1, 30, out.ctypes.data, out.size),
        ("radius NaN", t, 0.2, 30, np.nan, 30, out.ctypes.data, out.size),
        ("radius inf", t, 0.2, 30, np.inf, 30, out.ctypes.data, out.size),
        ("max_nn 3", t, 0.2, 30, 0.2, 3, out.ctypes.data, out.size),
        ("max_nn 33", t, 0.2, 30, 0.2, 33, out.ctypes.data, out.size),
        ("NULL buffer", t, 0.2, 30, 0.2, 30, None, out.size),
        ("short buffer", t, 0.2, 30, 0.2, 30, out.ctypes.data, 3 * t.count() - 1),
        ("NaN in the cloud", sn, 0.2, 30, 0.2, 30, out.ctypes.data, out.size),
        ("inf in the cloud", ti, 0.2, 30, 0.2, 30, out.ctypes.data, out.size),
    ]
    seen = []
    cw.cwipc_log_configure(cw.CWIPC_LOG_LEVEL_WARNING, lambda level, msg: seen.append((level, msg.decode())))
    try:
        for what, a, b, init, d, n, rf, rr, radius, max_nn, lam, has_result in cases:
            seen.clear()
            m = None if init is None else np.ascontiguousarray(init)
            rv = lib.cwipc_cuda_icp_colored(a.as_cwipc_p(), b.as_cwipc_p(), None if m is None else m.ctypes.data, d, n, rf, rr, radius, max_nn, lam,
                                            ctypes.byref(res) if has_result else None)
            assert rv == -1, what
            assert len(seen) == 1 and seen[0][0] == cw.CWIPC_LOG_LEVEL_ERROR and seen[0][1].startswith("cwipc_cuda_icp_colored: "), (what, seen)
        for what, pc, nr, nnn, radius, max_nn, buf, nfloats in gcases:
            seen.clear()
            rv = lib.cwipc_cuda_estimate_color_gradients(pc.as_cwipc_p(), nr, nnn, radius, max_nn, buf, nfloats)
            assert rv == -1, what
            assert len(seen) == 1 and seen[0][0] == cw.CWIPC_LOG_LEVEL_ERROR and seen[0][1].startswith("cwipc_cuda_estimate_color_gradients: "), (what, seen)
        for a, b in ((None, t), (s, None), (None, None)):
            seen.clear()
            rv = lib.cwipc_cuda_icp_colored(a.as_cwipc_p() if a else None, b.as_cwipc_p() if b else None, None, -1.0, -1, -1.0, -1.0, -1.0, 0, 2.0, None)
            assert rv == -1 and not seen
        seen.clear()
        assert lib.cwipc_cuda_estimate_color_gradients(None, -1.0, 0, -1.0, 0, None, 0) == -1 and not seen
    finally:
        cw.cwipc_log_configure(cw.CWIPC_LOG_LEVEL_WARNING, None)
    with pytest.raises(cw.CwipcError):
        cw.cwipc_icp_colored(s, t, 0.2, 0.2, lambda_geometric=2.0)
    with pytest.raises(cw.CwipcError):
        cw.cwipc_estimate_color_gradients(t, 0.2, 0.2, max_nn=40)
    for pc, p in ((s, pts), (t, pts[::2]), (sn, with_nan), (ti, with_inf)):
        assert pc.get_numpy_array().tobytes() == p.tobytes()
    again = cw.cwipc_icp_colored(s, t, 0.2, 0.2)
    assert (again.matrix.tobytes(), again.fitness, again.inlier_rmse, again.correspondences) == (want.matrix.tobytes(), want.fitness, want.inlier_rmse, want.correspondences)
    assert np.array_equal(cw.cwipc_estimate_color_gradients(t, 0.2, 0.2), want_g)
    for pc in (s, t, sn, ti):
        pc.free()
    assert cw.cwipc_dangling_allocations(False) == base


def test_clouds_on_two_devices(cw):
    if cw.cuda_device_count() < 2:
        pytest.skip("needs two GPUs")
    pts = synthetic.synthetic_cloud(10000)
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
        rv = cw.util.cwipc_util_dll_load().cwipc_cuda_icp_colored(s.as_cwipc_p(), t.as_cwipc_p(), None, 0.05, 30, 1e-6, 1e-6, 0.1, 30, 0.968, ctypes.byref(res))
    finally:
        cw.cwipc_log_configure(cw.CWIPC_LOG_LEVEL_WARNING, None)
    assert rv == -1
    assert len(seen) == 1 and seen[0][0] == cw.CWIPC_LOG_LEVEL_ERROR and seen[0][1].startswith("cwipc_cuda_icp_colored: "), seen
    assert cw.cwipc_icp_colored(s, s, 0.05, 0.1).fitness == 1.0 and cw.cwipc_icp_colored(t, t, 0.05, 0.1).fitness == 1.0
    assert np.array_equal(cw.cwipc_estimate_color_gradients(s, 0.1, 0.1), cw.cwipc_estimate_color_gradients(t, 0.1, 0.1))


# ---- 7. launches and leaks ----------------------------------------------------------------------------------------------------------
def test_index_normals_and_gradients_are_built_once_per_call_and_nothing_leaks(cw):
    lib = cw.util.cwipc_util_dll_load()
    base = cw.cwipc_dangling_allocations(False)
    pc, s, t = camera_pair(cw, n=200000, seed=11)
    init = pose(12, 3.0, 0.03, centre=xyz(s).mean(0))
    launches = []
    for n in (0, 1, 2, 5):
        lib.cwipc_cuda_profile_reset()
        lib.cwipc_cuda_profile_enable(1)
        before = cw.cuda_kernel_launches()
        r = cw.cwipc_icp_colored(s, t, 0.05, 0.01, init=init, max_iterations=n, relative_fitness=0.0, relative_rmse=0.0)
        launches.append(cw.cuda_kernel_launches() - before)
        lib.cwipc_cuda_profile_enable(0)
        need = lib.cwipc_cuda_profile_report(None, 0)
        buf = ctypes.create_string_buffer(need)
        lib.cwipc_cuda_profile_report(buf, need)
        prof = json.loads(buf.value.decode())
        assert r.iterations == n
        assert prof["knn_keygen_kernel"]["launches"] == 1 and prof["knn_layout_kernel"]["launches"] == 1
        assert prof["icp_normals_kernel"]["launches"] == 1 and prof["icp_gradients_kernel"]["launches"] == 1
        assert prof["icp_colored_match_kernel"]["launches"] == prof["icp_plane_reduce_kernel"]["launches"] == n + 1
        assert "icp_match_kernel" not in prof and "icp_plane_match_kernel" not in prof
    per = launches[1] - launches[0]
    assert per == 2 and launches[2] - launches[0] == 2 * per and launches[3] - launches[0] == 5 * per, launches
    for c in (pc, s, t):
        c.free()
    assert cw.cwipc_dangling_allocations(False) == base
