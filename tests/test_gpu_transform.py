"""cwipc_cuda_transform: every point moved by the 4x4 matrix of its tile value, on the device.

The reference in every case is numpy float64 elementwise arithmetic in the order the header states,
(((m[r][0]*x + m[r][1]*y) + m[r][2]*z) + m[r][3]).astype(float32), and the result must equal it in every byte of every
16-byte record.  The GPU tests are marked one by one: the binding's shape check runs without a device.
"""
import ctypes
import threading

import numpy as np
import pytest
from scipy.spatial.transform import Rotation

from cwipc_util_b200 import synthetic

DT = synthetic.cwipc_point_numpy_dtype
gpu = pytest.mark.gpu


def rigid(seed, translation_scale=1.0):
    """A seeded rotation with a translation."""
    rng = np.random.default_rng(seed)
    m = np.eye(4)
    m[:3, :3] = Rotation.random(random_state=seed).as_matrix()
    m[:3, 3] = rng.uniform(-translation_scale, translation_scale, 3)
    return m


def affine(seed):
    """A general affine map: rotation, anisotropic scale, shear and translation."""
    rng = np.random.default_rng(seed)
    shear = np.eye(3)
    shear[0, 1], shear[0, 2], shear[1, 2] = rng.uniform(-0.7, 0.7, 3)
    m = np.eye(4)
    m[:3, :3] = Rotation.random(random_state=seed).as_matrix() @ np.diag(rng.uniform(0.2, 5.0, 3)) @ shear
    m[:3, 3] = rng.uniform(-3, 3, 3)
    return m


def expected(pts, table):
    """table: {tile value: 4x4}.  The points of a listed value, or of any unlisted value when 0 is listed, moved by their
    matrix in float64 in the stated order; every other record copied."""
    out = pts.copy()
    x, y, z = (pts[a].astype(np.float64) for a in "xyz")
    for v in np.unique(pts["tile"]):
        m = table.get(int(v), table.get(0))
        if m is None:
            continue
        m = np.asarray(m, np.float64)
        sel = pts["tile"] == v
        for r, a in enumerate("xyz"):
            out[a][sel] = (((m[r, 0] * x[sel] + m[r, 1] * y[sel]) + m[r, 2] * z[sel]) + m[r, 3]).astype(np.float32)
    return out


def records(pc):
    return pc.get_numpy_array().copy()


def assert_identical(got, want):
    assert len(got) == len(want)
    assert np.array_equal(got.view(np.uint8), want.view(np.uint8))


def random_cloud(n, seed, tiles=(1, 2, 4, 8), lo=-1.0, hi=1.0):
    rng = np.random.default_rng(seed)
    pts = np.zeros(n, DT)
    for a in "xyz":
        pts[a] = rng.uniform(lo, hi, n).astype(np.float32)
    for c in "rgb":
        pts[c] = rng.integers(0, 256, n).astype(np.uint8)
    pts["tile"] = rng.choice(np.array(tiles, np.uint8), n)
    return pts


def denormal_cloud(n, seed):
    """x, y, z float32 denormals (and a few zeros) of either sign."""
    rng = np.random.default_rng(seed)
    pts = random_cloud(n, seed)
    for a in "xyz":
        bits = rng.integers(0, 0x00800000, n).astype(np.uint32) | (rng.integers(0, 2, n).astype(np.uint32) << 31)
        pts[a] = bits.view(np.float32)
    return pts


@pytest.fixture
def errors(cw):
    """The library's ERROR lines during a test."""
    seen = []
    cw.cwipc_log_configure(cw.CWIPC_LOG_LEVEL_ERROR, lambda level, msg: seen.append((level, msg.decode())))
    yield seen
    cw.cwipc_log_configure(cw.CWIPC_LOG_LEVEL_WARNING, None)


# ---- 1. whole cloud, bit for bit ---------------------------------------------------------------------------------------
CLOUDS = {
    "camera_1M": lambda: synthetic.camera_cloud(1000000, seed=1),
    "uniform_8M": lambda: random_cloud(8000000, 2),
    "far_1e4": lambda: random_cloud(300000, 3, lo=9990.0, hi=10010.0),
    "denormal": lambda: denormal_cloud(100000, 4),
}


@gpu
@pytest.mark.parametrize("cloud", list(CLOUDS))
def test_whole_cloud_is_the_numpy_formula(cw, cloud):
    pts = CLOUDS[cloud]()
    pc = cw.cwipc_from_numpy_array(pts, 1)
    for m in (rigid(11), rigid(12, translation_scale=1e4), affine(13), affine(14)):
        assert_identical(records(cw.cwipc_transform(pc, m)), expected(pts, {0: m}))


@gpu
def test_results_in_the_float_denormal_range(cw):
    pts = random_cloud(200000, 5)
    m = affine(15)
    m[:3, :] *= 1e-40   # |result| around 1e-40: below float's smallest normal (1.2e-38)
    want = expected(pts, {0: m})
    assert np.count_nonzero((np.abs(want["x"]) < np.finfo(np.float32).tiny) & (want["x"] != 0)) > len(pts) // 2
    assert_identical(records(cw.cwipc_transform(cw.cwipc_from_numpy_array(pts, 1), m)), want)


@gpu
@pytest.mark.parametrize("n", [0, 1, 3, 4, 5, 7, 255, 256, 257, 1023, 1024, 1025, 4099, 65537, 262147, 1000003])
def test_point_counts(cw, n):
    pts = random_cloud(n, n)
    pc = cw.cwipc_from_numpy_array(pts, 1) if n else cw.cwipc_from_points([], 1)
    out = cw.cwipc_transform(pc, affine(n))
    assert out.count() == n
    assert_identical(records(out), expected(pts, {0: affine(n)}))


# ---- 2. per tile ---------------------------------------------------------------------------------------------------------
@gpu
def test_listed_tiles_move_and_the_others_are_copied(cw):
    pts = synthetic.camera_cloud(400000, seed=6)
    assert set(np.unique(pts["tile"])) == {1, 2, 4, 8}
    pc = cw.cwipc_from_numpy_array(pts, 1)
    for table in ({1: rigid(1), 4: affine(2)}, {8: affine(3)}, {1: rigid(4), 2: rigid(5), 4: rigid(6), 8: rigid(7)}, {3: affine(8)}):
        got = records(cw.cwipc_transform(pc, table))
        assert_identical(got, expected(pts, table))
        unlisted = ~np.isin(pts["tile"], list(table))
        assert_identical(got[unlisted], pts[unlisted])


@gpu
def test_tile_zero_applies_to_exactly_the_unlisted_values(cw):
    pts = synthetic.camera_cloud(400000, seed=7)
    pc = cw.cwipc_from_numpy_array(pts, 1)
    a, b = affine(21), rigid(22)
    got = records(cw.cwipc_transform(pc, {2: a, 0: b}))
    assert_identical(got, expected(pts, {2: a, 0: b}))
    assert_identical(got[pts["tile"] == 2], expected(pts[pts["tile"] == 2], {0: a}))
    assert_identical(got[pts["tile"] != 2], expected(pts[pts["tile"] != 2], {0: b}))


@gpu
def test_or_ed_tiles_of_a_downsample_match_by_exact_value(cw):
    pc = cw.cwipc_from_numpy_array(synthetic.camera_cloud(1000000, seed=8), 1)
    ds = cw.cwipc_downsample(pc, 0.02)
    pts = records(ds)
    values = set(int(v) for v in np.unique(pts["tile"]))
    mixed = sorted(v for v in values if v & (v - 1))
    assert mixed, "the downsample should have voxels seen by two cameras"
    for table in ({1: affine(31), mixed[0]: rigid(32)}, {1: affine(33), 2: rigid(34)}, {mixed[0]: rigid(35), 0: affine(36)}):
        got = records(cw.cwipc_transform(ds, table))
        assert_identical(got, expected(pts, table))
        if 0 not in table:   # a voxel of tiles 1 and 2 (value 3) is not moved by the entries for 1 or 2
            untouched = ~np.isin(pts["tile"], list(table))
            assert_identical(got[untouched], pts[untouched])


@gpu
def test_shuffled_order_gives_the_shuffled_result(cw):
    pts = synthetic.camera_cloud(500000, seed=9)
    perm = np.random.default_rng(9).permutation(len(pts))
    table = {1: affine(41), 2: rigid(42), 8: affine(43)}
    got = records(cw.cwipc_transform(cw.cwipc_from_numpy_array(pts, 1), table))
    got_shuffled = records(cw.cwipc_transform(cw.cwipc_from_numpy_array(pts[perm], 1), table))
    assert_identical(got_shuffled, got[perm])
    assert_identical(got_shuffled, expected(pts[perm], table))


@gpu
def test_two_hundred_fifty_six_entries(cw):
    """Every tile value listed: slot 255 is a matrix like any other."""
    pts = random_cloud(300000, 10, tiles=tuple(range(256)))
    table = {v: affine(100 + v) for v in range(256)}
    assert_identical(records(cw.cwipc_transform(cw.cwipc_from_numpy_array(pts, 1), table)), expected(pts, table))


# ---- 3. identity ---------------------------------------------------------------------------------------------------------
@gpu
def test_identity_keeps_every_bit_except_negative_zero(cw):
    pts = random_cloud(100000, 11, tiles=(1, 2))
    for i, a in enumerate("xyz"):
        pts[a][i::7] = np.float32(-0.0)
        pts[a][i + 3::7] = np.float32(0.0)
    pc = cw.cwipc_from_numpy_array(pts, 1)
    got = records(cw.cwipc_transform(pc, {1: np.eye(4)}))
    want = pts.copy()
    listed = pts["tile"] == 1
    for a in "xyz":
        col = want[a]
        col[listed & (col == 0)] = np.float32(0.0)   # -0.0 + 0.0 is +0.0
    assert_identical(got, want)
    assert np.signbit(got["x"][~listed & (pts["x"] == 0)]).any()   # the unlisted -0.0 are still there
    assert_identical(got, expected(pts, {1: np.eye(4)}))
    got = records(cw.cwipc_transform(pc, np.eye(4)))
    for a in "xyz":
        col = want[a]
        col[col == 0] = np.float32(0.0)
    assert_identical(got, want)


# ---- 4. a first-class result ---------------------------------------------------------------------------------------------
@gpu
def test_moved_cloud_filters_like_a_fresh_cloud(cw):
    """A downsample result has a known box.  The moved cloud must not carry it: outlier removal and downsample of the moved
    cloud equal those of a fresh cloud made from the numpy-moved points."""
    n = 1000000
    pc = cw.cwipc_from_numpy_array(synthetic.camera_cloud(n, seed=12), 1)
    pc._set_cellsize(synthetic.cellsize_of(n))
    ds = cw.cwipc_downsample(pc, 0.01)
    m = rigid(51)
    m[0, 3] += 10.0
    moved = cw.cwipc_transform(ds, m)
    want = expected(records(ds), {0: m})
    assert_identical(records(moved), want)
    fresh = cw.cwipc_from_numpy_array(want, ds.timestamp())
    fresh._set_cellsize(moved.cellsize())
    for f in (lambda c: cw.cwipc_remove_outliers(c, 30, 1.0, False), lambda c: cw.cwipc_remove_outliers(c, 30, 1.0, True),
              lambda c: cw.cwipc_downsample(c, 0.01)):
        a, b = records(f(moved)), records(f(fresh))
        assert len(a) > 0
        assert_identical(a, b)


@gpu
def test_timestamp_cellsize_and_no_metadata(cw):
    lib = cw.util.cwipc_util_dll_load()
    lib.cwipc_pointcloud_access_metadata.argtypes = [cw.util.cwipc_pointcloud_p]
    lib.cwipc_pointcloud_access_metadata.restype = ctypes.c_void_p
    lib.cwipc_metadata_count.argtypes = [ctypes.c_void_p]
    lib.cwipc_metadata_count.restype = ctypes.c_int
    for pts in (random_cloud(5000, 13), np.zeros(0, DT)):
        pc = cw.cwipc_from_numpy_array(pts, 123456789012) if len(pts) else cw.cwipc_from_points([], 123456789012)
        pc._set_cellsize(0.0125)
        scale = np.diag([3.0, 3.0, 3.0, 1.0])
        out = cw.cwipc_transform(pc, scale)
        assert out.count() == len(pts)
        assert out.timestamp() == 123456789012
        assert out.cellsize() == np.float32(0.0125)    # unchanged, although the matrix scales the cloud
        assert lib.cwipc_metadata_count(lib.cwipc_pointcloud_access_metadata(out.as_cwipc_p())) == 0


# ---- 5. launches and leaks -----------------------------------------------------------------------------------------------
@gpu
def test_one_launch_per_call_and_no_leaks(cw):
    base = cw.cwipc_dangling_allocations(False)
    pc = cw.cwipc_from_numpy_array(random_cloud(300000, 14), 1)
    empty = cw.cwipc_from_points([], 1)
    outs = []
    for table in ({0: affine(61)}, {1: rigid(62), 2: affine(63)}, {v: rigid(v) for v in range(0, 256, 3)}):
        before = cw.cuda_kernel_launches()
        outs.append(cw.cwipc_transform(pc, table))
        assert cw.cuda_kernel_launches() == before + 1
        before = cw.cuda_kernel_launches()
        e = cw.cwipc_transform(empty, table)
        assert cw.cuda_kernel_launches() == before
        assert e.count() == 0
        outs.append(e)
    assert cw.cwipc_dangling_allocations(False) == base + 2 + len(outs)
    for o in outs:
        o.free()
    pc.free()
    empty.free()
    assert cw.cwipc_dangling_allocations(False) == base


# ---- 6. error contract ---------------------------------------------------------------------------------------------------
def bad_arguments():
    """(what, matrices, tiles, n): every argument cwipc_cuda_transform refuses."""
    eye = np.eye(4)
    def mats(*ms):
        return np.ascontiguousarray(np.array(ms, np.float64))
    def tiles(*ts):
        return np.array(ts, np.uint8)
    nan, inf = eye.copy(), eye.copy()
    nan[1, 2] = np.nan
    inf[0, 3] = np.inf
    ninf = eye.copy()
    ninf[2, 0] = -np.inf
    last_nan = eye.copy()
    last_nan[3, 3] = np.nan
    projective, scaled_w, last_x = eye.copy(), eye.copy(), eye.copy()
    projective[3, 2] = 0.5
    scaled_w[3, 3] = 2.0
    last_x[3, 0] = 1e-300
    all_values = np.arange(257) % 256
    return [
        ("n = 0", mats(eye), tiles(0), 0),
        ("n = -1", mats(eye), tiles(0), -1),
        ("NULL matrices", None, tiles(0), 1),
        ("NULL tiles", mats(eye), None, 1),
        ("repeated tile", mats(eye, eye, eye), tiles(1, 2, 1), 3),
        ("repeated tile 0", mats(eye, eye), tiles(0, 0), 2),
        ("n = 257", mats(*([eye] * 257)), all_values.astype(np.uint8), 257),
        ("NaN entry", mats(eye, nan), tiles(1, 2), 2),
        ("inf entry", mats(inf), tiles(0), 1),
        ("-inf entry", mats(ninf), tiles(4), 1),
        ("NaN in the last row", mats(last_nan), tiles(0), 1),
        ("projective last row", mats(projective), tiles(0), 1),
        ("last row (0, 0, 0, 2)", mats(scaled_w), tiles(0), 1),
        ("last row (1e-300, 0, 0, 1)", mats(eye, last_x), tiles(1, 0), 2),
    ]


@gpu
def test_invalid_arguments_fail_once_and_leave_the_input_usable(cw):
    lib = cw.util.cwipc_util_dll_load()
    base = cw.cwipc_dangling_allocations(False)
    pts = random_cloud(200000, 15)
    pc = cw.cwipc_from_numpy_array(pts, 1)
    table = {1: affine(71), 0: rigid(72)}
    want = expected(pts, table)
    cases = bad_arguments()
    outcomes, failures = [], []
    seen = []
    cw.cwipc_log_configure(cw.CWIPC_LOG_LEVEL_WARNING, lambda level, msg: seen.append((level, msg.decode())))
    try:
        def worker():
            try:
                for what, m, t, n in cases:
                    seen.clear()
                    rv = lib.cwipc_cuda_transform(pc.as_cwipc_p(), None if m is None else m.ctypes.data, None if t is None else t.ctypes.data, n)
                    outcomes.append((what, rv, list(seen)))
                seen.clear()
                rv = lib.cwipc_cuda_transform(None, None, None, 0)   # NULL input: NULL, silently, before any argument check
                outcomes.append(("NULL pc", rv, list(seen)))
                outcomes.append(("result", records(cw.cwipc_transform(pc, table)), None))
            except Exception as e:  # pragma: no cover
                failures.append(e)

        th = threading.Thread(target=worker)
        th.start()
        th.join()
    finally:
        cw.cwipc_log_configure(cw.CWIPC_LOG_LEVEL_WARNING, None)
    assert not failures, failures
    assert len(outcomes) == len(cases) + 2
    for what, rv, logged in outcomes[:len(cases)]:
        assert not rv, what
        assert len(logged) == 1 and logged[0][0] == cw.CWIPC_LOG_LEVEL_ERROR and logged[0][1].startswith("cwipc_cuda_transform: "), (what, logged)
    what, rv, logged = outcomes[len(cases)]
    assert not rv and not logged, (what, logged)
    assert_identical(outcomes[-1][1], want)
    assert_identical(records(cw.cwipc_transform(pc, table)), want)
    assert_identical(records(pc), pts)
    pc.free()
    assert cw.cwipc_dangling_allocations(False) == base


@gpu
def test_binding_passes_library_errors_on(cw, errors):
    pc = cw.cwipc_from_numpy_array(random_cloud(1000, 16), 1)
    bad = np.eye(4)
    bad[3, 3] = 0.0
    assert cw.cwipc_transform(pc, bad)._cwipc is None
    assert cw.cwipc_transform(pc, {})._cwipc is None
    assert len(errors) == 2 and all(m.startswith("cwipc_cuda_transform: ") for _, m in errors), errors


# ---- 7. second device ----------------------------------------------------------------------------------------------------
@gpu
def test_result_lives_on_the_input_device(cw):
    if cw.cuda_device_count() < 2:
        pytest.skip("needs two GPUs")
    lib = cw.util.cwipc_util_dll_load()
    pts = synthetic.camera_cloud(200000, seed=17)
    table = {2: affine(81), 0: rigid(82)}
    cw.cuda_set_device(1)
    try:
        pc = cw.cwipc_from_numpy_array(pts, 1)
    finally:
        cw.cuda_set_device(0)
    out = cw.cwipc_transform(pc, table)     # called from a thread whose current device is 0
    assert lib.cwipc_cuda_pointcloud_device(out.as_cwipc_p()) == 1
    assert_identical(records(out), expected(pts, table))


# ---- the binding's own check, no device needed ------------------------------------------------------------------------------
class _NoCloud:
    """Stands in for a cloud; the binding must reject the matrices before it asks for the cloud's pointer."""

    def as_cwipc_p(self):
        raise AssertionError("the library was called")


@pytest.mark.parametrize("matrices", [np.eye(3), np.eye(4)[:3], np.zeros(16), np.zeros((4, 4, 1)), [[1, 0, 0, 0]] * 4 + [[0, 0, 0, 1]],
                                      {1: np.eye(4), 2: np.eye(3)}, {0: np.zeros((2, 8))}])
def test_binding_rejects_a_wrong_shape_before_the_library(matrices):
    from cwipc_util_b200 import util
    with pytest.raises(ValueError):
        util.cwipc_transform(_NoCloud(), matrices)
