"""Every failure of the downsample host path, as a caller sees it.

Each failure gives the entry point's failure value (NULL, or -1 for cwipc_cuda_downsample_keys) and exactly one ERROR log,
whose whole line is pinned here: "<entry point>: Error: <message>".  The thread's next downsample of a good cloud gives
the same bytes as before the failure (a failure must not leave the thread's voxel workspace dirty), and every case leaves
cwipc_dangling_allocations where it found it.  Every case runs under each CWIPC_CUDA_DS_PATH value.
"""
import ctypes
import math

import numpy as np
import pytest

from cwipc_util_b200 import synthetic

pytestmark = pytest.mark.gpu

DT = synthetic.cwipc_point_numpy_dtype
PATHS = (None, "twopass", "generic", "smalltable")   # None: the default (fused single pass when voxelsize > 0)

NONFINITE = "pointcloud contains non-finite coordinates"
DEPTH16 = "pointcloud extent too large for voxel size (octree depth 16 > 14)"
OVERFLOW = "VoxelGrid std exception: leaf size is too small for the input dataset (integer indices would overflow)"
EMPTY = "VoxelGrid filter produced empty pointcloud"
ZERO = "invalid voxel size 0.000000"
NAN = "invalid voxel size nan"
FAR = "point coordinates out of range for voxel size 0.001000 (|x/voxelsize| must stay below 2^22)"
SORTBITS = "pointcloud too large for 64-bit voxel sort words (61 key bits + 4 index bits)"
NOSTATE = "planned downsample needs the octree state of the whole cloud"
RUNAWAY = "octree replay: runaway growth (non-finite coordinates?)"


def points(x, y, z, seed):
    rng = np.random.default_rng(seed)
    pts = np.zeros(len(x), DT)
    pts["x"], pts["y"], pts["z"] = x, y, z
    for c in "rgb":
        pts[c] = rng.integers(0, 256, len(x)).astype(np.uint8)
    pts["tile"] = 1
    return pts


def box(n, lo, hi, seed):
    rng = np.random.default_rng(seed)
    return points(*(rng.uniform(lo, hi, n).astype(np.float32) for _ in range(3)), seed)


def on_x_axis(n, x_end):
    return points(np.linspace(0, x_end, n).astype(np.float32), np.zeros(n, np.float32), np.zeros(n, np.float32), n)


def clouds():
    nonfinite = box(200, -1.0, 1.0, 1)
    nonfinite["x"][5] = np.inf
    far = box(200, 0.0, 0.1, 2)
    far["x"] += np.float32(5000.0)                   # 5000 / 0.001 >= 2^22
    return {
        "nonfinite": nonfinite,
        # leaves of 64 * 0.01 from the first point at 0: x up to 25600 needs 2^16 of them, 8000 needs 2^14
        "deep": on_x_axis(64, 25600.0),
        "depth14": on_x_axis(16, 8000.0),           # 16 voxels: 4 index bits on top of 19 + 3 * 14 key bits
        "wide": box(200, -1.0, 1.0, 3),             # one grid of 1e-5 over it needs more than 2^31 cells
        "far": far,
        "empty": np.zeros(0, DT),
    }


# (cloud, voxelsize, message) per entry point
DOWNSAMPLE = [
    ("nonfinite", 0.01, NONFINITE), ("nonfinite", -0.01, NONFINITE), ("deep", 0.01, DEPTH16), ("wide", -1e-5, OVERFLOW),
    ("empty", -0.01, EMPTY), ("wide", 0.0, ZERO), ("wide", math.nan, NAN), ("far", 0.001, FAR), ("far", -0.001, FAR),
    ("depth14", 0.01, SORTBITS),
]
PLANNED = [c for c in DOWNSAMPLE if c[0] != "empty"] + [("wide", 0.01, NOSTATE)]   # an empty part is an empty cloud
SLAB = [
    ("nonfinite", 0.01, RUNAWAY), ("nonfinite", -0.01, NONFINITE), ("deep", 0.01, DEPTH16), ("wide", -1e-5, OVERFLOW),
    ("wide", 0.0, RUNAWAY), ("far", 0.001, FAR), ("far", -0.001, FAR), ("depth14", 0.01, SORTBITS),
]
KEYS = [("nonfinite", 0.01, NONFINITE), ("nonfinite", -0.01, NONFINITE), ("deep", 0.01, DEPTH16), ("wide", -1e-5, OVERFLOW)]


def upload(cw, pts):
    pc = cw.cwipc_from_numpy_array(pts, 1) if len(pts) else cw.cwipc_from_points([], 1)
    pc._set_cellsize(0.0)
    return pc


def records(pc):
    out = pc.get_numpy_array().copy()
    pc.free()
    return out


def bounds_of(pts):
    return np.array([pts[a].min() for a in "xyz"] + [pts[a].max() for a in "xyz"], np.float32)


@pytest.fixture
def errors(cw):
    seen = []
    cw.cwipc_log_configure(cw.CWIPC_LOG_LEVEL_WARNING, lambda level, msg: seen.append((level, msg.decode())))
    yield seen
    cw.cwipc_log_configure(cw.CWIPC_LOG_LEVEL_WARNING, None)


@pytest.mark.parametrize("entry", ["cwipc_downsample", "cwipc_cuda_downsample_pertile", "cwipc_cuda_downsample_planned",
                                   "cwipc_cuda_slab_downsample", "cwipc_cuda_downsample_keys"])
@pytest.mark.parametrize("path", PATHS)
def test_failure_value_one_error_and_a_clean_thread(cw, errors, monkeypatch, entry, path):
    if path is None:
        monkeypatch.delenv("CWIPC_CUDA_DS_PATH", raising=False)
    else:
        monkeypatch.setenv("CWIPC_CUDA_DS_PATH", path)
    lib = cw.util.cwipc_util_dll_load()
    good = upload(cw, synthetic.camera_cloud(20000, seed=5))
    want = {v: records(cw.cwipc_downsample(good, v)) for v in (0.01, -0.01)}
    data = clouds()
    small = box(100, 0.0, 0.01, 4)                   # a group that downsamples at every voxel size below
    comm = cw.util.cuda_comm(None, 1, 0)
    cases = {"cwipc_downsample": DOWNSAMPLE, "cwipc_cuda_downsample_pertile": DOWNSAMPLE, "cwipc_cuda_downsample_planned": PLANNED,
             "cwipc_cuda_slab_downsample": SLAB, "cwipc_cuda_downsample_keys": KEYS}[entry]
    cases = cases + ([("two groups", v, m) for name, v, m in DOWNSAMPLE if name != "empty"] if entry == "cwipc_cuda_downsample_pertile" else [])
    try:
        for name, voxel, message in cases:
            base = cw.cwipc_dangling_allocations(False)
            expect = f"{entry}: Error: {message}"
            if name == "two groups":
                # tile 1 (good) first, then the failing cloud as tile 2; an invalid voxel size already fails tile 1
                bad = next(data[c] for c, v, m in DOWNSAMPLE if m == message).copy()
                bad["tile"] = 2
                pts = np.concatenate([small, bad])
                expect = f"{entry}: Error: tile {1 if message in (ZERO, NAN) else 2}: {message}"
            else:
                pts = data[name]
                if entry == "cwipc_cuda_downsample_pertile" and len(pts):
                    expect = f"{entry}: Error: tile 1: {message}"   # the only group is named; an empty cloud has none
            pc = upload(cw, pts)
            p = pc.as_cwipc_p()
            keys = np.zeros(max(1, len(pts)), np.uint64)
            state = cw.util.cwipc_cuda_octree_state()
            if entry == "cwipc_cuda_downsample_planned" and message != NOSTATE and not voxel < 0:
                if message in (NONFINITE, ZERO, NAN):   # the cloud's own replay cannot succeed: any valid state
                    cw.util.octree_replay(good, 0.01, state)
                else:
                    cw.util.octree_replay(pc, voxel, state)
            bounds = bounds_of(pts) if len(pts) else np.zeros(6, np.float32)
            errors.clear()
            if entry == "cwipc_cuda_downsample_keys":
                rv, failure = lib.cwipc_cuda_downsample_keys(p, voxel, keys.ctypes.data, len(pts)), -1
            else:
                rv = {"cwipc_downsample": lambda: lib.cwipc_downsample(p, voxel),
                      "cwipc_cuda_downsample_pertile": lambda: lib.cwipc_cuda_downsample_pertile(p, voxel),
                      "cwipc_cuda_downsample_planned": lambda: lib.cwipc_cuda_downsample_planned(p, voxel, ctypes.addressof(state), bounds.ctypes.data),
                      "cwipc_cuda_slab_downsample": lambda: lib.cwipc_cuda_slab_downsample(p, voxel, comm._c)}[entry]()
                failure = None
            logged = [m for level, m in errors if level == cw.CWIPC_LOG_LEVEL_ERROR]
            assert (rv == failure) if failure is not None else not rv, (name, voxel, rv)
            assert logged == [expect], (name, voxel, logged)
            for v in want:
                assert np.array_equal(records(cw.cwipc_downsample(good, v)).view(np.uint8), want[v].view(np.uint8)), (name, voxel, v)
            pc.free()
            assert cw.cwipc_dangling_allocations(False) == base, (name, voxel)
    finally:
        comm.free()
        good.free()
