"""cwipc_cuda_downsample_pertile: cwipc_downsample of every tile group on its own, in one call.

The result is defined as the composition python/cwipc/registration/util.py:170-182 builds from the library's own filters,
join(downsample(tilefilter(pc, t1)), downsample(tilefilter(pc, t2)), ...) over the tile values in first-appearance order,
and must equal it record for record, bit for bit.  Against the CPU oracle the bars of the downsample parity tests apply.
"""
import os

import numpy as np
import pytest

from cwipc_util_b200 import synthetic
from parity_helpers import assert_points_close

pytestmark = pytest.mark.gpu

DT = synthetic.cwipc_point_numpy_dtype


def random_cloud(n, tiles, layout, seed=0, extent=1.0):
    """`tiles` distinct values; layout "blocky": one contiguous run per value (in the given order), "interleaved": a random
    value per point (every value present)."""
    rng = np.random.default_rng(seed)
    pts = np.zeros(n, DT)
    pts["x"] = rng.uniform(-extent, extent, n).astype(np.float32)
    pts["y"] = rng.uniform(0, 2 * extent, n).astype(np.float32)
    pts["z"] = rng.uniform(-extent, extent, n).astype(np.float32)
    for c in "rgb":
        pts[c] = rng.integers(0, 256, n).astype(np.uint8)
    tiles = np.array(tiles, np.uint8)
    if layout == "blocky":
        pts["tile"] = tiles[np.arange(n) * len(tiles) // n]
    else:
        pts["tile"] = rng.choice(tiles, n)
        pts["tile"][rng.choice(n, len(tiles), replace=False)] = tiles
    return pts


def first_appearance(pts):
    _, first = np.unique(pts["tile"], return_index=True)
    return [int(t) for t in pts["tile"][np.sort(first)]]


def upload(cw, pts, timestamp=1234, cellsize=None):
    pc = cw.cwipc_from_numpy_array(pts, timestamp)
    if cellsize is not None:
        pc._set_cellsize(cellsize)
    return pc


def records(pc):
    return pc.get_numpy_array().copy()


def composition(cw, pc, pts, voxel):
    """What the registration helper computes with the library's own filters."""
    return records(cw.cwipc_join_multi([cw.cwipc_downsample(cw.cwipc_tilefilter(pc, t), voxel) for t in first_appearance(pts)]))


def oracle_pertile(orc, pts, voxel, pc_cellsize):
    """The same composition on the CPU oracle: (points, cellsize, points per voxel)."""
    outs, counts, cs = [], [], None
    for t in first_appearance(pts):
        out, cs, _, c = orc.downsample(orc.tilefilter(pts, t), voxel, pc_cellsize)
        assert out is not None
        outs.append(out)
        counts.append(c)
    return np.concatenate(outs), cs, np.concatenate(counts)


def assert_identical(got, want):
    assert len(got) == len(want)
    assert np.array_equal(got.view(np.uint8), want.view(np.uint8))


@pytest.fixture
def quiet(cw):
    """Collects the library's log lines (ERROR and up) for the duration of a test."""
    seen = []
    cw.cwipc_log_configure(cw.CWIPC_LOG_LEVEL_ERROR, lambda level, msg: seen.append((level, msg)))
    yield seen
    cw.cwipc_log_configure(cw.CWIPC_LOG_LEVEL_WARNING, None)


@pytest.mark.parametrize("n", [6400, 250000, 1000000])
@pytest.mark.parametrize("layout", ["blocky", "interleaved"])
@pytest.mark.parametrize("ntiles", [1, 2, 4, 8])
def test_matches_the_composition(cw, n, layout, ntiles):
    tiles = np.random.default_rng(ntiles).choice(np.arange(1, 256), ntiles, replace=False)
    pts = random_cloud(n, tiles, layout, seed=n % 101 + ntiles)
    pc = upload(cw, pts)
    for voxel in (0.05, -0.05):
        out = cw.cwipc_downsample_pertile(pc, voxel)
        assert_identical(records(out), composition(cw, pc, pts, voxel))


def test_two_hundred_tile_values(cw):
    tiles = np.random.default_rng(7).choice(np.arange(1, 256), 200, replace=False)
    pts = random_cloud(250000, tiles, "interleaved", seed=11)
    assert len(first_appearance(pts)) == 200
    pc = upload(cw, pts)
    for voxel in (0.05, -0.05):
        assert_identical(records(cw.cwipc_downsample_pertile(pc, voxel)), composition(cw, pc, pts, voxel))


def test_cloud_cellsize_larger_than_the_voxel(cw):
    pts = random_cloud(250000, (1, 2, 4, 8), "interleaved", seed=3)
    pc = upload(cw, pts, cellsize=0.08)
    for voxel in (0.05, -0.05):
        out = cw.cwipc_downsample_pertile(pc, voxel)
        assert out.cellsize() == np.float32(0.08)
        assert_identical(records(out), composition(cw, pc, pts, voxel))


@pytest.mark.parametrize("n,voxel,pc_cellsize", [(40000, 0.01, 0.0), (40000, -0.01, 0.0), (250000, 0.004, 0.0), (250000, -0.03, 0.0), (160000, 0.002, 0.005),
                                                 (1000000, 0.01, 0.002)])
def test_matches_oracle(cw, orc, n, voxel, pc_cellsize):
    pts = synthetic.camera_cloud(n, seed=n % 97)
    want, cs, counts = oracle_pertile(orc, pts, voxel, pc_cellsize)
    out = cw.cwipc_downsample_pertile(upload(cw, pts, timestamp=99, cellsize=pc_cellsize), voxel)
    assert out.timestamp() == 99
    assert out.cellsize() == np.float32(cs)
    assert_points_close(records(out), want, cs, counts)


def test_matches_oracle_with_tile_zero(cw, orc):
    pts = random_cloud(120000, (4, 0, 9), "interleaved", seed=5, extent=0.4)
    for voxel in (0.013, -0.013):
        want, cs, counts = oracle_pertile(orc, pts, voxel, 0.0)
        assert_points_close(records(cw.cwipc_downsample_pertile(upload(cw, pts), voxel)), want, cs, counts)


@pytest.mark.parametrize("tile", [1, 0])
def test_single_tile_is_cwipc_downsample(cw, tile):
    pts = random_cloud(250000, (tile,), "interleaved", seed=tile)
    pc = upload(cw, pts, cellsize=0.002)
    for voxel in (0.05, -0.05):
        out = cw.cwipc_downsample_pertile(pc, voxel)
        ref = cw.cwipc_downsample(pc, voxel)
        assert (out.timestamp(), out.cellsize()) == (ref.timestamp(), ref.cellsize())
        assert_identical(records(out), records(ref))


def test_tile_zero_is_the_whole_cloud_at_its_first_appearance(cw):
    pts = random_cloud(100000, (3, 0, 5), "interleaved", seed=8)
    pts["tile"][0], pts["tile"][1] = 3, 0      # first appearance: 3, 0, 5
    assert first_appearance(pts) == [3, 0, 5]
    pc = upload(cw, pts)
    for voxel in (0.05, -0.05):
        got = records(cw.cwipc_downsample_pertile(pc, voxel))
        assert_identical(got, composition(cw, pc, pts, voxel))
        g3 = records(cw.cwipc_downsample(cw.cwipc_tilefilter(pc, 3), voxel))
        whole = records(cw.cwipc_downsample(pc, voxel))
        assert_identical(got[len(g3):len(g3) + len(whole)], whole)


def test_empty_null_timestamp_and_cellsize(cw, quiet):
    lib = cw.util.cwipc_util_dll_load()
    empty = cw.cwipc_from_points([], 7)
    out = cw.cwipc_downsample_pertile(empty, 0.1)
    assert out.count() == 0 and out.timestamp() == 7
    assert not lib.cwipc_cuda_downsample_pertile(empty.as_cwipc_p(), -0.1)   # as cwipc_downsample: ERROR + NULL
    assert [level for level, _ in quiet] == [cw.CWIPC_LOG_LEVEL_ERROR]
    del quiet[:]
    assert not lib.cwipc_cuda_downsample_pertile(None, 0.1)                 # silently
    assert not quiet
    pts = random_cloud(20000, (2, 1), "blocky", seed=2)
    for voxel, cellsize, want in ((0.05, 0.0, 0.05), (-0.05, 0.0, 0.05), (0.05, 0.07, 0.07), (-0.05, 0.07, 0.07)):
        out = cw.cwipc_downsample_pertile(upload(cw, pts, timestamp=123456789012, cellsize=cellsize), voxel)
        assert out.timestamp() == 123456789012
        assert out.cellsize() == np.float32(want)


def test_failed_group_then_a_normal_call(cw, quiet):
    """Single grid: tile 2 spans too many voxels for the grid index, so the call fails as the composition would (one ERROR
    that names the tile); the thread's next call works."""
    small = random_cloud(5000, (1,), "interleaved", seed=1, extent=0.1)
    wide = random_cloud(1000, (2,), "interleaved", seed=2, extent=100.0)
    pts = np.concatenate([small, wide])
    lib = cw.util.cwipc_util_dll_load()
    pc = upload(cw, pts)
    tile2 = cw.cwipc_tilefilter(pc, 2)
    assert not lib.cwipc_downsample(tile2.as_cwipc_p(), -0.001)
    del quiet[:]
    assert not lib.cwipc_cuda_downsample_pertile(pc.as_cwipc_p(), -0.001)
    assert len(quiet) == 1 and quiet[0][0] == cw.CWIPC_LOG_LEVEL_ERROR and b"tile 2" in quiet[0][1], quiet
    good = synthetic.camera_cloud(50000, seed=4)
    gpc = upload(cw, good)
    for voxel in (-0.01, 0.01):
        assert_identical(records(cw.cwipc_downsample_pertile(gpc, voxel)), composition(cw, gpc, good, voxel))


@pytest.mark.parametrize("path", ["twopass", "generic", "smalltable"])
def test_every_internal_path_matches_the_composition(cw, path):
    clouds = [(synthetic.camera_cloud(250000, seed=3), 0.004, 0.0), (random_cloud(120000, (6, 0, 1, 200), "interleaved", seed=9, extent=0.4), 0.013, 0.0)]
    os.environ["CWIPC_CUDA_DS_PATH"] = path
    try:
        for pts, voxel, pc_cellsize in clouds:
            pc = upload(cw, pts, cellsize=pc_cellsize)
            for v in (voxel, -voxel):
                assert_identical(records(cw.cwipc_downsample_pertile(pc, v)), composition(cw, pc, pts, v))
    finally:
        del os.environ["CWIPC_CUDA_DS_PATH"]


def test_allocations_return_and_input_is_untouched(cw):
    pts = random_cloud(200000, (8, 0, 2, 1), "interleaved", seed=6)
    pc = upload(cw, pts)
    base = cw.cwipc_dangling_allocations(False)
    for voxel in (0.05, -0.05):
        out = cw.cwipc_downsample_pertile(pc, voxel)
        assert cw.cwipc_dangling_allocations(False) == base + 1
        out.free()
        assert cw.cwipc_dangling_allocations(False) == base
    assert_identical(records(pc), pts)


def test_result_lives_on_the_input_device(cw):
    if cw.cuda_device_count() < 2:
        pytest.skip("needs two GPUs")
    lib = cw.util.cwipc_util_dll_load()
    pts = synthetic.camera_cloud(100000, seed=12)
    cw.cuda_set_device(0)
    want = records(cw.cwipc_downsample_pertile(upload(cw, pts), 0.01))
    cw.cuda_set_device(1)
    try:
        pc = upload(cw, pts)
    finally:
        cw.cuda_set_device(0)
    out = cw.cwipc_downsample_pertile(pc, 0.01)     # called from a thread whose current device is 0
    assert lib.cwipc_cuda_pointcloud_device(out.as_cwipc_p()) == 1
    assert_identical(records(out), want)
