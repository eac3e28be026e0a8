"""Partitioned clouds on the GPU: the protocol of cwipc_util_b200/slab.py with the library's CUDA kernels as
local steps, against the single-GPU cwipc_downsample / cwipc_remove_outliers on the concatenated cloud.

Two ranks sharing GPU 0 (gloo, host staging) run on any box; the NCCL variant (one GPU per rank, device buffers
straight into ncclSend/ncclRecv) needs two GPUs and is skipped otherwise."""
import numpy
import pytest

from cwipc_util_b200 import synthetic

import _slab_runner as runner
from parity_helpers import assert_points_close, sor_group_check, sor_set_check
from test_slab_cpu import make_parts, sorted_records

pytestmark = pytest.mark.gpu


def check_against_single_gpu(cw, orc, parts, dsn, sorn, chainn, voxelsize, k, mul, cellsize):
    """Partitioned results against the single-GPU calls on the concatenated cloud AND against the CPU oracle."""
    whole = numpy.concatenate(parts)
    pc = cw.cwipc_from_numpy_array(whole, 7)
    pc._set_cellsize(cellsize)
    # downsample: same records as one GPU (bit-exact: integer sums do not depend on which rank added what), and that
    # result equals the oracle's in order
    ds = cw.cwipc_downsample(pc, voxelsize)
    got = numpy.concatenate(dsn)
    assert len(got) == ds.count()
    assert numpy.array_equal(sorted_records(got), sorted_records(ds.get_numpy_array()))
    want, cs, _, _ = orc.downsample(whole, voxelsize, cellsize)
    assert_points_close(ds.get_numpy_array(), want, cs)
    assert sum(len(p) > 0 for p in dsn) == len(dsn), "every slab owns voxels"
    # outlier removal: the oracle's keep mask, threshold ties (1e-6) excepted (the all-reduced sums are added in
    # another order than on one GPU)
    got = numpy.concatenate(sorn)
    assert sor_group_check(whole, got, 0, orc.knn_mean_distances(whole, k), mul) == len(got)
    # chain: outlier removal of the partitioned downsample result (order = rank order, so compared as a set)
    gds = ds.get_numpy_array()
    sor_set_check(gds, numpy.concatenate(chainn), orc.knn_mean_distances(gds, k), mul)


@pytest.mark.parametrize("world,voxelsize", [(2, 0.01), (3, -0.02)])
def test_slabs_sharing_one_gpu(cw, orc, world, voxelsize, tmp_path):
    parts = make_parts(40000, world, seed=20 + world)
    args = dict(voxelsize=voxelsize, k=30, mul=1.0, cellsize=0.002)
    dsn, sorn, chainn = runner.launch(world, "cuda-shared", parts, str(tmp_path), port=29661 + world, **args)
    check_against_single_gpu(cw, orc, parts, dsn, sorn, chainn, **args)


def test_slabs_unordered_parts_and_tiny_halo(cw, orc, tmp_path):
    """Parts that are NOT slabs (interleaved points): ownership still puts every voxel on one rank, the halo
    exchange degenerates to all-to-all, and the open-query merge keeps the statistics exact."""
    pts = synthetic.camera_cloud(30000, seed=5, outliers=0.01)
    parts = [pts[0::2].copy(), pts[1::2].copy()]
    args = dict(voxelsize=0.015, k=16, mul=1.5, cellsize=0.0)
    dsn, sorn, chainn = runner.launch(2, "cuda-shared", parts, str(tmp_path), port=29671, halo=1e-3, **args)
    whole = numpy.concatenate(parts)
    pc = cw.cwipc_from_numpy_array(whole, 7)
    ds = cw.cwipc_downsample(pc, 0.015)
    assert numpy.array_equal(sorted_records(numpy.concatenate(dsn)), sorted_records(ds.get_numpy_array()))
    got = numpy.concatenate(sorn)
    assert sor_group_check(whole, got, 0, orc.knn_mean_distances(whole, 16), 1.5) == len(got)


def test_slabs_with_an_empty_part(cw, orc, tmp_path):
    parts = make_parts(20000, 2, seed=77)
    parts = [parts[0], parts[1][:0], parts[1]]  # rank 1 holds nothing
    args = dict(voxelsize=0.02, k=10, mul=1.0, cellsize=0.0)
    dsn, sorn, chainn = runner.launch(3, "cuda-shared", parts, str(tmp_path), port=29691, **args)
    whole = numpy.concatenate(parts)
    pc = cw.cwipc_from_numpy_array(whole, 7)
    ds = cw.cwipc_downsample(pc, 0.02)
    assert len(dsn[1]) == 0 and len(sorn[1]) == 0
    assert numpy.array_equal(sorted_records(numpy.concatenate(dsn)), sorted_records(ds.get_numpy_array()))
    got = numpy.concatenate(sorn)
    assert sor_group_check(whole, got, 0, orc.knn_mean_distances(whole, 10), 1.0) == len(got)


def test_slabs_nccl_one_gpu_per_rank(cw, orc, tmp_path):
    if cw.cuda_device_count() < 2:
        pytest.skip("needs two GPUs")
    world = min(cw.cuda_device_count(), 4)
    parts = make_parts(200000, world, seed=31)
    args = dict(voxelsize=0.005, k=30, mul=1.0, cellsize=0.002)
    dsn, sorn, chainn = runner.launch(world, "cuda-nccl", parts, str(tmp_path), port=29681, **args)
    check_against_single_gpu(cw, orc, parts, dsn, sorn, chainn, **args)


# ---- the protocol inside the library (csrc/slab.cpp, NCCL) ------------------------------------------------------------------
def test_library_slab_entry_points_with_one_rank(cw, orc):
    """A communicator of size 1 needs no NCCL: the collective entry points reduce to the plain filters (same code path as
    with several ranks, minus the transfers)."""
    from cwipc_util_b200 import util
    from parity_helpers import per_tile_check
    pts = synthetic.camera_cloud(60000, seed=9)
    pc = cw.cwipc_from_numpy_array(pts, 5)
    pc._set_cellsize(0.002)
    comm = util.cuda_comm(None, 1, 0)
    for voxel in (0.01, -0.02):
        want, cs, _, _ = orc.downsample(pts, voxel, 0.002)
        got = comm.downsample(pc, voxel)
        assert got.cellsize() == numpy.float32(cs) and got.timestamp() == 5
        assert_points_close(got.get_numpy_array(), want, cs)
    got = comm.remove_outliers(pc, 30, 1.0).get_numpy_array()
    assert sor_group_check(pts, got, 0, orc.knn_mean_distances(pts, 30), 1.0) == len(got)
    per_tile_check(orc, pts, comm.remove_outliers(pc, 30, 1.0, True).get_numpy_array(), 30, 1.0)
    tf, off, tot = comm.tilefilter(pc, 4)
    assert off == 0 and tot == tf.count() and numpy.array_equal(tf.get_numpy_array(), pts[pts["tile"] == 4])
    comm.free()


@pytest.mark.parametrize("voxelsize", [0.005, -0.01])
def test_library_slabs_over_nccl(cw, orc, voxelsize, tmp_path):
    """One GPU per rank, the library's own NCCL protocol: downsample / remove_outliers (whole cloud and per tile) /
    tilefilter of the partitioned cloud against the single-GPU calls and the oracle.  Needs >= 2 GPUs."""
    from parity_helpers import per_tile_check
    if cw.cuda_device_count() < 2:
        pytest.skip("needs two GPUs")
    world = min(cw.cuda_device_count(), 4)
    parts = make_parts(200000, world, seed=31)
    args = dict(voxelsize=voxelsize, k=30, mul=1.0, cellsize=0.002)
    dsn, sorn, chainn, pertile, tf, tfmeta = runner.launch(world, "lib", parts, str(tmp_path), port=29711, **args)
    check_against_single_gpu(cw, orc, parts, dsn, sorn, chainn, **args)
    whole = numpy.concatenate(parts)
    # tilefilter: the pieces in rank order are the single-GPU result, and every rank knows where its piece sits
    want = whole[whole["tile"] == 2]
    assert numpy.array_equal(numpy.concatenate(tf), want)
    off = 0
    for r in range(world):
        assert tfmeta[r][0] == off and tfmeta[r][1] == len(want)
        off += len(tf[r])
    # per tile: tile by tile (first-appearance order of the whole cloud), the ranks' pieces in rank order
    _, first = numpy.unique(whole["tile"], return_index=True)
    tiles = whole["tile"][numpy.sort(first)]
    pos = [0] * world
    rebuilt = []
    for t in tiles:
        grp_total = 0
        for r in range(world):
            grp_r = parts[r] if t == 0 else parts[r][parts[r]["tile"] == t]
            # this rank's survivors of the group are a subsequence of its part of the group: walk it
            piece = pertile[r][pos[r]:]
            take, j = 0, 0
            for row in grp_r:
                if j < len(piece) and piece[j] == row:
                    j += 1
            take = j
            rebuilt.append(piece[:take])
            pos[r] += take
            grp_total += take
    assert all(pos[r] == len(pertile[r]) for r in range(world))
    per_tile_check(orc, whole, numpy.concatenate(rebuilt), 30, 1.0)


def test_library_slabs_clean_synthetic_cloud_over_nccl(cw, orc, tmp_path):
    """The clean synthetic cloud cut into x-quantile slabs (what bench.py's config4.slabs measures): the first point sits on
    two coordinate planes, whole rings lie exactly on leaf faces, and the single-GPU call takes the fused pass while the
    slabs take the planned one -- the records must still be the same, bit for bit."""
    if cw.cuda_device_count() < 2:
        pytest.skip("needs two GPUs")
    world = min(cw.cuda_device_count(), 4)
    pts = synthetic.simulate_cameras(synthetic.synthetic_cloud(640000), 4)
    edges = numpy.quantile(pts["x"], numpy.linspace(0, 1, world + 1))
    edges[0], edges[-1] = -numpy.inf, numpy.inf
    slab_of = numpy.clip(numpy.searchsorted(edges, pts["x"], side="right") - 1, 0, world - 1)
    parts = [pts[slab_of == r] for r in range(world)]
    args = dict(voxelsize=0.005, k=30, mul=1.0, cellsize=float(synthetic.cellsize_of(640000)))
    dsn, sorn, chainn, pertile, tf, tfmeta = runner.launch(world, "lib", parts, str(tmp_path), port=29731, **args)
    whole = numpy.concatenate(parts)
    pc = cw.cwipc_from_numpy_array(whole, 7)
    pc._set_cellsize(args["cellsize"])
    ds = cw.cwipc_downsample(pc, 0.005).get_numpy_array()
    got = numpy.concatenate(dsn)
    assert len(got) == len(ds)
    a, b = sorted_records(got), sorted_records(ds)
    only_slabs, only_single = numpy.setdiff1d(a, b), numpy.setdiff1d(b, a)
    dt = got.dtype
    assert len(only_slabs) == 0 and len(only_single) == 0, (only_slabs.view(dt), only_single.view(dt))
    want, cs, _, _ = orc.downsample(whole, 0.005, args["cellsize"])
    assert_points_close(ds, want, cs)
