"""The kernels each outlier-removal entry point launches for one small cloud, by name and count.

cwipc_remove_outliers, cwipc_cuda_knn_query_open and cwipc_cuda_slab_remove_outliers string the same kNN, statistics and
compaction kernels together on the host, each in its own way.  LAUNCHES is what each call below launched on a B200 before
that host code was gathered into shared helpers: host code that is reorganised must launch the same kernels, as many
times.  Every result is checked against the oracle or tests/knn_reference.py too.
"""
import ctypes
import gc
import json

import numpy as np
import pytest

from cwipc_util_b200 import synthetic

import knn_reference as ref
from parity_helpers import per_tile_check, sor_group_check

pytestmark = pytest.mark.gpu

K, MUL, N = 30, 1.0, 6000
X_LO, X_HI = -1.0, 0.1   # about half the queries open

LAUNCHES = {
    "remove_outliers_whole": {"bbox_octree_kernel": 1, "compact_kernel": 1, "knn_far_kernel": 1, "knn_keygen_kernel": 1, "knn_layout_kernel": 1, "knn_tile_kernel": 1, "radix_cluster_kernel": 1, "stats_kernel": 1},
    "remove_outliers_per_tile": {"bbox_octree_kernel": 1, "compact_kernel": 4, "first_tile_kernel": 1, "knn_far_kernel": 1, "knn_keygen_kernel": 1, "knn_layout_kernel": 1, "knn_tile_kernel": 1, "radix_cluster_kernel": 1, "stats_kernel": 4},
    "remove_outliers_per_tile_with_tile0": {"bbox_octree_kernel": 5, "compact_kernel": 9, "first_tile_kernel": 1, "knn_far_kernel": 5, "knn_keygen_kernel": 5, "knn_layout_kernel": 5, "knn_tile_kernel": 5, "radix_cluster_kernel": 5, "stats_kernel": 5},
    "knn_query_open": {"bbox_octree_kernel": 1, "knn_far_kernel": 1, "knn_keygen_kernel": 1, "knn_layout_kernel": 1, "knn_tile_kernel": 1, "mark_open_kernel": 1, "radix_cluster_kernel": 1},
    "knn_query_open_at_most_k_points": {"mark_open_kernel": 1},
    "slab_remove_outliers_whole": {"bbox_octree_kernel": 2, "compact_kernel": 1, "knn_far_kernel": 1, "knn_keygen_kernel": 1, "knn_layout_kernel": 1, "knn_tile_kernel": 1, "mark_open_kernel": 1, "radix_cluster_kernel": 1, "stats_kernel": 1},
    "slab_remove_outliers_per_tile_with_tile0": {"bbox_octree_kernel": 10, "compact_kernel": 9, "first_tile_kernel": 1, "knn_far_kernel": 5, "knn_keygen_kernel": 5, "knn_layout_kernel": 5, "knn_tile_kernel": 5, "mark_open_kernel": 5, "radix_cluster_kernel": 5, "stats_kernel": 5},
    "slab_remove_outliers_empty_part": {},
}


def launches(lib, call):
    """call() under the library's profiler: what it returned, and {kernel name: launches}."""
    lib.cwipc_cuda_profile_reset()
    lib.cwipc_cuda_profile_enable(1)
    try:
        out = call()
    finally:
        lib.cwipc_cuda_profile_enable(0)
    need = lib.cwipc_cuda_profile_report(None, 0)
    buf = ctypes.create_string_buffer(need)
    lib.cwipc_cuda_profile_report(buf, need)
    return out, {name: v["launches"] for name, v in json.loads(buf.value.decode()).items() if v["launches"]}


def cloud(tile0=False):
    pts = synthetic.camera_cloud(N, seed=7)
    if tile0:   # tile 0 among the values: the whole cloud is a group of its own
        pts["tile"][5] = 0
    return pts


def upload(cw, pts):
    pc = cw.cwipc_from_numpy_array(pts, 1)
    pc._set_cellsize(synthetic.cellsize_of(N))
    return pc


def remove_outliers(cw, lib, orc, per_tile, tile0=False, comm=None):
    pts = cloud(tile0)
    pc = upload(cw, pts)
    call = (lambda: comm.remove_outliers(pc, K, MUL, per_tile)) if comm else (lambda: cw.cwipc_remove_outliers(pc, K, MUL, per_tile))
    out, kernels = launches(lib, call)
    got = out.get_numpy_array().copy()
    if per_tile:
        per_tile_check(orc, pts, got, K, MUL)
    else:
        assert sor_group_check(pts, got, 0, orc.knn_mean_distances(pts, K), MUL) == len(got)
    out.free()
    pc.free()
    return kernels


def query_open(cw, lib, n):
    """cwipc_cuda_knn_query_open of the first n // 2 points of n against all n"""
    pts = cloud()[:n].copy()
    nq = max(1, n // 2)
    pc = upload(cw, pts)
    h, kernels = launches(lib, lambda: cw.util.cuda_distances(pc, K, nq, X_LO, X_HI))
    idx, opts, okth2 = h.open_queries()
    order = np.argsort(idx)
    idx, opts, okth2 = idx[order], opts[order], okth2[order]
    if n > K:
        lists = ref.ref_lists(pts, pts[:nq], K)
        mean, kth2 = ref.ref_mean(lists, K), ref.ref_kth2(lists, K)
        assert np.array_equal(idx, ref.ref_open(pts["x"], kth2, nq, X_LO, X_HI))
        assert np.array_equal(okth2, kth2[idx])
        assert h.stats() == cw.util.distance_stats(mean)
    else:   # no neighbourhood is known: every query is open, with a huge finite bound
        assert np.array_equal(idx, np.arange(nq, dtype=np.uint32))
        assert np.all(okth2.view(np.uint32) == 0x7F7F7F7F)
    assert opts.tobytes() == pts[idx].tobytes()
    h.free()
    pc.free()
    return kernels


def slab_remove_outliers(cw, lib, orc, per_tile, tile0=False):
    comm = cw.util.cuda_comm(None, 1, 0)
    try:
        return remove_outliers(cw, lib, orc, per_tile, tile0, comm)
    finally:
        comm.free()


def slab_empty_part(cw, lib, orc):
    comm = cw.util.cuda_comm(None, 1, 0)
    pc = cw.cwipc_from_points([], 1)
    out, kernels = launches(lib, lambda: comm.remove_outliers(pc, K, MUL, True))
    assert out.count() == 0
    out.free()
    pc.free()
    comm.free()
    return kernels


CASES = {
    "remove_outliers_whole": lambda cw, lib, orc: remove_outliers(cw, lib, orc, False),
    "remove_outliers_per_tile": lambda cw, lib, orc: remove_outliers(cw, lib, orc, True),
    "remove_outliers_per_tile_with_tile0": lambda cw, lib, orc: remove_outliers(cw, lib, orc, True, tile0=True),
    "knn_query_open": lambda cw, lib, orc: query_open(cw, lib, N),
    "knn_query_open_at_most_k_points": lambda cw, lib, orc: query_open(cw, lib, K),
    "slab_remove_outliers_whole": lambda cw, lib, orc: slab_remove_outliers(cw, lib, orc, False),
    "slab_remove_outliers_per_tile_with_tile0": lambda cw, lib, orc: slab_remove_outliers(cw, lib, orc, True, tile0=True),
    "slab_remove_outliers_empty_part": slab_empty_part,
}


def record(cw, lib, orc):
    """{case: launches} of every case, for LAUNCHES"""
    return {name: case(cw, lib, orc) for name, case in CASES.items()}


@pytest.mark.parametrize("case", list(CASES))
def test_launches(cw, lib, orc, case):
    gc.collect()
    base = cw.cwipc_dangling_allocations(False)
    assert CASES[case](cw, lib, orc) == LAUNCHES[case]
    gc.collect()
    assert cw.cwipc_dangling_allocations(False) == base
