"""The error contract of the entry points that read a cloud.

A failure that happens after the input has been taken -- a kNeighbors the kNN cannot do, a voxel size too small for the
cloud, a missing octree state -- gives the call's failure value (-1 or NULL) and one ERROR log naming the entry point.
The input is left usable: the cloud, made on one thread and failed on from another, gives the same results as before
from both threads, and freeing it leaves no allocation behind.
"""
import ctypes
import threading

import numpy as np
import pytest

from cwipc_util_b200 import synthetic

pytestmark = pytest.mark.gpu

DT = synthetic.cwipc_point_numpy_dtype
N, NQUERY, K = 20000, 10000, 30
X_LO, X_HI = -0.5, 0.5


def cloud():
    rng = np.random.default_rng(17)
    pts = np.zeros(N, DT)
    for a in "xyz":
        pts[a] = rng.uniform(-1.0, 1.0, N).astype(np.float32)
    for c in "rgb":
        pts[c] = rng.integers(0, 256, N).astype(np.uint8)
    pts["tile"] = rng.choice(np.array([1, 2, 4], np.uint8), N)
    return pts


def records(pc):
    out = pc.get_numpy_array().copy()
    pc.free()
    return out


def results(cw, pc):
    """What the cloud-reading diagnostic and partition entry points return for pc: name -> arrays."""
    u = cw.util
    got = {"knn_mean_distances": (u.knn_mean_distances(pc, K),), "knn_query": u.knn_query(pc, K, NQUERY)}
    h = u.cuda_distances(pc, K, NQUERY, X_LO, X_HI)
    idx, pts, kth2 = h.open_queries()
    h.free()
    order = np.argsort(idx)   # the open queries are a set: warps append them in whatever order they finish
    idx, pts, kth2 = idx[order], pts[order], kth2[order]
    got["knn_query_open"] = (idx, pts, kth2)
    got["knn_lists"] = (u.knn_lists(pc, pts, K, kth2),)
    state = u.cwipc_cuda_octree_state()
    bounds = u.octree_replay(pc, 0.01, state)
    got["octree_replay"] = (bounds, state.to_array())
    got["downsample_planned"] = (records(u.downsample_planned(pc, 0.01, state, bounds)),)
    got["downsample_keys"] = (u.downsample_keys(pc, 0.01),)
    comm = u.cuda_comm(None, 1, 0)
    try:
        got["slab_remove_outliers"] = (records(comm.remove_outliers(pc, K, 1.0)),)
    finally:
        comm.free()
    return got


def failing_calls(cw, pc):
    """(entry point, call, failure value) for each entry point, with an argument that fails after the input is taken."""
    lib = cw.util.cwipc_util_dll_load()
    p = pc.as_cwipc_p()
    dist = np.zeros(N, np.float32)
    mean, kth2 = np.zeros(NQUERY, np.float32), np.zeros(NQUERY, np.float32)
    queries = pc.get_numpy_array()[:100].copy()
    lists = np.zeros((len(queries), 601), np.float32)
    state = cw.util.cwipc_cuda_octree_state()   # all zero: no points replayed yet
    bounds = np.zeros(6, np.float32)
    keys = np.zeros(N, np.uint64)
    nopen = ctypes.c_int(0)
    comm = cw.util.cuda_comm(None, 1, 0)
    calls = [
        ("cwipc_cuda_knn_mean_distances", lambda: lib.cwipc_cuda_knn_mean_distances(p, 600, dist.ctypes.data, N), -1),
        ("cwipc_cuda_knn_query", lambda: lib.cwipc_cuda_knn_query(p, 600, NQUERY, mean.ctypes.data, kth2.ctypes.data), -1),
        ("cwipc_cuda_knn_query_open", lambda: lib.cwipc_cuda_knn_query_open(p, 600, NQUERY, X_LO, X_HI, ctypes.byref(nopen)), "NULL"),
        ("cwipc_cuda_knn_lists", lambda: lib.cwipc_cuda_knn_lists(p, queries.ctypes.data, None, len(queries), 600, lists.ctypes.data), -1),
        # a leaf of 64 * 1e-12 would need more than 30 doublings of the octree box to reach the cloud's extent
        ("cwipc_cuda_octree_replay", lambda: lib.cwipc_cuda_octree_replay(p, 1e-12, ctypes.addressof(state), bounds.ctypes.data), -1),
        ("cwipc_cuda_downsample_planned", lambda: lib.cwipc_cuda_downsample_planned(p, 0.01, ctypes.addressof(state), bounds.ctypes.data), "NULL"),
        # one grid of 1e-5 over a cloud 2 wide: more cells than 32-bit indices can number
        ("cwipc_cuda_downsample_keys", lambda: lib.cwipc_cuda_downsample_keys(p, -1e-5, keys.ctypes.data, N), -1),
        ("cwipc_cuda_slab_remove_outliers", lambda: lib.cwipc_cuda_slab_remove_outliers(p, 600, 1.0, False, 0.0, comm._c), "NULL"),
    ]
    return calls, comm


def test_failures_after_the_input_is_taken_leave_the_cloud_usable(cw):
    base = cw.cwipc_dangling_allocations(False)
    pc = cw.cwipc_from_numpy_array(cloud(), 1)
    want = results(cw, pc)
    seen, outcomes, errors = [], [], []
    cw.cwipc_log_configure(cw.CWIPC_LOG_LEVEL_WARNING, lambda level, msg: seen.append((level, msg.decode())))
    try:
        def worker():
            try:
                calls, comm = failing_calls(cw, pc)
                try:
                    for name, call, failure in calls:
                        seen.clear()
                        rv = call()
                        outcomes.append((name, rv, failure, [m for level, m in seen if level == cw.CWIPC_LOG_LEVEL_ERROR]))
                finally:
                    comm.free()
                outcomes.append(("results", results(cw, pc), None, None))
            except Exception as e:  # pragma: no cover
                errors.append(e)

        t = threading.Thread(target=worker)
        t.start()
        t.join()
    finally:
        cw.cwipc_log_configure(cw.CWIPC_LOG_LEVEL_WARNING, None)
    assert not errors, errors
    assert len(outcomes) == 9
    for name, rv, failure, logged in outcomes[:-1]:
        assert (not rv) if failure == "NULL" else rv == failure, (name, rv)
        assert len(logged) == 1 and logged[0].startswith(name + ": "), (name, logged)
    for got in (outcomes[-1][1], results(cw, pc)):
        for name in want:
            assert all(np.array_equal(a, b) for a, b in zip(got[name], want[name])), name
    pc.free()
    assert cw.cwipc_dangling_allocations(False) == base
