"""A plain numpy/scipy reference of cwipc_cuda_estimate_normals and cwipc_cuda_icp_point_to_plane (no library calls): the
rules include/cwipc_util_cuda.h states, step by step.  The moving, matching and looping are tests/icp_reference.py's.

- Neighbourhoods: a float64 cKDTree proposes the nearest max_nn + CAND points within the radius.  They are ranked by the exact
  float32 d2 = (dx*dx + dy*dy) + dz*dz and then by index; where the proposal cannot settle the max_nn-th place (every
  proposed point lies within (1 + 1e-5) times the distance of that place), query_ball_point lists every candidate.
- Normals: mean, then covariance relative to it, in float64; numpy.linalg.eigh; the eigenvector of the smallest eigenvalue.
  (0, 0, 0) for fewer than 3 neighbours or a zero covariance.
- Step: r = (p' - q) . n and J = [p' x n, n] relative to the target's box centre; the minimum-norm solution of
  (J^T J) x = -J^T r from eigh, eigenvalues <= 1e-12 times the largest dropped; dT = [Rz Ry Rx, t] about the box centre.
"""
from typing import NamedTuple

import numpy as np
from scipy.spatial import cKDTree

from icp_reference import Matcher, Result, d2f, evaluate, limit32, move, xyz32  # noqa: F401  (move: used by the tests)

CAND = 8        # proposed candidates beyond max_nn
CHUNK = 100000  # queries re-ranked at a time


class Normals(NamedTuple):
    normals: np.ndarray   # (n, 3) float32, (0, 0, 0) where there is none
    count: np.ndarray     # (n,) neighbourhood sizes
    eigvals: np.ndarray   # (n, 3) ascending eigenvalues of the covariance (0 where the normal is zero)


def neighbourhoods(p32, radius, max_nn, tree=None):
    """(n, max_nn) int64 indices per point, ascending by (float32 d2, index), -1 padded: the points of the same cloud with
    d2 <= float32(radius**2), at most max_nn of them."""
    p32 = np.ascontiguousarray(p32, np.float32)
    n = len(p32)
    out = np.full((n, max_nn), -1, np.int64)
    if n == 0:
        return out
    tree = tree or cKDTree(p32.astype(np.float64))
    limit = limit32(radius)
    bound = float(np.sqrt(np.float64(limit))) * (1.0 + 1e-5) + 1e-30
    take = min(n, max_nn + CAND)
    for lo in range(0, n, CHUNK):
        q = p32[lo:lo + CHUNK]
        nq = len(q)
        dist, cand = tree.query(q.astype(np.float64), k=take, distance_upper_bound=bound, workers=-1)
        dist, cand = dist.reshape(nq, take), cand.reshape(nq, take)
        valid = cand < n
        cd2 = np.where(valid, d2f(q[:, None, :], p32[np.minimum(cand, n - 1)]), np.float32(np.inf))
        cd2[~(cd2 <= limit)] = np.inf
        order = np.lexsort((np.where(valid, cand, n), cd2), axis=1)[:, :max_nn]
        rows = np.arange(nq)[:, None]
        kd2, ki = cd2[rows, order], cand[rows, order]
        ki = np.where(np.isfinite(kd2), ki, -1)
        if take < max_nn:  # a cloud of fewer than max_nn points
            ki = np.concatenate([ki, np.full((nq, max_nn - take), -1, np.int64)], 1)
            kd2 = np.concatenate([kd2, np.full((nq, max_nn - take), np.inf, np.float32)], 1)
        # a proposal that stops short of the ball can leave out a point that ties with or beats the max_nn-th place
        full = valid[:, -1] & (take < n)
        last = kd2[:, -1]
        reach = np.where(np.isfinite(last), np.sqrt(last.astype(np.float64)) * (1.0 + 1e-5) + 1e-30, bound)
        for i in np.flatnonzero(full & ~(dist[:, -1] > reach)):
            ball = np.asarray(tree.query_ball_point(q[i].astype(np.float64), min(reach[i], bound)), np.int64)
            bd2 = d2f(q[i][None, :], p32[ball])
            ok = bd2 <= limit
            ball, bd2 = ball[ok], bd2[ok]
            sel = np.lexsort((ball, bd2))[:max_nn]
            ki[i] = -1
            ki[i, :len(sel)] = ball[sel]
        out[lo:lo + nq] = ki
    return out


def estimate_normals(p32, radius, max_nn, tree=None):
    p32 = np.ascontiguousarray(p32, np.float32)
    nb = neighbourhoods(p32, radius, max_nn, tree)
    have = nb >= 0
    count = have.sum(1)
    pts = np.where(have[..., None], p32[np.maximum(nb, 0)].astype(np.float64), 0.0)
    mean = pts.sum(1) / np.maximum(count, 1)[:, None]
    dev = np.where(have[..., None], pts - mean[:, None, :], 0.0)
    cov = np.einsum("nka,nkb->nab", dev, dev)
    w, v = np.linalg.eigh(cov)
    zero = (count < 3) | np.all(cov.reshape(len(cov), 9) == 0.0, axis=1)
    normals = np.where(zero[:, None], 0.0, v[:, :, 0]).astype(np.float32)
    return Normals(normals, count, np.where(zero[:, None], 0.0, w))


def box_centre(t32):
    t = np.asarray(t32, np.float64)
    return 0.5 * (t.min(0) + t.max(0))


def min_norm_solve(A, rhs, cut=1e-12):
    """The minimum-norm least-squares solution of A x = rhs (A symmetric), eigenvalues <= cut * the largest dropped."""
    w, V = np.linalg.eigh(A)
    top = w.max()
    keep = w > cut * top if top > 0 else np.zeros(len(w), bool)
    return V[:, keep] @ ((V[:, keep].T @ rhs) / w[keep])


def euler_matrix(x):
    """open3d's TransformVector6dToMatrix4d: [Rz(x[2]) Ry(x[1]) Rx(x[0]), x[3:]]."""
    ca, sa, cb, sb, cg, sg = np.cos(x[0]), np.sin(x[0]), np.cos(x[1]), np.sin(x[1]), np.cos(x[2]), np.sin(x[2])
    Rx = np.array([[1, 0, 0], [0, ca, -sa], [0, sa, ca]])
    Ry = np.array([[cb, 0, sb], [0, 1, 0], [-sb, 0, cb]])
    Rz = np.array([[cg, -sg, 0], [sg, cg, 0], [0, 0, 1]])
    T = np.eye(4)
    T[:3, :3] = Rz @ Ry @ Rx
    T[:3, 3] = x[3:]
    return T


def plane_step(p, q, nrm, origin):
    """dT (4x4) of one point-to-plane step over the pairs (p, q) with target normals nrm, about `origin`."""
    o = np.asarray(origin, np.float64)
    p, q, nrm = np.asarray(p, np.float64) - o, np.asarray(q, np.float64) - o, np.asarray(nrm, np.float64)
    r = np.einsum("na,na->n", p - q, nrm)
    J = np.concatenate([np.cross(p, nrm), nrm], 1)
    x = min_norm_solve(J.T @ J, -(J.T @ r))
    dT = euler_matrix(x)
    shift, back = np.eye(4), np.eye(4)
    shift[:3, 3], back[:3, 3] = -o, o
    return back @ dT @ shift


def icp_point_to_plane(source, target, max_distance, normal_radius, init=None, max_iterations=30, relative_fitness=1e-6, relative_rmse=1e-6, normal_max_nn=30,
                       origin=None):
    """origin: the centre of the box the library takes for the target (by default the target's own bounding box)."""
    s32, t32 = xyz32(source), xyz32(target)
    T = np.eye(4) if init is None else np.array(init, np.float64)
    if len(s32) == 0 or len(t32) == 0:
        return Result(T, 0.0, 0.0, 0, 0)
    o = box_centre(t32) if origin is None else np.asarray(origin, np.float64)
    nrm = estimate_normals(t32, normal_radius, normal_max_nn).normals
    matcher = Matcher(t32)
    e = evaluate(s32, matcher, T, max_distance)
    it = 0
    while it < max_iterations and e.correspondences >= 3:
        T = plane_step(e.src, e.dst, nrm[e.index[e.index >= 0]], o) @ T
        prev, e = e, evaluate(s32, matcher, T, max_distance)
        it += 1
        if abs(prev.fitness - e.fitness) < relative_fitness and abs(prev.inlier_rmse - e.inlier_rmse) < relative_rmse:
            break
    return Result(T, e.fitness, e.inlier_rmse, it, e.correspondences)
