"""A plain numpy/scipy reference of cwipc_cuda_icp (no library calls): the loop the header states, step by step.

- Moving: p' = float32((((m[r][0]*x + m[r][1]*y) + m[r][2]*z) + m[r][3])) in float64 -- cwipc_cuda_transform's arithmetic.
- Matching: a float64 cKDTree proposes candidates, the nearest 8 and, where those do not settle it, every target point
  within (1 + 1e-5) times the nearest distance.  They are ranked by the exact float32 d2 = (dx*dx + dy*dy) + dz*dz and then
  by index, as tests/knn_reference.py ranks distances; a pair counts iff d2 <= float32(max_distance**2).
- Solving: Kabsch with numpy.linalg.svd on the pairs in float64, the sign of the last singular vector fixed so that the
  rotation is proper.
- Looping: T <- dT * T, always applied to the original source points; stop after max_iterations updates, with fewer than
  3 correspondences, or when fitness and rmse both change by less than the criteria.
"""
from typing import NamedTuple

import numpy as np
from scipy.spatial import cKDTree

CAND = 8  # nearest candidates per query before the ball check


def xyz32(pts):
    """(n, 3) float32 from a cwipc point record array, or an (n, 3) array as it is."""
    if pts.dtype.names:
        return np.stack([np.asarray(pts[a], np.float32) for a in "xyz"], 1)
    return np.asarray(pts, np.float32)


def move(p32, T):
    """float32 (n, 3): every point moved by the 4x4 T in float64, in the order the header states, rounded to float32."""
    T = np.asarray(T, np.float64)
    x, y, z = (p32[:, a].astype(np.float64) for a in range(3))
    return np.stack([(((T[r, 0] * x + T[r, 1] * y) + T[r, 2] * z) + T[r, 3]).astype(np.float32) for r in range(3)], 1)


def d2f(q32, c32):
    """float32 ((dx*dx + dy*dy) + dz*dz), elementwise over matching rows (or broadcast)."""
    d = q32 - c32
    return (d[..., 0] * d[..., 0] + d[..., 1] * d[..., 1]) + d[..., 2] * d[..., 2]


def limit32(max_distance):
    return np.float32(np.float64(max_distance) * np.float64(max_distance))


class Matcher:
    """The target's search structure, built once (as the library builds its index once per call)."""

    def __init__(self, target32):
        self.t32 = np.ascontiguousarray(target32, np.float32)
        self.tree = cKDTree(self.t32.astype(np.float64)) if len(self.t32) else None

    def nearest(self, q32, limit):
        """(index, d2) per query: the smallest (float32 d2, index) with d2 <= limit; index -1 (and d2 inf) when none."""
        nq, n = len(q32), len(self.t32)
        idx = np.full(nq, -1, np.int64)
        d2 = np.full(nq, np.inf, np.float32)
        if nq == 0 or n == 0:
            return idx, d2
        bound = float(np.sqrt(np.float64(limit))) * (1.0 + 1e-5) + 1e-30
        take = min(n, CAND)
        dist, cand = self.tree.query(q32.astype(np.float64), k=take, distance_upper_bound=bound, workers=-1)
        dist, cand = dist.reshape(nq, take), cand.reshape(nq, take)
        found = np.isfinite(dist[:, 0])
        valid = cand < n
        cd2 = np.where(valid, d2f(q32[:, None, :], self.t32[np.minimum(cand, n - 1)]), np.float32(np.inf))
        # every point that can tie with or beat the best float32 d2 lies within (1 + 1e-5) of the nearest float64 distance
        radius = dist[:, 0] * (1.0 + 1e-5) + 1e-30
        short = np.flatnonzero(found & valid[:, -1] & ~(dist[:, -1] > radius)) if take < n else np.zeros(0, np.int64)
        key_d2 = cd2.copy()
        key_d2[~(cd2 <= limit)] = np.inf
        order = np.lexsort((np.where(valid, cand, n), key_d2), axis=1)[:, 0]
        rows = np.arange(nq)
        best_d2, best_i = key_d2[rows, order], cand[rows, order]
        for i in short:
            ball = np.asarray(self.tree.query_ball_point(q32[i].astype(np.float64), radius[i]), np.int64)
            bd2 = d2f(q32[i][None, :], self.t32[ball])
            ok = bd2 <= limit
            if ok.any():
                j = np.lexsort((ball[ok], bd2[ok]))[0]
                best_d2[i], best_i[i] = bd2[ok][j], ball[ok][j]
        hit = best_d2 <= limit
        idx[hit] = best_i[hit]
        d2[hit] = best_d2[hit]
        return idx, d2


def kabsch(p, q):
    """The proper rigid motion (4x4) that minimises sum |R p_i + t - q_i|^2, from numpy.linalg.svd."""
    o = np.asarray(q[0], np.float64)  # coordinates relative to a point of the pairs keep clouds far from the origin accurate
    p, q = np.asarray(p, np.float64) - o, np.asarray(q, np.float64) - o
    mp, mq = p.mean(0), q.mean(0)
    H = (p - mp).T @ (q - mq)
    U, _, Vt = np.linalg.svd(H)
    D = np.diag([1.0, 1.0, np.sign(np.linalg.det(Vt.T @ U.T)) or 1.0])
    R = Vt.T @ D @ U.T
    T = np.eye(4)
    T[:3, :3] = R
    T[:3, 3] = (mq + o) - R @ (mp + o)
    return T


class Evaluation(NamedTuple):
    correspondences: int
    fitness: float
    inlier_rmse: float
    src: np.ndarray    # the moved source points of the pairs, float32
    dst: np.ndarray    # their target points, float32
    index: np.ndarray  # per source point: the target index of its pair, -1 without one


def evaluate(source32, matcher, T, max_distance):
    moved = move(source32, T)
    idx, d2 = matcher.nearest(moved, limit32(max_distance))
    hit = idx >= 0
    n = int(hit.sum())
    fitness = n / len(source32) if len(source32) else 0.0
    rmse = float(np.sqrt(np.sum(d2[hit].astype(np.float64)) / n)) if n else 0.0
    return Evaluation(n, fitness, rmse, moved[hit], matcher.t32[idx[hit]], idx)


class Result(NamedTuple):
    matrix: np.ndarray
    fitness: float
    inlier_rmse: float
    iterations: int
    correspondences: int


def icp(source, target, max_distance, init=None, max_iterations=30, relative_fitness=1e-6, relative_rmse=1e-6):
    s32, t32 = xyz32(source), xyz32(target)
    T = np.eye(4) if init is None else np.array(init, np.float64)
    if len(s32) == 0 or len(t32) == 0:
        return Result(T, 0.0, 0.0, 0, 0)
    matcher = Matcher(t32)
    e = evaluate(s32, matcher, T, max_distance)
    it = 0
    while it < max_iterations and e.correspondences >= 3:
        T = kabsch(e.src, e.dst) @ T
        prev, e = e, evaluate(s32, matcher, T, max_distance)
        it += 1
        if abs(prev.fitness - e.fitness) < relative_fitness and abs(prev.inlier_rmse - e.inlier_rmse) < relative_rmse:
            break
    return Result(T, e.fitness, e.inlier_rmse, it, e.correspondences)
