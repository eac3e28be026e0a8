"""A plain numpy/scipy reference of the kNN partition building blocks and of the outlier threshold (no library calls).

The distances are exact: d² = (dx*dx + dy*dy) + dz*dz with every operation in float32, as the library computes it
(`-fmad=false`) and as PCL's L2_Simple<float> does.  A float64 cKDTree only proposes candidates: the k+1 nearest, then
every point within sqrt(max d²) * (1 + 1e-5) of the query, which holds every point whose float32 d² can be among the
k+1 smallest.  Means are a sequential float64 sum of sqrt(d²[1..k]) divided by k, cast to float32 -- np.cumsum adds
in order; np.sum adds pairwise and gives other bits.
"""
import math

import numpy as np
from scipy.spatial import cKDTree

U = 2.0 ** -53   # unit roundoff of float64
CHUNK = 8192     # queries per block of the candidate search (bounds the memory of k = 511)


def _xyz32(pts):
    return [np.ascontiguousarray(pts[a], np.float32) for a in "xyz"]


def _xyz64(pts):
    return np.stack([np.asarray(pts[a], np.float64) for a in "xyz"], 1)


def d2f(q, c):
    """float32 ((dx*dx + dy*dy) + dz*dz) for every pair: shape (len(q), len(c))."""
    qx, qy, qz = (v[:, None] for v in _xyz32(q))
    cx, cy, cz = (v[None, :] for v in _xyz32(c))
    dx, dy, dz = qx - cx, qy - cy, qz - cz
    return (dx * dx + dy * dy) + dz * dz


def _d2_rows(q32, c32, idx):
    """float32 d² from query i to cloud points idx[i, :]."""
    dx = q32[0][:, None] - c32[0][idx]
    dy = q32[1][:, None] - c32[1][idx]
    dz = q32[2][:, None] - c32[2][idx]
    return (dx * dx + dy * dy) + dz * dz


def ref_lists(cloud, queries, k, limits=None):
    """(nq, k+1) float32: per query the k+1 smallest float32 d² to `cloud` with d² <= limit, ascending, +inf padded.
    limits=None: no limit.  A NaN limit selects nothing (d² <= NaN is false)."""
    kk = k + 1
    nq, n = len(queries), len(cloud)
    out = np.full((nq, kk), np.inf, np.float32)
    if n == 0 or nq == 0:
        return out
    c32, q32 = _xyz32(cloud), _xyz32(queries)
    tree = cKDTree(_xyz64(cloud))
    q64 = _xyz64(queries)
    take = min(n, kk + 8)
    for lo in range(0, nq, CHUNK):
        hi = min(nq, lo + CHUNK)
        rows = slice(lo, hi)
        dist, idx = tree.query(q64[rows], k=take, workers=-1)
        idx = idx.reshape(hi - lo, take)
        dist = dist.reshape(hi - lo, take)
        qs = [v[rows] for v in q32]
        d2 = np.sort(_d2_rows(qs, c32, idx), axis=1)
        # the candidates hold the answer when every point they miss is farther than the ball around the kk-th
        radius = np.sqrt(d2[:, min(kk, take) - 1].astype(np.float64)) * (1.0 + 1e-5)
        short = np.flatnonzero(~(dist[:, -1] > radius)) if take < n else np.zeros(0, np.int64)
        out[rows, :min(kk, take)] = d2[:, :kk]
        for i in short:
            ball = np.asarray(tree.query_ball_point(q64[lo + i], radius[i]), np.int64)
            d = np.sort(_d2_rows([v[i:i + 1] for v in qs], c32, ball[None, :])[0])[:kk]
            out[lo + i, :] = np.inf
            out[lo + i, :len(d)] = d
    return out if limits is None else with_limits(out, limits)


def with_limits(lists, limits):
    """The lists of ref_lists(..., limits=None) cut to d² <= limit: the k+1 smallest within the limit are a prefix of the
    k+1 smallest overall."""
    out = lists.copy()
    out[~(out <= np.asarray(limits, np.float32)[:, None])] = np.inf
    return out


def ref_mean(lists, k):
    """float32 mean distance to the k nearest (element 0 is the query itself): a sequential float64 sum.  +inf where
    the list is padded inside [1..k]."""
    s = np.cumsum(np.sqrt(lists[:, 1:k + 1].astype(np.float64)), axis=1)[:, -1]
    return (s / k).astype(np.float32)


def ref_kth2(lists, k):
    return lists[:, k]


def ref_open(x, kth2, nquery, x_lo, x_hi):
    """Sorted indices of the queries whose (k+1)-th neighbour sphere is not strictly inside (x_lo, x_hi), in float64 as
    mark_open_kernel: rk = sqrt(kth2) * (1 + 1e-6).  kth2=None: every query is open."""
    if kth2 is None:
        return np.arange(nquery, dtype=np.uint32)
    xx = np.asarray(x[:nquery], np.float32).astype(np.float64)
    rk = np.sqrt(np.asarray(kth2[:nquery], np.float32).astype(np.float64)) * (1.0 + 1e-6)
    lo, hi = float(np.float32(x_lo)), float(np.float32(x_hi))
    return np.flatnonzero(~((xx - rk > lo) & (xx + rk < hi))).astype(np.uint32)


def exact_sums(d):
    """Correctly rounded sum d and sum float32(d*d), both over float64 terms."""
    d = np.asarray(d, np.float32)
    return math.fsum(d.astype(np.float64)), math.fsum((d * d).astype(np.float64))


def sum_bound(n, d):
    """Bounds of the rounding error of the library's fixed-order double sums (stats_kernel: at most ceil(n/65536) serial
    adds per thread, an 8-level tree, 256 serial adds): 2 * depth * 2^-53 * sum |term|, for (sum, sum of squares)."""
    d = np.asarray(d, np.float32)
    depth = -(-n // 65536) + 8 + 256
    return (2.0 * depth * U * math.fsum(np.abs(d).astype(np.float64)),
            2.0 * depth * U * math.fsum((d * d).astype(np.float64)))


def threshold_formula(s, sq, n, mul):
    """outlier_threshold's order of operations, in float64 (pcl::StatisticalOutlierRemoval); n = 1 gives NaN or inf."""
    s, sq, n = np.float64(s), np.float64(sq), np.float64(n)
    with np.errstate(divide="ignore", invalid="ignore"):
        mean = s / n
        variance = (sq - s * s / n) / (n - np.float64(1.0))
        return float(mean + np.float64(np.float32(mul)) * np.sqrt(variance))


def threshold_error(s, sq, n, mul, d):
    """Bound of |library threshold - threshold from the exact sums|: the sums' error propagated through the formula, plus
    the formula's own rounding (a few ulps of each intermediate, on both sides)."""
    bs, bsq = sum_bound(n, d)
    m = abs(float(np.float32(mul)))
    var_num = sq - s * s / n
    sigma = math.sqrt(max(var_num, 0.0) / (n - 1.0))
    num_err = bsq + 2 * abs(s) / n * bs + 16 * U * (abs(sq) + s * s / n)
    if sigma == 0.0:
        return math.inf
    return (bs / n + m * num_err / (2.0 * sigma * (n - 1.0)) + 16 * U * (abs(s) / n + m * sigma))


def exact_keep_check(pts, got, d, mul, whole=True):
    """`got` must be pts[!(d > thr)] in order, with thr from the exact sums of `d` by outlier_threshold's formula.  Only
    points whose d lies within the propagated error of the library's fixed-order sums may go either way.  whole=False:
    `got` may go on behind the kept points of `pts` (the next tile group).  Returns how many records of `got` are pts'."""
    d = np.asarray(d, np.float32)
    n = len(d)
    s, sq = exact_sums(d)
    thr = threshold_formula(s, sq, n, mul)
    eps = threshold_error(s, sq, n, mul, d)
    dd = d.astype(np.float64)
    amb = np.abs(dd - thr) <= eps
    assert amb.sum() <= 8, f"{amb.sum()} points within {eps} of the threshold {thr}"
    drop = (dd > thr) & ~amb
    keep = ~(dd > thr) & ~amb
    gi = 0
    for i in range(n):
        if gi < len(got) and not drop[i] and got[gi] == pts[i]:
            gi += 1
        else:
            assert not keep[i], f"point {i} (d={dd[i]!r}, thr={thr!r}, eps={eps:g}) was dropped"
    assert gi == len(got) or not whole, f"{len(got) - gi} kept points are not inliers of the input in order (thr={thr!r})"
    return gi
