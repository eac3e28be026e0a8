"""Comparisons shared by the GPU parity tests and __graft_entry__.smoke() (bars: BASELINE.json north_star)."""
import itertools

import numpy as np


def sor_group_check(grp, got, pos, d, mul):
    """`got[pos:]` must start with the inliers of `grp` as decided by the oracle's distances `d`, except that points
    within 1e-6 (relative) of the threshold may go either way.  Returns the position behind the group."""
    n = len(grp)
    dd = d.astype(np.float64)
    s, sq = dd.sum(), (d * d).astype(np.float64).sum()
    thr = s / n + mul * np.sqrt((sq - s * s / n) / (n - 1))
    keep = ~(dd > thr)
    ambiguous = np.flatnonzero(np.abs(dd - thr) <= 1e-6 * abs(thr))
    assert len(ambiguous) <= 12, f"{len(ambiguous)} points within 1e-6 of the threshold"
    for choice in itertools.product((False, True), repeat=len(ambiguous)):
        k2 = keep.copy()
        k2[ambiguous] = choice
        want = grp[k2]
        if pos + len(want) <= len(got) and np.array_equal(got[pos:pos + len(want)], want):
            return pos + len(want)
    raise AssertionError(f"group of {n} points at output position {pos}: kept points differ from the oracle's beyond threshold ties (thr={thr}, {len(ambiguous)} ties)")


def sor_set_check(grp, got, d, mul):
    """Order-free variant for partitioned results: `got` (any order) must contain every point of `grp` that is an
    inlier by more than 1e-6 of the threshold, and none that is an outlier by more than that."""
    n = len(grp)
    dd = d.astype(np.float64)
    s, sq = dd.sum(), (d * d).astype(np.float64).sum()
    thr = s / n + mul * np.sqrt((sq - s * s / n) / (n - 1))
    void = np.dtype((np.void, grp.dtype.itemsize))
    g = np.ascontiguousarray(grp).view(void).reshape(-1)
    o = np.ascontiguousarray(got).view(void).reshape(-1)
    present = np.isin(g, o)
    sure_keep, sure_drop = dd <= thr * (1 - 1e-6), dd > thr * (1 + 1e-6)
    assert present[sure_keep].all(), "an inlier was dropped"
    # a dropped point may still be `present` when an identical record survives elsewhere: count instead
    assert np.isin(o, g).all(), "output holds a point that is not in the input"
    assert len(got) <= int((~sure_drop).sum()) and len(got) >= int(sure_keep.sum())


def per_tile_check(orc, pts, got, k, mul):
    """ref: src/cwipc_filters.cpp:238-261 -- groups in first-appearance order of the tile value, tile 0 = the whole cloud"""
    _, first = np.unique(pts["tile"], return_index=True)
    tiles = pts["tile"][np.sort(first)]
    pos = 0
    for t in tiles:
        grp = pts if t == 0 else pts[pts["tile"] == t]
        if len(grp) <= k:
            assert np.array_equal(got[pos:pos + len(grp)], grp)
            pos += len(grp)
        else:
            pos = sor_group_check(grp, got, pos, orc.knn_mean_distances(grp, k), mul)
    assert pos == len(got)


def canonical_ranks(keys6):
    l = keys6[:, :3].astype(np.int64)
    m = np.zeros(len(l), np.int64)
    for b in range(21):
        m |= ((l[:, 0] >> b) & 1) << (3 * b + 2)
        m |= ((l[:, 1] >> b) & 1) << (3 * b + 1)
        m |= ((l[:, 2] >> b) & 1) << (3 * b)
    v = keys6[:, 3:].astype(np.int64)
    order = np.lexsort((v[:, 0], v[:, 1], v[:, 2], m))
    full = np.concatenate([m[:, None], v[:, ::-1]], axis=1)[order]
    heads = np.ones(len(full), bool)
    heads[1:] = np.any(full[1:] != full[:-1], axis=1)
    ranks = np.empty(len(full), np.int64)
    ranks[order] = np.cumsum(heads) - 1
    return ranks


def assert_points_close(got, want, cs, counts=None):
    """xyz within 1e-5 relative (scale = max(|coordinate|, voxel size)), colours within 1 LSB, tiles exact, same order.

    `want` is the restated pcl::CentroidPoint: a FLOAT running sum in input order.  For a voxel of n points that sum is
    itself only accurate to about n * 2^-25 relative (every add rounds the partial sum), which passes 1e-5 from a few
    hundred points per voxel on -- 8 M points at voxel 0.01 put 8 600 points into the voxels at the tip of the synthetic
    cloud and the oracle is 1.8e-5 away from the true mean there.  With `counts` the bar per voxel is therefore
    max(1e-5, n * 2^-25); assert_exact_means() states what the GPU itself guarantees."""
    assert len(got) == len(want)
    bar = 1e-5 if counts is None else np.maximum(1e-5, counts.astype(np.float64) * 2.0 ** -25)
    for a in "xyz":
        scale = np.maximum(np.abs(want[a].astype(np.float64)), cs)
        err = np.abs(got[a].astype(np.float64) - want[a].astype(np.float64)) / scale
        assert np.all(err <= bar), f"{a}: max rel err {err.max()} (bar {np.max(bar)})"
    for c in "rgb":
        assert np.abs(got[c].astype(np.int32) - want[c].astype(np.int32)).max(initial=0) <= 1
    assert np.array_equal(got["tile"], want["tile"])


def exact_voxels(pts, ranks, nvox=None):
    """Plain reference of a voxel downsample, given each point's voxel rank (its output position): the point count
    (int64), the float64 mean of x, y, z, the int64 sums of r, g, b, the colours as sum // count, and the OR of the
    tiles."""
    nvox = int(ranks.max()) + 1 if nvox is None else nvox
    ranks = np.asarray(ranks, np.int64)
    ref = {"count": np.bincount(ranks, minlength=nvox).astype(np.int64)}
    assert np.all(ref["count"] > 0), "a voxel rank without points"
    for a in "xyz":
        ref[a] = np.bincount(ranks, weights=pts[a].astype(np.float64), minlength=nvox) / ref["count"]
    for c in "rgb":  # float64 sums of integers below 2^53 are exact
        s = np.bincount(ranks, weights=pts[c].astype(np.float64), minlength=nvox).astype(np.int64)
        ref["sum_" + c] = s
        ref[c] = s // ref["count"]
    tile = np.zeros(nvox, np.uint8)
    for b in range(8):
        tile |= (np.bincount(ranks, weights=(pts["tile"] >> b) & 1, minlength=nvox) > 0).astype(np.uint8) << b
    ref["tile"] = tile
    return ref


def assert_exact_means(got, pts, ranks, counts, cs, want=None):
    """The library's centroids are sums in exact integer arithmetic (offsets from the voxel's origin in 2^-46-ish fixed
    point), rounded once: equal to the float64 mean of the voxel's points to within one float32 ulp -- the ulp taken at
    max(|coordinate|, cellsize / 1024), since next to a coordinate plane a float32 resolves more than the fixed point does.
    Colours are the exact integer means floor(sum / count) and tiles the OR of the voxel's tiles, both bit for bit.  With
    `want` (the oracle's output, pcl::CentroidPoint's float running sum) the colours must also equal the oracle's wherever
    the voxel's channel sum is below 2^24, where that float sum is exact.  `counts` (or None) are the expected counts."""
    ref = exact_voxels(pts, ranks, len(got) if counts is None else len(counts))
    assert len(got) == len(ref["count"]), f"{len(got)} voxels, the reference has {len(ref['count'])}"
    if counts is not None:
        assert np.array_equal(ref["count"], counts)
    errors = []

    def report(what, bad, got_v, want_v):
        if len(bad):
            v = bad[0]
            errors.append(f"{what}: {len(bad)} voxels differ, first voxel {v} ({ref['count'][v]} points): got {got_v[v]!r}, want {want_v[v]!r}")

    for c in "rgb":
        report(f"{c} != floor(sum / count)", np.flatnonzero(got[c].astype(np.int64) != ref[c]), got[c], ref[c])
        if want is not None:
            report(f"{c} != oracle where sum < 2^24", np.flatnonzero((ref["sum_" + c] < (1 << 24)) & (got[c] != want[c])), got[c], want[c])
    report("tile != OR of the tiles", np.flatnonzero(got["tile"] != ref["tile"]), got["tile"], ref["tile"])
    for a in "xyz":
        ulp = np.spacing(np.maximum(np.abs(ref[a]), cs / 1024.0).astype(np.float32)).astype(np.float64)
        report(f"{a} more than one float32 ulp from the exact mean", np.flatnonzero(~(np.abs(got[a].astype(np.float64) - ref[a]) <= ulp)), got[a], ref[a])
    assert not errors, "; ".join(errors)
