"""The kNN reference of tests/knn_reference.py checked on its own, without a GPU: it must reproduce the CPU oracle's
mean distances bit for bit, and its lists must equal a full brute force, limits included."""
import math

import numpy as np
import pytest

from cwipc_util_b200 import synthetic

import knn_reference as ref

DT = synthetic.cwipc_point_numpy_dtype


def shifted(pts, by):
    out = pts.copy()
    for a in "xyz":
        out[a] = (pts[a].astype(np.float64) + by).astype(np.float32)
    return out


def with_duplicates(pts, m, seed):
    """m copies of one point spread over the cloud, plus pairs of copies of others."""
    out = pts.copy()
    rng = np.random.default_rng(seed)
    where = rng.choice(len(pts), m, replace=False)
    out[where[: m // 2]] = out[where[0]]
    out[where[m // 2:]] = pts[rng.choice(len(pts), m - m // 2)]
    return out


def random_volume(n, seed, extent=0.3):
    rng = np.random.default_rng(seed)
    pts = np.zeros(n, DT)
    for a in "xyz":
        pts[a] = rng.uniform(-extent, extent, n).astype(np.float32)
    pts["tile"] = 1
    return pts


@pytest.mark.parametrize("k", [1, 30, 63, 64, 200, 511])
def test_reference_mean_equals_the_oracle(orc, k):
    n = 20000 if k <= 64 else 6000
    base = synthetic.add_outliers(synthetic.camera_cloud(n, seed=k), 0.02, seed=k)
    for pts in (with_duplicates(base, 50, seed=k), shifted(base, 3e3), shifted(base, -1e4)):
        lists = ref.ref_lists(pts, pts, k)
        assert np.array_equal(ref.ref_mean(lists, k), orc.knn_mean_distances(pts, k))
        assert np.all(lists[:, 0] == 0.0) and np.all(np.diff(lists, axis=1) >= 0)


@pytest.mark.parametrize("n,k", [(2, 1), (40, 30), (700, 30), (1500, 64), (600, 511)])
def test_reference_mean_equals_the_oracle_brute_force(orc, n, k):
    pts = with_duplicates(random_volume(n, seed=n + k, extent=0.05), max(2, n // 20), seed=n)
    k = min(k, n - 1)
    want = orc.knn_mean_distances(pts, k, bruteforce=True)
    assert np.array_equal(ref.ref_mean(ref.ref_lists(pts, pts, k), k), want)
    assert np.array_equal(ref.ref_mean(ref.ref_lists(shifted(pts, -1e4), shifted(pts, -1e4), k), k),
                          orc.knn_mean_distances(shifted(pts, -1e4), k, bruteforce=True))


def brute_lists(cloud, queries, k, limits=None):
    d2 = ref.d2f(queries, cloud)
    if limits is not None:
        d2[~(d2 <= np.asarray(limits, np.float32)[:, None])] = np.inf
    out = np.full((len(queries), k + 1), np.inf, np.float32)
    s = np.sort(d2, axis=1)[:, :k + 1]
    out[:, :s.shape[1]] = s
    return out


@pytest.mark.parametrize("k", [1, 7, 31, 32, 100])
def test_reference_lists_equal_brute_force_with_limits(k):
    cloud = with_duplicates(random_volume(3000, seed=k), 40, seed=k)
    rng = np.random.default_rng(k)
    queries = np.concatenate([cloud[rng.choice(3000, 300, replace=False)], random_volume(200, seed=k + 1, extent=0.4),
                              shifted(random_volume(50, seed=k + 2), 100.0)])
    full = brute_lists(cloud, queries, k)
    assert np.array_equal(ref.ref_lists(cloud, queries, k), full)
    nq = len(queries)
    j = int(rng.integers(0, k + 1))
    exact = full[:, j]
    below = np.nextafter(exact, np.float32(-np.inf))
    for limits in (np.zeros(nq, np.float32), np.full(nq, -1.0, np.float32), np.full(nq, np.nan, np.float32),
                   np.full(nq, np.inf, np.float32), exact, below):
        got = ref.ref_lists(cloud, queries, k, limits)
        assert np.array_equal(got, brute_lists(cloud, queries, k, limits))
    assert np.all(ref.ref_lists(cloud, queries, k, np.full(nq, np.nan, np.float32)) == np.inf)
    assert np.all(ref.ref_lists(cloud, queries, k, np.full(nq, -1.0, np.float32)) == np.inf)
    assert np.array_equal(ref.ref_lists(cloud, queries, k, exact)[:, j], exact)       # the limit itself is reported
    got = ref.ref_lists(cloud, queries, k, below)
    assert not np.any(got == exact[:, None]) and np.all(got[:, j] == np.inf)   # ... and nothing above it


def test_reference_lists_of_small_and_empty_clouds():
    cloud = random_volume(5, seed=3)
    q = random_volume(4, seed=4)
    got = ref.ref_lists(cloud, q, 7)
    assert np.array_equal(got, brute_lists(cloud, q, 7))
    assert np.all(np.isinf(got[:, 5:])) and np.all(np.isfinite(got[:, :5]))
    assert np.all(ref.ref_lists(cloud[:0], q, 7) == np.inf)
    assert np.all(np.isinf(ref.ref_mean(got, 7)))       # padding inside [1..k]: the mean is +inf
    assert np.all(np.isfinite(ref.ref_mean(got, 4)))


def test_reference_open_set_and_sums():
    x = np.array([0.0, 0.5, 0.85, -0.9, 2.0], np.float32)
    kth2 = np.array([0.01, 0.01, 0.01, 0.04, np.inf], np.float32)
    assert list(ref.ref_open(x, kth2, 5, -1.0, 1.0)) == [3, 4]     # -0.9 - 0.2 < -1; an infinite sphere
    assert list(ref.ref_open(x, kth2, 5, -np.inf, np.inf)) == [4]  # an infinite sphere is never inside
    assert list(ref.ref_open(x, kth2, 5, 1.0, -1.0)) == [0, 1, 2, 3, 4]
    assert list(ref.ref_open(x, None, 3, -1.0, 1.0)) == [0, 1, 2]
    d = np.random.default_rng(0).uniform(0, 1, 100001).astype(np.float32)
    s, sq = ref.exact_sums(d)
    assert s == math.fsum(float(v) for v in d)
    assert abs(s - d.astype(np.float64).sum()) <= ref.sum_bound(len(d), d)[0]


def test_exact_keep_check_holds_the_exact_threshold():
    pts = random_volume(5000, seed=5)
    d = np.random.default_rng(5).gamma(4.0, 0.01, 5000).astype(np.float32)
    s, sq = ref.exact_sums(d)
    thr = ref.threshold_formula(s, sq, len(d), 1.0)
    keep = ~(d.astype(np.float64) > thr)
    assert ref.exact_keep_check(pts, pts[keep], d, 1.0) == keep.sum()
    nearest = int(np.argmin(np.abs(d.astype(np.float64) - thr)))
    flipped = keep.copy()
    flipped[nearest] = not flipped[nearest]
    with pytest.raises(AssertionError):   # the point nearest the threshold is still far outside the sums' error
        ref.exact_keep_check(pts, pts[flipped], d, 1.0)
