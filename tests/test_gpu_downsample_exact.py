"""Every downsample path against exact per-voxel sums.

The kernels sum each voxel in integers (fixed-point coordinates, integer colour sums and counts), so the output is fully
determined: centroids within one float32 ulp of the float64 mean, colours exactly floor(sum / count), tiles exactly the
OR (parity_helpers.assert_exact_means).  Every cloud goes through every path that fills a voxel slot: cwipc_downsample
with both voxel signs and each internal path (CWIPC_CUDA_DS_PATH), cwipc_cuda_downsample_pertile group by group, and the
slab downsample with a one-rank communicator.  The clouds aim at where this kernel can go wrong: run lengths around the
lane (8 points), warp tile (256) and queue (80 records) sizes, heavy contended voxels, colour sums across 2^24 (the
float division) and 2^32 (the width of the slot's sums), the fixed-point scale at its limits, and awkward geometry.
"""
import functools

import numpy as np
import pytest

from cwipc_util_b200 import synthetic
from parity_helpers import assert_exact_means, canonical_ranks, exact_voxels

DT = synthetic.cwipc_point_numpy_dtype
PATHS = (None, "twopass", "generic", "smalltable")   # None: the default (fused single pass when voxelsize > 0)


def upload(cw, pts, cellsize=0.0):
    pc = cw.cwipc_from_numpy_array(pts, 1)
    pc._set_cellsize(cellsize)
    return pc


def first_appearance(pts):
    _, first = np.unique(pts["tile"], return_index=True)
    return [int(t) for t in pts["tile"][np.sort(first)]]


def oracle_ranks(orc, pts, voxel, pc_cellsize):
    want, cs, keys6, counts = orc.downsample(pts, voxel, pc_cellsize, want_keys=True)
    assert want is not None
    return want, cs, canonical_ranks(keys6), counts


def check_every_path(cw, orc, monkeypatch, pts, voxel, pc_cellsize=0.0):
    from cwipc_util_b200 import util
    pc = upload(cw, pts, pc_cellsize)
    for v in (voxel, -voxel):
        want, cs, ranks, counts = oracle_ranks(orc, pts, v, pc_cellsize)
        for path in PATHS:
            if path is None:
                monkeypatch.delenv("CWIPC_CUDA_DS_PATH", raising=False)
            else:
                monkeypatch.setenv("CWIPC_CUDA_DS_PATH", path)
            try:
                assert_exact_means(cw.cwipc_downsample(pc, v).get_numpy_array(), pts, ranks, counts, cs, want)
            except AssertionError as e:
                raise AssertionError(f"cwipc_downsample voxelsize {v}, path {path or 'default'}: {e}") from None
        monkeypatch.delenv("CWIPC_CUDA_DS_PATH", raising=False)
        comm = util.cuda_comm(None, 1, 0)
        try:
            assert_exact_means(comm.downsample(pc, v).get_numpy_array(), pts, ranks, counts, cs, want)
        except AssertionError as e:
            raise AssertionError(f"slab downsample voxelsize {v}: {e}") from None
        finally:
            comm.free()
        got = cw.cwipc_downsample_pertile(pc, v).get_numpy_array()
        pos = 0
        for t in first_appearance(pts):
            grp = pts if t == 0 else pts[pts["tile"] == t]
            gwant, gcs, granks, gcounts = oracle_ranks(orc, grp, v, pc_cellsize)
            try:
                assert_exact_means(got[pos:pos + len(gwant)], grp, granks, gcounts, gcs, gwant)
            except AssertionError as e:
                raise AssertionError(f"cwipc_downsample_pertile voxelsize {v}, tile {t}: {e}") from None
            pos += len(gwant)
        assert pos == len(got)


def voxel_blocks(lengths, voxel, seed, colour=None, shuffle=False):
    """One voxel per entry of `lengths`, that many points each, the voxels on a 3-D grid of pitch 2 * voxel and every
    point well inside its voxel.  colour: (r, g, b) per voxel (a channel None = random per point).  With voxelsize > 0
    the octree has leaf faces through its first point: four anchor points (one per tile value, so that every per-tile
    group starts with one) come first, in a voxel below all others on every axis, so that no face cuts those voxels."""
    rng = np.random.default_rng(seed)
    n = int(sum(lengths))
    vid = np.repeat(np.arange(len(lengths)), lengths)
    cell = np.stack([vid % 8, (vid // 8) % 8, vid // 64], axis=1) * 2 - 5
    pts = np.zeros(n, DT)
    for a, name in enumerate("xyz"):
        pts[name] = ((cell[:, a] + rng.uniform(0.1, 0.9, n)) * voxel).astype(np.float32)
    for k, c in enumerate("rgb"):
        pts[c] = rng.integers(0, 256, n)
        if colour is not None:
            for i, col in enumerate(colour):
                if col[k] is not None:
                    pts[c][vid == i] = col[k]
    pts["tile"] = np.array([1, 2, 4, 8], np.uint8)[vid % 4]
    if shuffle:
        pts = pts[rng.permutation(n)]
    anchors = np.zeros(4, DT)
    for name in "xyz":
        anchors[name] = ((-7 + rng.uniform(0.1, 0.9, 4)) * voxel).astype(np.float32)
    anchors["tile"] = [1, 2, 4, 8]
    return np.concatenate([anchors, pts])


RUN_LENGTHS = [1, 7, 8, 9, 255, 256, 257, 511, 512, 513, 4097]


@pytest.mark.gpu
def test_runs_around_the_lane_tile_and_queue_sizes(cw, orc, monkeypatch):
    """Sorted input: voxel runs of every length around 8 (points per lane), 256 (points per warp tile) and the 80 records of
    the queue, three times over with the tiles falling at different offsets.  r = 255 and b = 0 everywhere, so that a carry
    between the 16-bit fields of a run (sum r | sum b << 16) shows as a wrong r or a non-zero b."""
    lengths = [3] + RUN_LENGTHS + [5] + RUN_LENGTHS[::-1] + [100] + RUN_LENGTHS
    pts = voxel_blocks(lengths, 0.01, seed=1, colour=[(255, None, 0)] * len(lengths))
    check_every_path(cw, orc, monkeypatch, pts, 0.01)


@pytest.mark.gpu
def test_a_new_voxel_on_every_point(cw, orc, monkeypatch):
    """Every point starts a run: each warp tile closes 256 runs, so the queue is flushed several times per tile."""
    pts = voxel_blocks([1] * 40000, 0.004, seed=2)
    check_every_path(cw, orc, monkeypatch, pts, 0.004)


@pytest.mark.gpu
def test_contended_heavy_voxels(cw, orc, monkeypatch):
    """1.5 M points in random order over at most 64 voxels: every reduction of a warp lands on a handful of slots."""
    rng = np.random.default_rng(3)
    n = 1500000
    pts = np.zeros(n, DT)
    for a in "xyz":
        pts[a] = rng.uniform(-0.06, 0.06, n).astype(np.float32)
    for c in "rgb":
        pts[c] = rng.integers(0, 256, n)
    pts["tile"] = rng.choice(np.array([1, 2, 4, 8], np.uint8), n)
    check_every_path(cw, orc, monkeypatch, pts, 0.05)


# voxels of uniform colour whose channel sums cross 2^24, where a float32 sum / count no longer truncates to the colour
COLOUR_2_24 = [(65795, 255), (217889, 77), (671089, 200)]


@pytest.mark.gpu
def test_colour_sums_across_2_24(cw, orc, monkeypatch):
    lengths = [n for n, _ in COLOUR_2_24] * 2 + [1000, 65000]
    colour = [(c, None, 255 - c) for _, c in COLOUR_2_24] + [(None, c, c) for _, c in COLOUR_2_24] + [(255, 255, 255)] * 2
    pts = voxel_blocks(lengths, 0.05, seed=4, colour=colour, shuffle=True)
    ref = exact_voxels(pts, canonical_ranks(orc.downsample(pts, 0.05, 0.0, want_keys=True)[2]))
    assert (ref["sum_r"] >= 1 << 24).sum() >= 3 and (ref["sum_g"] >= 1 << 24).sum() >= 3
    check_every_path(cw, orc, monkeypatch, pts, 0.05)


@pytest.mark.gpu
@pytest.mark.parametrize("n", [16843009, 16843010])
def test_colour_sums_across_2_32(cw, n):
    """The whole cloud in one voxel, colour (255, 255, 255): 255 * 16843009 = 2^32 - 1, 255 * 16843010 = 2^32 + 254."""
    rng = np.random.default_rng(n)
    pts = np.zeros(n, DT)
    for a in "xyz":
        pts[a] = rng.uniform(0.1, 0.9, n).astype(np.float32)
    for c in "rgb":
        pts[c] = 255
    pts["tile"] = rng.choice(np.array([1, 2, 4, 8], np.uint8), n)
    pts["x"][0] = pts["y"][0] = pts["z"][0] = 0.05   # the octree's leaf faces pass through the first point: not through the cloud
    ranks = np.zeros(n, np.int64)
    pc = upload(cw, pts)
    for v in (1.0, -1.0):
        got = cw.cwipc_downsample(pc, v).get_numpy_array()
        assert_exact_means(got, pts, ranks, np.array([n]), 1.0)


@pytest.mark.gpu
@pytest.mark.parametrize("k", [16, 20])
def test_fixed_point_scale_limits(cw, orc, monkeypatch, k):
    """shift = 61 - bit_length(n) - frexp_exp(voxelsize): n = 2^k - 1 and 2^k points, voxel sizes that are powers of two
    and the float just below each.  Most points sit just below the upper faces of one voxel, so its offset sums come
    close to the range the scale allows."""
    for n in ((1 << k) - 1, 1 << k):
        for voxel in (0.5, 2.0 ** -7):
            for vs in (voxel, float(np.nextafter(np.float32(voxel), np.float32(0)))):
                rng = np.random.default_rng(n)
                pts = np.zeros(n, DT)
                heavy = rng.random(n) < 0.75
                for a in "xyz":
                    spread = rng.uniform(-2 * vs, 2 * vs, n)
                    near = vs * (1 - rng.uniform(0, 2.0 ** -12, n))
                    pts[a] = np.where(heavy, near, spread).astype(np.float32)
                for c in "rgb":
                    pts[c] = rng.integers(0, 256, n)
                pts["tile"] = rng.choice(np.array([1, 2, 4, 8], np.uint8), n)
                pts["x"][0] = pts["y"][0] = pts["z"][0] = -2 * vs   # leaf faces through the first point: below the heavy voxel
                check_every_path(cw, orc, monkeypatch, pts, vs)


@functools.lru_cache(maxsize=1)
def geometry_clouds():
    rng = np.random.default_rng(7)
    n = 200000

    def cloud(lo, hi):
        pts = np.zeros(n, DT)
        for a in range(3):
            pts["xyz"[a]] = rng.uniform(lo[a], hi[a], n).astype(np.float32)
        for c in "rgb":
            pts[c] = rng.integers(0, 256, n)
        pts["tile"] = rng.choice(np.array([1, 2, 4, 8], np.uint8), n)
        return pts

    far = cloud((1000.0, 0.0, 0.0), (1000.05, 0.05, 0.05))            # |x / voxel| ~ 10^6: float voxel arithmetic at 2^20
    edge = cloud((4194.0, -0.05, 0.0), (4194.3, 0.0, 0.05))           # |x / voxel| just under 2^22
    negative = cloud((-3.0, -2.0, -1.1), (-2.9, -1.9, -1.0))
    faces = cloud((-1.0, -1.0, -1.0), (1.0, 1.0, 1.0))
    q = rng.integers(-8, 8, (n, 3))                                  # exactly on faces of the 0.25 grid for half the points
    on = rng.random(n) < 0.5
    for a in range(3):
        faces["xyz"[a]][on] = (q[on, a] * 0.25).astype(np.float32)
    faces["x"][:20000:2] = (q[:20000:2, 0] * np.float32(0.01)).astype(np.float32)   # faces of a grid that is not a power of two
    tiny = synthetic.simulate_cameras(synthetic.synthetic_cloud(250000), 4)
    tiny["x"][1000:1010] = [1e-20, -1e-20, 1e-30, -1e-38, 1e-44, -1e-45, 3e-17, -3e-17, 1e-12, -1e-12]
    tiny["y"][2000:2004] = [1e-20, 1e-41, -1e-20, 2e-17]
    return [("far_from_origin", far, 0.001), ("just_under_2_22_voxels", edge, 0.001), ("negative", negative, 0.01),
            ("on_faces_025", faces, 0.25), ("on_faces_001", faces, 0.01), ("denormal_first_point_planes", tiny, 0.005)]


@pytest.mark.gpu
@pytest.mark.parametrize("case", range(6), ids=["far_from_origin", "just_under_2_22_voxels", "negative", "on_faces_025", "on_faces_001",
                                                "denormal_first_point_planes"])
def test_geometry(cw, orc, monkeypatch, case):
    name, pts, voxel = geometry_clouds()[case]
    check_every_path(cw, orc, monkeypatch, pts, voxel)


def test_reference_matches_a_plain_loop(orc):
    """The reference of this file against a point-by-point loop and the oracle, and the check against subtly wrong
    results: a colour rounded instead of truncated, one point dropped from a voxel, a tile bit lost."""
    pts = voxel_blocks([1, 7, 300, 2, 40], 0.1, seed=5)
    want, cs, ranks, counts = oracle_ranks(orc, pts, 0.1, 0.0)
    ref = exact_voxels(pts, ranks)
    assert np.array_equal(ref["count"], counts)
    for v in range(len(counts)):
        grp = pts[ranks == v]
        assert ref["count"][v] == len(grp)
        for a in "xyz":
            assert ref[a][v] == sum(float(x) for x in grp[a]) / len(grp)
        for c in "rgb":
            s = sum(int(x) for x in grp[c])
            assert ref["sum_" + c][v] == s and ref[c][v] == s // len(grp) == want[c][v]
        t = 0
        for x in grp["tile"]:
            t |= int(x)
        assert ref["tile"][v] == t == want["tile"][v]
    exact = np.zeros(len(counts), DT)
    for k in ("x", "y", "z", "r", "g", "b", "tile"):
        exact[k] = ref[k]
    assert_exact_means(exact, pts, ranks, counts, cs, want)
    rounded = exact.copy()
    rounded["r"] = np.minimum(np.rint(ref["sum_r"] / ref["count"]), 255)
    assert np.any(rounded["r"] != exact["r"])
    heavy = int(np.argmax(counts))
    assert counts[heavy] == 300
    dropped = exact.copy()
    dropped["x"][heavy] = np.float32(pts["x"][ranks == heavy][1:].astype(np.float64).mean())
    spilled = exact.copy()
    spilled["tile"][heavy] &= spilled["tile"][heavy] - 1
    for bad in (rounded, dropped, spilled):
        with pytest.raises(AssertionError):
            assert_exact_means(bad, pts, ranks, counts, cs, want)
