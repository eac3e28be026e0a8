"""The compaction kernel, the per-point maps, the join, the tile bookkeeping of the per-tile filters and the cellsize
heuristic against the plain numpy reference of tests/pointops_reference.py, byte for byte.

Every result passes through one of these last: tilefilter, masked tilefilter, crop, the distance filters and the
outlier removal all compact with compact_kernel (csrc/pointops.cu), whose look-back words live in the thread's zeroed
workspace up to 8158 tiles of 2048 points and in memset scratch above that.  The cases aim at where such kernels go
wrong: sizes on both sides of a tile and of the workspace limit, keep patterns at tile boundaries, back-to-back launches
that switch between the two look-back homes, float edges of the crop predicate, every tile value and every colour bit,
all 255 tile groups of a per-tile filter, subsets that inherit a loose bounding box, and the min-reduction of the
cellsize heuristic at its float edges.  Records are compared as bytes, so NaN payloads and the sign of zero count.
"""
import gc
import os
import sys
import threading

import numpy as np
import pytest

from cwipc_util_b200 import synthetic
from parity_helpers import assert_exact_means, canonical_ranks

import pointops_reference as ref

pytestmark = pytest.mark.gpu

DT = synthetic.cwipc_point_numpy_dtype
TESTS = os.path.dirname(os.path.abspath(__file__))
REPO = os.path.dirname(TESTS)

TILE = 2048                      # points per block of compact_kernel
WORKSPACE_TILES = 8158           # look-back words that fit the thread's zeroed workspace: (65536 - 256 - 16) / 8
EDGE = WORKSPACE_TILES * TILE    # 16 707 584: the largest cloud compacted without memset scratch
BIG = 20_000_003
SIZES = [1, 2047, 2048, 2049, EDGE - 1, EDGE, EDGE + 1, BIG]
PATTERNS = ["none", "all", "every_other", "first", "last", "one_per_tile", "runs", "random_1pc"]
UNIT_BOX = (0.0, 1.0, 0.0, 1.0, 0.0, 1.0)
F32 = np.float32
FLT_MIN = np.finfo(np.float32).tiny


@pytest.fixture(autouse=True)
def no_leaks(cw):
    gc.collect()
    base = cw.cwipc_dangling_allocations(False)
    yield
    gc.collect()
    assert cw.cwipc_dangling_allocations(False) == base


def upload(cw, pts, timestamp=1, cellsize=None):
    pc = cw.cwipc_from_numpy_array(pts, timestamp)
    if cellsize is not None:
        pc._set_cellsize(cellsize)
    return pc


def take(pc):
    """The cloud's records (host copy); the cloud is freed."""
    got = pc.get_numpy_array()
    pc.free()
    return got


def assert_same(got, want, what):
    assert ref.same_bytes(got, want), f"{what}: {len(got)} records, the reference has {len(want)}, first difference at {ref.first_difference(got, want)}"


def keep_pattern(name, n, seed=0):
    i = np.arange(n)
    if name == "none":
        return np.zeros(n, bool)
    if name == "all":
        return np.ones(n, bool)
    if name == "every_other":
        return i % 2 == 0
    if name == "first":
        return i == 0
    if name == "last":
        return i == n - 1
    if name == "one_per_tile":     # one point per 2048-point block, at a different lane and warp in each
        keep = np.zeros(n, bool)
        t = np.arange((n + TILE - 1) // TILE)
        idx = t * TILE + (t * 37) % TILE
        keep[idx[idx < n]] = True
        return keep
    if name == "runs":             # runs of 1500 kept / 1500 dropped, offset so that they straddle block boundaries
        return ((i + 700) // 1500) % 2 == 0
    return np.random.default_rng(seed).random(n) < 0.01


@pytest.fixture(scope="module")
def base20m():
    """BIG points, x, y, z uniform in [0, 1): every point lies in UNIT_BOX until a pattern moves it out."""
    rng = np.random.default_rng(2024)
    pts = np.zeros(BIG, DT)
    for a in "xyz":
        pts[a] = rng.random(BIG, dtype=np.float32)
    for c in "rgb":
        pts[c] = rng.integers(0, 256, BIG, dtype=np.uint8)
    return pts


@pytest.fixture(scope="module")
def bits20m(base20m):
    """The BIG cloud with keep pattern p in tile bit p: cwipc_cuda_tilefilter_masked(pc, 1 << p) selects pattern p."""
    pts = base20m.copy()
    pts["tile"] = 0
    for p, name in enumerate(PATTERNS):
        pts["tile"] |= keep_pattern(name, BIG, seed=p).astype(np.uint8) << p
    return pts


@pytest.fixture(scope="module")
def bits20m_pc(cw, bits20m):
    pc = upload(cw, bits20m, timestamp=20)
    yield pc
    pc.free()


def pattern_cloud(work, base, n, keep, axis):
    """base[:n], written to work[:n], with tile 5 where kept and 2 where not (5 & 4 != 0, 2 & 4 == 0) and the dropped
    points moved out of UNIT_BOX by +2 along `axis`."""
    pts = work[:n]
    np.copyto(pts.view(np.uint32), base[:n].view(np.uint32))   # as words: a record-wise copy is several times slower
    pts["tile"] = np.where(keep, np.uint8(5), np.uint8(2))
    col = pts[axis]
    np.add(col, F32(2.0), out=col, where=~keep)
    return pts


# ---- compaction: sizes, keep patterns, both homes of the look-back words ------------------------------------------------
@pytest.mark.parametrize("n", SIZES)
def test_compaction_sizes_and_patterns(cw, base20m, n):
    """Tilefilter, masked tilefilter and crop of every keep pattern at sizes around one block and around the workspace
    limit: above EDGE points the look-back words live in memset scratch, not in the thread's workspace."""
    work = np.empty(n, DT)
    for p, name in enumerate(PATTERNS):
        keep = keep_pattern(name, n, seed=p)
        pts = pattern_cloud(work, base20m, n, keep, "xyz"[p % 3])
        masks = {"tilefilter 5": ref.tile_equals_mask(pts, 5), "masked 4": ref.tile_mask_mask(pts, 4), "crop": ref.crop_mask(pts, UNIT_BOX)}
        for what, m in masks.items():
            assert np.array_equal(m, keep), f"reference {what} does not select pattern {name}"
        want = ref.compact(pts, keep)
        pc = upload(cw, pts)
        assert_same(take(cw.cwipc_tilefilter(pc, 5)), want, f"n={n} {name} tilefilter")
        assert_same(take(cw.cwipc_tilefilter_masked(pc, 4)), want, f"n={n} {name} masked tilefilter")
        assert_same(take(cw.cwipc_crop(pc, UNIT_BOX)), want, f"n={n} {name} crop")
        pc.free()
        del pts, want, masks


@pytest.mark.parametrize("n", [EDGE + 1, BIG])
def test_filter_by_distance_past_the_workspace(cw, bits20m, bits20m_pc, n):
    """cwipc_cuda_filter_by_distance on the scratch path: a threshold that keeps a random 1 %, NaN distances (kept:
    NaN > threshold is false), and the thresholds that keep everything and nothing."""
    pts = bits20m[:n]
    pc = bits20m_pc if n == BIG else upload(cw, pts)
    rng = np.random.default_rng(n)
    dist = rng.random(n, dtype=np.float32)
    dist[rng.choice(n, 1000, replace=False)] = np.nan
    for thr in (0.01, 1.0, -1.0):
        want = ref.compact(pts, ref.distance_mask(dist, thr))
        assert_same(take(cw.util.filter_by_distance(pc, dist, thr)), want, f"n={n} threshold {thr}")
    if pc is not bits20m_pc:
        pc.free()


def compaction_sequence(cw, bits20m, big_pc):
    """Back to back on the calling thread: scratch path, workspace path, one point, scratch again, workspace again with
    another pattern and tile count, a per-tile outlier removal (a chain of compactions) before and after."""
    mid_n = 5_000_000
    mid = upload(cw, bits20m[:mid_n])
    one = upload(cw, bits20m[BIG - 1:])
    small_pts = synthetic.camera_cloud(60000, seed=5)
    small = upload(cw, small_pts, cellsize=synthetic.cellsize_of(60000))
    chain_before = take(cw.cwipc_remove_outliers(small, 8, 1.0, True))
    steps = [(big_pc, bits20m, "random_1pc"), (mid, bits20m[:mid_n], "every_other"), (one, bits20m[BIG - 1:], "all"), (big_pc, bits20m, "runs"),
             (mid, bits20m[:mid_n], "one_per_tile"), (mid, bits20m[:mid_n], "random_1pc"), (one, bits20m[BIG - 1:], "last"), (big_pc, bits20m, "every_other")]
    try:
        for pc, pts, name in steps:
            bit = PATTERNS.index(name)
            want = ref.compact(pts, ref.tile_mask_mask(pts, 1 << bit))
            assert_same(take(cw.cwipc_tilefilter_masked(pc, 1 << bit)), want, f"{len(pts)} points, pattern {name}")
        assert_same(take(cw.cwipc_remove_outliers(small, 8, 1.0, True)), chain_before, "per-tile outlier removal after the sequence")
    finally:
        for pc in (mid, one, small):
            pc.free()


def test_workspace_hygiene_back_to_back(cw, bits20m, bits20m_pc):
    """The last block of a workspace launch clears the look-back words, the ticket and the done counter for the next
    launch: compactions of different tile counts alternate between the workspace and scratch, on this thread and then on
    a second one (a workspace of its own)."""
    compaction_sequence(cw, bits20m, bits20m_pc)
    errors = []

    def second():
        try:
            compaction_sequence(cw, bits20m, bits20m_pc)
        except BaseException as e:     # reported on the test's thread
            errors.append(e)

    t = threading.Thread(target=second)
    t.start()
    t.join()
    if errors:
        raise errors[0]


# ---- crop at its float edges ------------------------------------------------------------------------------------------
SPECIALS = [0.0, -0.0, 1e-45, -1e-45, FLT_MIN, -FLT_MIN, np.inf, -np.inf, np.nan]

CROP_BOXES = {
    "finite": (-1.5, 2.25, 0.125, 3.0, -7.0, -0.5),
    "signed_zero_faces": (-0.0, 1.0, 0.0, 1.0, -1.0, -0.0),
    "infinite_faces": (-np.inf, np.inf, -np.inf, 0.0, 0.0, np.inf),
    "denormal_faces": (1e-45, FLT_MIN, -FLT_MIN, -1e-45, -1e-45, 1e-45),
    "zero_width": (1.0, 1.0, -1.0, 1.0, -1.0, 1.0),
    "nan_low_face": (np.nan, 1.0, -1.0, 1.0, -1.0, 1.0),
    "nan_high_face": (-1.0, 1.0, -1.0, 1.0, -1.0, np.nan),
    "inverted": (2.0, 1.0, -1.0, 1.0, -1.0, 1.0),
}
EMPTY_BOXES = {"zero_width", "nan_low_face", "nan_high_face", "inverted"}


def axis_values(lo, hi):
    """The faces, the floats on either side of each, and the special values; distinct as bit patterns."""
    v = [lo, hi] + SPECIALS
    for f in (F32(lo), F32(hi)):
        v += [np.nextafter(f, F32(-np.inf)), np.nextafter(f, F32(np.inf))]
    a = np.array(v, np.float32)
    _, idx = np.unique(a.view(np.uint32), return_index=True)
    return a[np.sort(idx)]


def crop_grid(box, seed):
    xs, ys, zs = (axis_values(box[2 * k], box[2 * k + 1]) for k in range(3))
    X, Y, Z = np.meshgrid(xs, ys, zs, indexing="ij")
    g = np.zeros(X.size, DT)
    g["x"], g["y"], g["z"] = X.ravel(), Y.ravel(), Z.ravel()
    rng = np.random.default_rng(seed)
    pts = np.concatenate([g[rng.permutation(len(g))] for _ in range(3)])   # three orders: every value in many lanes
    for c in ("r", "g", "b", "tile"):
        pts[c] = rng.integers(0, 256, len(pts), dtype=np.uint8)
    return pts


@pytest.mark.parametrize("box", list(CROP_BOXES))
def test_crop_edges(cw, box):
    """x0 <= x < x1 on each axis, in float32 with no flush to zero: points on a face, one float either side of it,
    -0.0 against a +0.0 face, denormals, NaN and infinities against finite, infinite, signed-zero and denormal faces.
    A NaN face or an inverted or zero-width box keeps nothing."""
    b = CROP_BOXES[box]
    pts = crop_grid(b, seed=len(box))
    want = ref.compact(pts, ref.crop_mask(pts, b))
    if box in EMPTY_BOXES:
        assert len(want) == 0
    else:
        assert 0 < len(want) < len(pts)
    pc = upload(cw, pts)
    assert_same(take(cw.cwipc_crop(pc, b)), want, f"crop {box}")
    pc.free()


# ---- every tile value -------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def all_tiles():
    """Every tile value 0..255: 32 distinct values in every warp, then one run of 600 per value (shuffled runs), then
    random values.  Coordinates include NaN, -0.0 and denormals, which must come through as bytes."""
    rng = np.random.default_rng(77)
    inter = (np.arange(256 * 64) * 37) % 256
    runs = np.repeat(rng.permutation(256), 600)
    rand = rng.integers(0, 256, 40000)
    tiles = np.concatenate([inter, runs, rand]).astype(np.uint8)
    pts = np.zeros(len(tiles), DT)
    for a in "xyz":
        pts[a] = rng.standard_normal(len(pts)).astype(np.float32)
    specials = np.array([np.nan, -0.0, 1e-45, -np.inf], np.float32)
    where = rng.choice(len(pts), 4000, replace=False)
    pts["x"][where] = specials[np.arange(4000) % 4]
    for c in "rgb":
        pts[c] = rng.integers(0, 256, len(pts), dtype=np.uint8)
    pts["tile"] = tiles
    return pts


def test_tilefilter_every_tile_value(cw, orc, all_tiles):
    """tile = -1 .. 256 and 300: an int compared with an 8-bit tile, so -1, 256 and 300 keep nothing and 0 keeps all."""
    pc = upload(cw, all_tiles)
    for t in list(range(-1, 257)) + [300]:
        want = ref.compact(all_tiles, ref.tile_equals_mask(all_tiles, t))
        assert ref.same_bytes(want, orc.tilefilter(all_tiles, t))
        assert_same(take(cw.cwipc_tilefilter(pc, t)), want, f"tilefilter {t}")
    pc.free()


def test_masked_tilefilter_every_mask(cw, all_tiles):
    """(tile & (mask & 0xff)) != 0 for every 8-bit mask, and masks with bits above 0xff."""
    pc = upload(cw, all_tiles)
    for mask in list(range(256)) + [0x100, 0x1FF, -1, 0x7FFFFF01]:
        want = ref.compact(all_tiles, ref.tile_mask_mask(all_tiles, mask))
        assert_same(take(cw.cwipc_tilefilter_masked(pc, mask)), want, f"mask {mask:#x}")
    pc.free()


def test_tilemap_tables(cw, all_tiles):
    rng = np.random.default_rng(3)
    tables = {"identity": np.arange(256), "zero": np.zeros(256, int), "reverse": np.arange(256)[::-1]}
    for k in range(3):
        tables[f"random{k}"] = rng.permutation(256)
    pc = upload(cw, all_tiles)
    for name, table in tables.items():
        got = take(cw.cwipc_tilemap(pc, [int(v) for v in table]))
        assert_same(got, ref.tilemap(all_tiles, table), f"tilemap {name}")
    pc.free()


# ---- colour map: every bit ---------------------------------------------------------------------------------------------
def colour_cloud():
    """r, g, b and tile each take every byte value, in different combinations."""
    n = 65536
    i = np.arange(n)
    rng = np.random.default_rng(9)
    pts = np.zeros(n, DT)
    for a in "xyz":
        pts[a] = rng.standard_normal(n).astype(np.float32)
    pts["r"] = i & 0xFF
    pts["g"] = i >> 8
    pts["b"] = rng.permutation(256)[(i * 7 + (i >> 8)) & 0xFF]
    pts["tile"] = rng.permutation(256)[(i * 13 + 5 * (i >> 8)) & 0xFF]
    return pts


def test_colormap_every_bit(cw):
    pts = colour_cloud()
    for c in ("r", "g", "b", "tile"):
        assert len(np.unique(pts[c])) == 256
    rng = np.random.default_rng(10)
    pairs = [(1 << b, 0) for b in range(32)] + [(0, 1 << b) for b in range(32)]
    pairs += [(0xFFFFFFFF, 0), (0, 0xFFFFFFFF), (0, 0), (0xFFFFFFFF, 0xFFFFFFFF)]
    pairs += [(int(a), int(b)) for a, b in rng.integers(0, 1 << 32, (32, 2), dtype=np.uint64)]
    pc = upload(cw, pts)
    for clear, set_ in pairs:
        assert_same(take(cw.cwipc_colormap(pc, clear, set_)), ref.colormap(pts, clear, set_), f"colormap clear {clear:#010x} set {set_:#010x}")
    pc.free()


# ---- join --------------------------------------------------------------------------------------------------------------
def test_join_empty_sides_timestamp_and_cellsize(cw):
    rng = np.random.default_rng(12)
    pts = np.zeros(3001, DT)
    for a in "xyz":
        pts[a] = rng.standard_normal(len(pts)).astype(np.float32)
    pts["tile"] = rng.integers(0, 256, len(pts), dtype=np.uint8)
    empty_a, empty_b = cw.cwipc_from_points([], 50), cw.cwipc_from_points([], 40)
    full = upload(cw, pts, timestamp=45, cellsize=0.25)
    empty_a._set_cellsize(0.5)
    empty_b._set_cellsize(0.0)
    cases = [(empty_a, empty_b, pts[:0], 40, 0.0), (empty_a, full, pts, 45, 0.25), (full, empty_b, pts, 40, 0.0), (full, empty_a, pts, 45, 0.25),
             (full, full, ref.join(pts, pts), 45, 0.25)]
    for a, b, want, ts, cs in cases:
        out = cw.cwipc_join(a, b)
        assert (out.count(), out.timestamp(), out.cellsize()) == (len(want), ts, np.float32(cs))
        assert_same(take(out), want, "join")
    lib = cw.util.cwipc_util_dll_load()
    assert not lib.cwipc_join(full.as_cwipc_p(), None)
    for pc in (empty_a, empty_b, full):
        pc.free()


def test_join_past_the_workspace_then_compact(cw, bits20m, bits20m_pc):
    """A join of BIG + 1 M points, then compactions of the joined cloud (scratch path)."""
    other = bits20m[:1_000_000].copy()
    other["tile"] = np.random.default_rng(13).integers(0, 256, len(other), dtype=np.uint8)
    opc = upload(cw, other, timestamp=3)
    joined = cw.cwipc_join(bits20m_pc, opc)
    whole = ref.join(bits20m, other)
    assert joined.count() == len(whole) > EDGE and joined.timestamp() == 3
    for mask in (1 << PATTERNS.index("random_1pc"), 1 << PATTERNS.index("runs")):
        assert_same(take(cw.cwipc_tilefilter_masked(joined, mask)), ref.compact(whole, ref.tile_mask_mask(whole, mask)), f"masked {mask:#x}")
    box = (0.25, 0.5, 0.0, 1.0, 0.0, 1.0)
    assert_same(take(cw.cwipc_crop(joined, box)), ref.compact(whole, ref.crop_mask(whole, box)), "crop")
    assert_same(take(joined), whole, "join")
    opc.free()


# ---- tile bookkeeping of the per-tile filters at 255 / 256 values --------------------------------------------------------
TILE_CASES = ["255", "255+0", "2+0", "64+0", "128+0"]


def tile_case_cloud(case):
    """Non-zero values 1..255 (or the first 2, 64, 128 of a shuffle of them) at 120 points each, random order (many
    distinct values per warp); '+0' adds tile-0 points interleaved, one in nine."""
    rng = np.random.default_rng(len(case) * 1000 + int(case.split("+")[0]))
    nvals = int(case.split("+")[0])
    values = np.arange(1, 256) if nvals == 255 else rng.permutation(np.arange(1, 256))[:nvals]
    per = max(120, 30000 // nvals)
    tiles = np.repeat(values, per)
    if case.endswith("+0"):
        tiles = np.concatenate([tiles, np.zeros(len(tiles) // 8, int)])
    tiles = rng.permutation(tiles).astype(np.uint8)
    pts = np.zeros(len(tiles), DT)
    for a in "xyz":
        pts[a] = rng.uniform(0.1, 0.9, len(pts)).astype(np.float32)
    for c in "rgb":
        pts[c] = rng.integers(0, 256, len(pts), dtype=np.uint8)
    pts["tile"] = tiles
    return pts


def first_appearance(pts):
    _, first = np.unique(pts["tile"], return_index=True)
    return [int(t) for t in pts["tile"][np.sort(first)]]


def groups(pts):
    return [(t, pts if t == 0 else pts[pts["tile"] == t]) for t in first_appearance(pts)]


@pytest.mark.parametrize("case", TILE_CASES)
def test_pertile_downsample_at_the_group_count_edges(cw, orc, case):
    """All 255 non-zero values (the split's 'none' rank is 255) with and without tile 0, and 2, 64, 128 values plus
    tile 0 (none a power of two: the split's bit count at its edge, the tile-0 points taking the none rank).  The result
    must equal the library's own composition and the exact per-group means; with a voxel that holds every point, one
    record per group whose count is the group's size (the counts of first_tile_kernel)."""
    pts = tile_case_cloud(case)
    grps = groups(pts)
    nvals = int(case.split("+")[0])
    assert len(grps) == nvals + case.endswith("+0")
    pc = upload(cw, pts)
    for voxel in (0.05, -0.05):
        got = take(cw.cwipc_downsample_pertile(pc, voxel))
        parts = [cw.cwipc_downsample(cw.cwipc_tilefilter(pc, t), voxel) for t, _ in grps]
        assert_same(got, take(cw.cwipc_join_multi(parts)), f"{case} voxel {voxel}: composition")
        pos = 0
        for t, grp in grps:
            want, cs, keys6, counts = orc.downsample(grp, voxel, 0.0, want_keys=True)
            try:
                assert_exact_means(got[pos:pos + len(want)], grp, canonical_ranks(keys6), counts, cs, want)
            except AssertionError as e:
                raise AssertionError(f"{case} voxel {voxel} tile {t}: {e}") from None
            pos += len(want)
        assert pos == len(got)
    got = take(cw.cwipc_downsample_pertile(pc, -8.0))
    assert len(got) == len(grps)
    for j, (t, grp) in enumerate(grps):
        assert_exact_means(got[j:j + 1], grp, np.zeros(len(grp), np.int64), np.array([len(grp)]), 8.0)
    pc.free()


def dump_pertile_outliers(path):
    """Child process of test_pertile_outliers_at_the_group_count_edges: per-tile outlier removal of every TILE_CASES cloud."""
    import cwipc_util_b200 as cw
    out = {}
    for case in TILE_CASES:
        pc = cw.cwipc_from_numpy_array(tile_case_cloud(case), 1)
        out[case] = cw.cwipc_remove_outliers(pc, 4, 1.0, True).get_numpy_array().copy()
        pc.free()
    np.savez(path, **out)


def test_pertile_outliers_at_the_group_count_edges(cw, tmp_path):
    """Per-tile outlier removal (k = 4) of the same clouds: byte-identical to the group-after-group path, which
    CWIPC_CUDA_SOR_PER_TILE=sequential forces in a child process (the setting is read once per process)."""
    import subprocess
    path = str(tmp_path / "sor.npz")
    code = f"import sys; sys.path[:0] = [{REPO!r}, {TESTS!r}]; import test_gpu_pointops_exact as t; t.dump_pertile_outliers({path!r})"
    subprocess.run([sys.executable, "-c", code], env=dict(os.environ, CWIPC_CUDA_SOR_PER_TILE="sequential"), check=True, timeout=600)
    want = np.load(path)
    for case in TILE_CASES:
        pc = upload(cw, tile_case_cloud(case))
        got = take(cw.cwipc_remove_outliers(pc, 4, 1.0, True))
        pc.free()
        assert len(got) > 0
        assert_same(got, want[case], f"{case}: one pass vs group after group")


# ---- subsets that inherit a loose bounding box ------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def boxed_subsets(cw):
    """A downsampled 1 M-point camera cloud (its result carries a bounding box) and three compactions of it, which inherit
    that box: one tile, a corner of about 1 % of the frame, and a thin slab."""
    raw = upload(cw, synthetic.camera_cloud(1_000_000, seed=31), cellsize=synthetic.cellsize_of(1_000_000))
    ds = cw.cwipc_downsample(raw, 0.006)
    raw.free()
    p = ds.get_numpy_array()
    lo = [float(p[a].min()) for a in "xyz"]
    hi = [float(p[a].max()) for a in "xyz"]
    w = [h - l for l, h in zip(lo, hi)]
    corner = (lo[0], lo[0] + 0.5 * w[0], lo[1], lo[1] + 0.1 * w[1], lo[2], lo[2] + 0.5 * w[2])
    slab = (lo[0], hi[0] + 1, 1.0, 1.02, lo[2], hi[2] + 1)
    subsets = {"tile1": cw.cwipc_tilefilter(ds, 1), "corner": cw.cwipc_crop(ds, corner), "slab": cw.cwipc_crop(ds, slab)}
    assert 100 < subsets["corner"].count() < 0.05 * ds.count()
    assert 100 < subsets["slab"].count() < 0.05 * ds.count()
    ds.free()
    yield subsets
    for pc in subsets.values():
        pc.free()


@pytest.mark.parametrize("name", ["tile1", "corner", "slab"])
def test_knn_on_subsets_with_an_inherited_box(cw, orc, boxed_subsets, name):
    """The kNN grid of a subset is planned from the box it inherited, sized for the whole frame.  The mean distances must
    not depend on it: bit-identical to the same points uploaded fresh (no box) and to the oracle; the outlier removal,
    whole cloud and per tile, byte-identical to the fresh upload."""
    sub = boxed_subsets[name]
    pts = sub.get_numpy_array().copy()
    fresh = upload(cw, pts, cellsize=sub.cellsize())
    for k in (8, 30, 100):
        got = cw.util.knn_mean_distances(sub, k)
        assert np.array_equal(got, cw.util.knn_mean_distances(fresh, k)), (name, k)
        assert np.array_equal(got, orc.knn_mean_distances(pts, k)), (name, k)
        for per_tile in (False, True):
            assert_same(take(cw.cwipc_remove_outliers(sub, k, 1.0, per_tile)), take(cw.cwipc_remove_outliers(fresh, k, 1.0, per_tile)), f"{name} k={k} per_tile={per_tile}")
    fresh.free()


# ---- the cellsize heuristic ----------------------------------------------------------------------------------------------
def cellsize_clouds(bits20m):
    rng = np.random.default_rng(41)

    def cloud(n, lo=1.0, hi=2.0):
        pts = np.zeros(n, DT)
        for a in "xyz":
            pts[a] = rng.uniform(lo, hi, n).astype(np.float32)
        return pts

    out = {"n1": cloud(1), "n2": cloud(2)}
    c = cloud(100000)
    c[7777] = c[0]
    c["tile"][7777] ^= 1                                   # a later duplicate of p0's position: 0.0
    out["duplicate_of_p0"] = c
    c = cloud(50000, -3e38, 3e38)
    c["x"][0], c["x"][1:] = 3e38, -3e38                    # every dx overflows: d2 = inf, no finite distance
    out["all_overflow"] = c
    c = out["all_overflow"].copy()
    c["y"][0], c["z"][0] = 0.0, 0.0
    c[31000] = c[0]
    c["y"][31000] = np.float32(1e19)                       # one finite d2 (1e38) among the overflows
    out["one_finite_among_overflows"] = c
    c = np.zeros(20000, DT)
    c["x"][1:] = (rng.uniform(1.0, 2.0, 19999) * 1e-25).astype(np.float32)   # d2 underflows to 0
    c["x"][0] = 0.0
    out["underflow_to_zero"] = c
    c = np.zeros(20000, DT)
    c["x"][1:] = (rng.uniform(3.0, 9.0, 19999) * 1e-22).astype(np.float32)   # d2 denormal
    out["denormal_d2"] = c
    c = cloud(100000)
    c["x"][rng.choice(np.arange(1, 100000), 10000, replace=False)] = np.nan
    c["x"][99999] = np.nan
    out["nan_in_later_points"] = c
    c = cloud(1000)
    c["z"][0] = np.nan
    out["nan_in_p0"] = c
    n = 1_000_000
    for where, i in (("last_point", n - 1), ("last_block", 1 + 1183 * 256 + 255), ("last_block_mid_warp", 1 + 1183 * 256 + 17)):
        c = cloud(n)
        c["x"][0], c["y"][0], c["z"][0] = 0.0, 0.0, 0.0
        c["x"][i], c["y"][i], c["z"][i] = 0.01, 0.02, 0.03      # the unique minimum
        out[f"unique_min_at_{where}"] = c
    out["20M"] = bits20m
    return out


CELLSIZE_CASES = ["n1", "n2", "duplicate_of_p0", "all_overflow", "one_finite_among_overflows", "underflow_to_zero", "denormal_d2", "nan_in_later_points", "nan_in_p0",
                  "unique_min_at_last_point", "unique_min_at_last_block", "unique_min_at_last_block_mid_warp", "20M"]


def test_cellsize_heuristic(cw, orc, bits20m, bits20m_pc):
    """_set_cellsize(-1): min over i >= 1 of |p_i - p_0|, taken on the device as the min of d2 bit patterns and one
    sqrtf, must equal the oracle's min of sqrtf(d2) bit for bit at the float edges where the two could part."""
    clouds = cellsize_clouds(bits20m)
    assert list(clouds) == CELLSIZE_CASES
    for name, pts in clouds.items():
        want = np.float32(orc.min_distance_to_first(pts))
        pc = bits20m_pc.clone() if name == "20M" else upload(cw, pts)
        pc._set_cellsize(-1)
        got = np.float32(pc.cellsize())
        assert got.view(np.uint32) == want.view(np.uint32), (name, got, want)
        pc.free()
    assert np.float32(orc.min_distance_to_first(clouds["duplicate_of_p0"])) == 0.0
    assert np.float32(orc.min_distance_to_first(clouds["denormal_d2"])) > 0.0
    assert np.float32(orc.min_distance_to_first(clouds["one_finite_among_overflows"])) == np.float32(1e19)
    assert 0.0 < np.float32(orc.min_distance_to_first(clouds["unique_min_at_last_block"])) < 0.1


# ---- cwipc_cuda_from_device_points ----------------------------------------------------------------------------------------
def test_from_device_points(cw, lib, all_tiles):
    src = upload(cw, all_tiles, timestamp=5)
    ptr = cw.util.pointcloud_device_ptr(src)
    assert ptr
    copy = cw.util.from_device_points(ptr, src.count(), 1234)
    assert (copy.count(), copy.timestamp(), copy.cellsize()) == (len(all_tiles), 1234, 0.0)
    assert_same(take(copy), all_tiles, "whole copy")
    part = cw.util.from_device_points(ptr + 16 * 1001, 2049, 7)     # a slice starting inside the source
    assert_same(take(part), all_tiles[1001:1001 + 2049], "slice")
    empty = lib.cwipc_cuda_from_device_points(ptr, 0, 9)
    assert empty
    empty = cw.util.cwipc_pointcloud_wrapper(empty)
    assert (empty.count(), empty.timestamp()) == (0, 9)
    empty.free()
    empty = cw.util.cwipc_pointcloud_wrapper(lib.cwipc_cuda_from_device_points(None, 0, 9))
    assert empty.count() == 0
    empty.free()
    assert not lib.cwipc_cuda_from_device_points(None, 5, 0)
    assert not lib.cwipc_cuda_from_device_points(ptr, -1, 0)
    assert not lib.cwipc_cuda_from_device_points(None, -1, 0)
    src.free()
