"""The per-point filter reference of tests/pointops_reference.py checked on its own, without a GPU: hand-worked answers
for every predicate at its edges, the colour map's byte shuffle, and the tile predicate against the CPU oracle."""
import numpy as np
import pytest

from cwipc_util_b200 import synthetic

import pointops_reference as ref

DT = synthetic.cwipc_point_numpy_dtype
F32 = np.float32
INF, NAN = F32(np.inf), F32(np.nan)
TINY, FMIN = F32(1e-45), np.finfo(np.float32).tiny


def points(rows):
    pts = np.zeros(len(rows), DT)
    for i, row in enumerate(rows):
        for name, v in zip(("x", "y", "z", "r", "g", "b", "tile"), row):
            pts[name][i] = v
    return pts


def test_point_dtype_is_the_library_layout():
    assert ref.POINT_DTYPE == DT and ref.POINT_DTYPE.itemsize == 16


def test_crop_is_half_open_per_axis():
    box = (0.0, 1.0, 0.0, 1.0, 0.0, 1.0)
    x = [0.0, np.nextafter(F32(0), F32(-1)), np.nextafter(F32(1), F32(0)), 1.0, -0.0, TINY, -TINY, INF, -INF, NAN, 0.5]
    pts = points([(v, 0.5, 0.5) for v in x])
    assert ref.crop_mask(pts, box).tolist() == [True, False, True, False, True, True, False, False, False, False, True]
    # the same values on y and z
    for a in "yz":
        q = points([(0.5, 0.5, 0.5)] * len(x))
        q[a] = np.array(x, F32)
        assert ref.crop_mask(q, box).tolist() == [True, False, True, False, True, True, False, False, False, False, True]


def test_crop_box_faces_at_their_edges():
    pts = points([(v, 0, 0) for v in (-INF, -1e30, -0.0, 0.0, TINY, FMIN, 1e30, INF, NAN)])
    everything_finite = [False, True, True, True, True, True, True, False, False]
    assert ref.crop_mask(pts, (-np.inf, np.inf, -1, 1, -1, 1)).tolist() == [True] + everything_finite[1:]
    assert ref.crop_mask(pts, (-0.0, np.inf, -1, 1, -1, 1)).tolist() == [False, False, True, True, True, True, True, False, False]
    assert ref.crop_mask(pts, (-np.inf, -0.0, -1, 1, -1, 1)).tolist() == [True, True, False, False, False, False, False, False, False]
    assert ref.crop_mask(pts, (1e-45, 1.2e-38, -1, 1, -1, 1)).tolist() == [False, False, False, False, True, True, False, False, False]
    assert ref.crop_mask(pts, (1e-45, FMIN, -1, 1, -1, 1)).tolist() == [False, False, False, False, True, False, False, False, False]
    assert not ref.crop_mask(pts, (np.nan, np.inf, -1, 1, -1, 1)).any()     # NaN face: every comparison false
    assert not ref.crop_mask(pts, (-np.inf, np.nan, -1, 1, -1, 1)).any()
    assert not ref.crop_mask(pts, (1.0, -1.0, -1, 1, -1, 1)).any()          # inverted


def test_crop_faces_are_rounded_to_float32():
    """0.1 as a double lies between two floats; the library receives float[6]."""
    f = F32(0.1)
    pts = points([(f, 0, 0), (np.nextafter(f, F32(0)), 0, 0)])
    assert ref.crop_mask(pts, (0.1, 1, -1, 1, -1, 1)).tolist() == [True, False]


def test_tile_predicates():
    pts = points([(0, 0, 0, 0, 0, 0, t) for t in (0, 1, 2, 3, 255, 128)])
    assert ref.tile_equals_mask(pts, 0).all()
    assert ref.tile_equals_mask(pts, 3).tolist() == [False, False, False, True, False, False]
    assert ref.tile_equals_mask(pts, 255).tolist() == [False, False, False, False, True, False]
    for t in (-1, 256, 300, -256):
        assert not ref.tile_equals_mask(pts, t).any()
    assert ref.tile_mask_mask(pts, 2).tolist() == [False, False, True, True, True, False]
    assert ref.tile_mask_mask(pts, 0x100).tolist() == [False] * 6      # bits above 0xff are dropped
    assert ref.tile_mask_mask(pts, 0x181).tolist() == [False, True, False, True, True, True]
    assert ref.tile_mask_mask(pts, -1).tolist() == [False, True, True, True, True, True]


def test_tile_predicate_is_the_oracles(orc):
    rng = np.random.default_rng(1)
    pts = np.zeros(4096, DT)
    pts["tile"] = rng.integers(0, 256, len(pts))
    pts["x"] = rng.random(len(pts), dtype=np.float32)
    for t in (-1, 0, 1, 7, 128, 255, 256, 300):
        assert ref.same_bytes(ref.compact(pts, ref.tile_equals_mask(pts, t)), orc.tilefilter(pts, t))


def test_distance_predicate_compares_in_double():
    d = np.array([0.5, np.nextafter(F32(0.5), F32(1)), NAN, INF, -INF, 0.1], F32)
    assert ref.distance_mask(d, 0.5).tolist() == [True, False, True, False, True, True]
    # 0.1f is above 0.1 in double: a float32 comparison would keep it
    assert ref.distance_mask(d, 0.1).tolist() == [False, False, True, False, True, False]
    assert ref.distance_mask(d, np.nan).all()


def test_colormap_goes_through_the_packed_word():
    pts = points([(1, 2, 3, 0x11, 0x22, 0x33, 0x44)])
    same = ref.colormap(pts, 0, 0)
    assert ref.same_bytes(same, pts)
    # bit 0 is b's lowest bit, bit 16 r's, bit 24 the tile's
    out = ref.colormap(pts, 0, 1)
    assert (out["r"][0], out["g"][0], out["b"][0], out["tile"][0]) == (0x11, 0x22, 0x33, 0x44)
    out = ref.colormap(pts, 1, 0)
    assert (out["r"][0], out["g"][0], out["b"][0], out["tile"][0]) == (0x11, 0x22, 0x32, 0x44)
    out = ref.colormap(pts, 0, 1 << 16)
    assert (out["r"][0], out["g"][0], out["b"][0], out["tile"][0]) == (0x11, 0x22, 0x33, 0x44)
    out = ref.colormap(pts, 1 << 16, 1 << 31)
    assert (out["r"][0], out["g"][0], out["b"][0], out["tile"][0]) == (0x10, 0x22, 0x33, 0xC4)
    out = ref.colormap(pts, 0xFFFFFFFF, 0x01020304)
    assert (out["r"][0], out["g"][0], out["b"][0], out["tile"][0]) == (0x02, 0x03, 0x04, 0x01)
    assert all(out[a][0] == pts[a][0] for a in "xyz")


def test_tilemap_and_join():
    pts = points([(1, 2, 3, 4, 5, 6, t) for t in (0, 1, 255)])
    table = np.arange(256)[::-1]
    assert ref.tilemap(pts, table)["tile"].tolist() == [255, 254, 0]
    assert ref.tilemap(pts, np.zeros(256))["tile"].tolist() == [0, 0, 0]
    assert len(ref.join(pts[:0], pts[:0])) == 0
    assert ref.same_bytes(ref.join(pts[:0], pts), pts) and ref.same_bytes(ref.join(pts, pts[:0]), pts)
    assert ref.same_bytes(ref.join(pts[:1], pts[1:]), pts)


def test_same_bytes_sees_nan_payloads_and_signed_zeros():
    a = points([(0.0, 1, 2)])
    b = a.copy()
    b["x"] = -0.0
    assert not ref.same_bytes(a, b) and ref.first_difference(a, b) == 0
    c, d = a.copy(), a.copy()
    c.view(np.uint32).reshape(-1, 4)[0, 1] = 0x7FC00000
    d.view(np.uint32).reshape(-1, 4)[0, 1] = 0x7FC00001
    assert not ref.same_bytes(c, d)
    assert ref.same_bytes(c, c.copy())
    assert not ref.same_bytes(a, ref.join(a, a)) and ref.first_difference(a, ref.join(a, a)) == 1


def test_min_distance_to_first_hand_worked(orc):
    """The oracle the cellsize tests use: min over i >= 1 of sqrtf(float32 d2), 0 when none is finite."""
    pts = points([(0, 0, 0), (3, 4, 0), (0, 0, 2)])
    assert orc.min_distance_to_first(pts) == 2.0
    assert orc.min_distance_to_first(points([(1, 1, 1), (1, 1, 1)])) == 0.0
    assert orc.min_distance_to_first(points([(3e38, 0, 0), (-3e38, 0, 0)])) == 0.0      # d2 overflows: no finite distance
    assert orc.min_distance_to_first(points([(NAN, 0, 0), (1, 0, 0)])) == 0.0
    assert orc.min_distance_to_first(points([(0, 0, 0), (NAN, 0, 0), (0, 0, 5)])) == 5.0
    assert orc.min_distance_to_first(points([(0, 0, 0), (1e-25, 0, 0)])) == 0.0           # d2 underflows to 0
    assert orc.min_distance_to_first(points([(0, 0, 0), (1e-22, 0, 0)])) == np.sqrt(F32(1e-22) * F32(1e-22))
