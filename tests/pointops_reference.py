"""A plain numpy reference of the per-point filters: stable compaction by a predicate, the tile map, the colour map and
the join (no library calls).

Every predicate is evaluated in float32 or on the 8-bit tile exactly as it is written in the reference filters, so that
comparisons with NaN, -0.0, denormals and infinities come out as they do there:
  crop                (x0 <= x) & (x < x1) & (y0 <= y) & (y < y1) & (z0 <= z) & (z < z1)
  tilefilter          tile == 0 (the argument) keeps every point, else int(point.tile) == tile
  masked tilefilter   (point.tile & (mask & 0xff)) != 0
  distance filter     !(double(dist) > threshold)
The result of a compaction is pts[mask]: the kept records, in input order, byte for byte.
"""
import numpy as np

POINT_DTYPE = np.dtype([("x", "<f4"), ("y", "<f4"), ("z", "<f4"), ("r", "u1"), ("g", "u1"), ("b", "u1"), ("tile", "u1")])


def crop_mask(pts, box):
    """box = (x0, x1, y0, y1, z0, z1), each face rounded to float32 as the C ABI's float[6] holds it."""
    x0, x1, y0, y1, z0, z1 = (np.float32(v) for v in box)
    return (x0 <= pts["x"]) & (pts["x"] < x1) & (y0 <= pts["y"]) & (pts["y"] < y1) & (z0 <= pts["z"]) & (pts["z"] < z1)


def tile_equals_mask(pts, tile):
    """`tile == 0 || tile == pt.tile` with an int argument and an 8-bit tile: -1, 256 or 300 select nothing."""
    if tile == 0:
        return np.ones(len(pts), bool)
    return pts["tile"].astype(np.int64) == int(tile)


def tile_mask_mask(pts, mask):
    return (pts["tile"] & np.uint8(int(mask) & 0xFF)) != 0


def distance_mask(dist, threshold):
    return ~(np.asarray(dist, np.float32).astype(np.float64) > float(threshold))


def compact(pts, mask):
    return pts[np.asarray(mask, bool)]


def tilemap(pts, table):
    """Every point's tile replaced by table[tile]; everything else unchanged."""
    out = pts.copy()
    out["tile"] = np.asarray(table, np.uint8)[pts["tile"]]
    return out


def colormap(pts, clear_bits, set_bits):
    """Through PCL's packed word rgba = tile<<24 | r<<16 | g<<8 | b: (rgba & ~clear) | set, then unpacked."""
    rgba = (pts["tile"].astype(np.uint32) << 24) | (pts["r"].astype(np.uint32) << 16) | (pts["g"].astype(np.uint32) << 8) | pts["b"].astype(np.uint32)
    rgba = (rgba & np.uint32(~int(clear_bits) & 0xFFFFFFFF)) | np.uint32(int(set_bits) & 0xFFFFFFFF)
    out = pts.copy()
    out["tile"] = (rgba >> 24).astype(np.uint8)
    out["r"] = ((rgba >> 16) & 0xFF).astype(np.uint8)
    out["g"] = ((rgba >> 8) & 0xFF).astype(np.uint8)
    out["b"] = (rgba & 0xFF).astype(np.uint8)
    return out


def join(a, b):
    return np.concatenate([np.asarray(a, POINT_DTYPE), np.asarray(b, POINT_DTYPE)])


def same_bytes(got, want):
    """Record for record, byte for byte: NaN payloads and the sign of zero count."""
    got, want = np.ascontiguousarray(got), np.ascontiguousarray(want)
    return len(got) == len(want) and np.array_equal(got.view(np.uint8), want.view(np.uint8))


def first_difference(got, want):
    """Index of the first record that differs (or the shorter length), for failure messages."""
    m = min(len(got), len(want))
    a = np.ascontiguousarray(got[:m]).view(np.uint8).reshape(m, 16)
    b = np.ascontiguousarray(want[:m]).view(np.uint8).reshape(m, 16)
    bad = np.flatnonzero(np.any(a != b, axis=1))
    return int(bad[0]) if len(bad) else m
