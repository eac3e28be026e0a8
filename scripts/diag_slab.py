import os, sys
import numpy as np
REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO); sys.path.insert(0, os.path.join(REPO, "oracle")); sys.path.insert(0, os.path.join(REPO, "tests"))
import cwipc_util_b200 as cw
from cwipc_util_b200 import synthetic
import oracle as orc
world = 2
pts = synthetic.simulate_cameras(synthetic.synthetic_cloud(640000), 4)
edges = np.quantile(pts["x"], np.linspace(0, 1, world + 1)); edges[0], edges[-1] = -np.inf, np.inf
slab_of = np.clip(np.searchsorted(edges, pts["x"], side="right") - 1, 0, world - 1)
whole = np.concatenate([pts[slab_of == r] for r in range(world)])
cs0 = float(synthetic.cellsize_of(640000))
want, cs, keys6, counts = orc.downsample(whole, 0.005, cs0, want_keys=True)
def run(path):
    if path: os.environ["CWIPC_CUDA_DS_PATH"] = path
    else: os.environ.pop("CWIPC_CUDA_DS_PATH", None)
    pc = cw.cwipc_from_numpy_array(whole, 7); pc._set_cellsize(cs0)
    return cw.cwipc_downsample(pc, 0.005).get_numpy_array().copy()
res = {p or "fused": run(p) for p in (None, "twopass", "generic")}
for name, got in res.items():
    same_len = len(got) == len(want)
    ok_tile = same_len and np.array_equal(got["tile"], want["tile"])
    dx = np.abs(got["x"].astype(np.float64) - want["x"]).max() if same_len else None
    bad = np.flatnonzero((np.abs(got["x"] - want["x"]) > 1e-6) | (np.abs(got["y"] - want["y"]) > 1e-6) | (np.abs(got["z"] - want["z"]) > 1e-6) | (got["tile"] != want["tile"])) if same_len else []
    print(name, "len", len(got), len(want), "tile ok", ok_tile, "max dx", dx, "bad", len(bad), bad[:5])
    for i in bad[:3]:
        print("   got", got[i], "want", want[i], "count", counts[i])
a, b = res["fused"], res["twopass"]
print("fused == twopass:", np.array_equal(a, b), "twopass == generic:", np.array_equal(b, res["generic"]))
if not np.array_equal(a, b) and len(a) == len(b):
    d = np.flatnonzero(a != b); print("differs at", d[:10]); print(a[d[:3]], b[d[:3]])
