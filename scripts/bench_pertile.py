#!/usr/bin/env python
"""cwipc_cuda_downsample_pertile against the composition python/cwipc/registration/util.py:170-182 makes of the library's
filters (cwipc_tilefilter for each tile, cwipc_downsample of each, cwipc_join_multi of the results), on 4- and 8-camera
synthetic clouds (synthetic.camera_cloud, cellsize metadata as the synthetic source records it).

Both arms run in the same process and alternate (the order flips every repetition).  Every call is timed with CUDA events
on the calling thread's stream, from before the first launch to after the call returned (host work and read-backs in
between included), with the L2 flushed before it; two warm-ups, then the median of --reps.  The two arms' outputs are
compared record for record on every row.  The card's name and power limit are read, never set.

    python scripts/bench_pertile.py [--reps 9]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)
sys.dont_write_bytecode = True

# (points, cameras, voxel size): config 2's shape at both signs, 8 M points, 8 cameras, and a small cloud
WORKLOADS = [(1000000, 4, 0.01), (1000000, 4, -0.01), (8000000, 4, 0.005), (1000000, 8, 0.01), (160000, 4, 0.01)]


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True, timeout=30).stdout
        name, power = [f.strip() for f in out.strip().split(",")[:2]]
        return {"name": name, "power_limit": power}
    except Exception as e:  # pragma: no cover
        return {"name": None, "power_limit": None, "error": repr(e)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=9)
    args = ap.parse_args()
    if args.reps < 7:
        ap.error("--reps must be at least 7")
    import cwipc_util_b200 as cw
    from cwipc_util_b200 import synthetic
    lib = cw.util.cwipc_util_dll_load()
    if cw.cuda_device_count() <= 0:
        raise SystemExit("bench_pertile.py: no CUDA device")

    def timed(fn):
        lib.cwipc_cuda_flush_l2()
        cw.cuda_synchronize()
        t = lib.cwipc_cuda_timer_create()
        lib.cwipc_cuda_timer_start(t)
        res = fn()
        lib.cwipc_cuda_timer_stop(t)
        cw.cuda_synchronize()
        ms = lib.cwipc_cuda_timer_elapsed_ms(t)
        lib.cwipc_cuda_timer_destroy(t)
        return ms, res

    res = {"card": card(), "reps": args.reps, "rows": []}
    print(json.dumps(res["card"]), file=sys.stderr)
    for n_req, ncam, voxel in WORKLOADS:
        pts = synthetic.camera_cloud(n_req, seed=1, ncamera=ncam)
        _, first = np.unique(pts["tile"], return_index=True)
        tiles = [int(t) for t in pts["tile"][np.sort(first)]]
        pc = cw.cwipc_from_numpy_array(pts, 1)
        pc._set_cellsize(synthetic.cellsize_of(n_req))
        arms = {
            "pertile": lambda: cw.cwipc_downsample_pertile(pc, voxel),
            "composition": lambda: cw.cwipc_join_multi([cw.cwipc_downsample(cw.cwipc_tilefilter(pc, t), voxel) for t in tiles]),
        }
        times = {k: [] for k in arms}
        outs = {}
        for i in range(args.reps + 2):
            for k in (("pertile", "composition") if i % 2 == 0 else ("composition", "pertile")):
                ms, out = timed(arms[k])
                if i >= 2:
                    times[k].append(ms)
                outs[k] = out
        a, b = outs["pertile"].get_numpy_array(), outs["composition"].get_numpy_array()
        identical = len(a) == len(b) and bool(np.array_equal(a.view(np.uint8), b.view(np.uint8)))
        med = {k: float(np.median(v)) for k, v in times.items()}
        row = {"points": len(pts), "cameras": ncam, "tiles": len(tiles), "voxelsize": voxel, "voxels": len(a),
               "pertile_ms": round(med["pertile"], 4), "composition_ms": round(med["composition"], 4),
               "pertile_range_ms": [round(min(times["pertile"]), 4), round(max(times["pertile"]), 4)],
               "composition_range_ms": [round(min(times["composition"]), 4), round(max(times["composition"]), 4)],
               "saved_ms": round(med["composition"] - med["pertile"], 4), "speedup": round(med["composition"] / med["pertile"], 3), "outputs_identical": identical}
        res["rows"].append(row)
        print(json.dumps(row), file=sys.stderr)
        outs.clear()
        pc.free()
    print(json.dumps(res))
    if not all(r["outputs_identical"] for r in res["rows"]):
        raise SystemExit("bench_pertile.py: the two arms' outputs differ")


if __name__ == "__main__":
    main()
