#!/usr/bin/env python
"""cwipc_remove_outliers timing on the bench's own frames (1M points -> downsample 0.01 -> ~47K voxels) and on raw clouds,
CUDA-event timed, per-kernel profile.  The kNN index settings come from the environment (CWIPC_CUDA_KNN_PITCH / _RC_FAR).

    python scripts/bench_sor.py [--reps 20]
"""
import argparse
import ctypes
import json
import os
import sys

import numpy as np

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--raw", type=int, default=1000000)
    ap.add_argument("--clean", action="store_true", help="the raw cloud is the clean synthetic cloud (as cwipc_synthetic generates it) instead of the jittered one")
    args = ap.parse_args()
    import bench
    import cwipc_util_b200 as cw
    from cwipc_util_b200 import synthetic
    lib = cw.util.cwipc_util_dll_load()
    frame = bench.make_frames(0, 1, 1)[0]
    pc = cw.cwipc_from_numpy_array(frame, 0)
    pc._set_cellsize(synthetic.cellsize_of(len(frame)))
    ds = cw.cwipc_downsample(pc, 0.01)
    raw_pts = synthetic.simulate_cameras(synthetic.synthetic_cloud(args.raw), 4) if args.clean else synthetic.camera_cloud(args.raw, seed=0)
    raw = cw.cwipc_from_numpy_array(raw_pts, 0)
    raw._set_cellsize(synthetic.cellsize_of(args.raw))

    def timed(fn, reps):
        times = []
        for i in range(reps + 3):
            cw.cuda_synchronize()
            t = lib.cwipc_cuda_timer_create()
            lib.cwipc_cuda_timer_start(t)
            out = fn()
            lib.cwipc_cuda_timer_stop(t)
            cw.cuda_synchronize()
            if i >= 3:
                times.append(lib.cwipc_cuda_timer_elapsed_ms(t))
            lib.cwipc_cuda_timer_destroy(t)
        return float(np.median(times)), out

    def profiled(fn, reps=5):
        lib.cwipc_cuda_profile_reset()
        lib.cwipc_cuda_profile_enable(1)
        for _ in range(reps):
            fn()
        cw.cuda_synchronize()
        lib.cwipc_cuda_profile_enable(0)
        need = lib.cwipc_cuda_profile_report(None, 0)
        buf = ctypes.create_string_buffer(need)
        lib.cwipc_cuda_profile_report(buf, need)
        prof = json.loads(buf.value.decode())
        return {k: round(v["total_ms"] * 1e3 / reps, 1) for k, v in sorted(prof.items(), key=lambda kv: -kv[1]["total_ms"])}

    res = {"env": {k: v for k, v in os.environ.items() if k.startswith("CWIPC_CUDA_KNN")}}
    for name, cloud, per_tile, reps in (("frame47k", ds, False, args.reps), ("raw1m", raw, False, 5), ("raw1m_pertile", raw, True, 5)):
        ms, out = timed(lambda: cw.cwipc_remove_outliers(cloud, 30, 1.0, per_tile), reps)
        res[name] = {"points": cloud.count(), "kept": out.count(), "ms": round(ms, 4), "kernels_us": profiled(lambda: cw.cwipc_remove_outliers(cloud, 30, 1.0, per_tile))}
    print(json.dumps(res))


if __name__ == "__main__":
    main()
