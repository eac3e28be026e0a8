#!/usr/bin/env python
"""Quick A/B of the bench's `value` (device-resident frame chain, 15 host threads on one GPU) for another build of the
library or a setting read from the environment at load time: one process per variant, a fraction of bench.py's run time.

    CWIPC_CUDA_LIBRARY=/path/to/libcwipc_util_cuda.so python scripts/ab_value.py [--frames 60] [--steps 6] [--pageable] [--profile]

Prints one JSON line: value (Mpoints/s), optionally the pageable end-to-end figure and the per-kernel times of a
single-stream replay.  Diagnostics only; the numbers of record come from bench.py.
"""
import argparse
import ctypes
import json
import os
import sys
import threading

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)
import bench  # noqa: E402  (exports CUDA_DEVICE_MAX_CONNECTIONS before the first CUDA call)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=60)
    ap.add_argument("--steps", type=int, default=6)
    ap.add_argument("--passes", type=int, default=8)
    ap.add_argument("--workers", type=int, default=bench.WORKERS)
    ap.add_argument("--pageable", action="store_true")
    ap.add_argument("--e2e", action="store_true")
    ap.add_argument("--profile", action="store_true")
    ap.add_argument("--tag", default="")
    args = ap.parse_args()
    import cwipc_util_b200 as cw
    from cwipc_util_b200 import synthetic
    lib = cw.util.cwipc_util_dll_load()
    cw.cuda_set_device(0)
    n = bench.POINTS_PER_FRAME
    cellsize = synthetic.cellsize_of(n)
    frames = bench.make_frames(0, args.frames, 1)
    device_frames, host_ptrs = [], []
    for f, pts in enumerate(frames):
        pc = cw.cwipc_from_numpy_array(pts, f)
        pc._set_cellsize(cellsize)
        device_frames.append(pc)
        if args.e2e:
            hp = lib.cwipc_cuda_host_alloc(n * 16)
            ctypes.memmove(hp, pts.ctypes.data, n * 16)
            host_ptrs.append(hp)
    nworkers = args.workers
    host_out = [lib.cwipc_cuda_host_alloc(n * 16) for _ in range(nworkers)]
    state = {"frames": frames, "device_frames": device_frames, "host_ptrs": host_ptrs, "host_out": host_out, "cellsize": cellsize, "stop": False,
             "mode": "resident", "mid_frames": [cw.cwipc_downsample(pc, bench.VOXEL) for pc in device_frames] if os.environ.get("BENCH_STAGE", "") == "outliers" else []}
    barrier = threading.Barrier(nworkers + 1)
    workers = [bench.Worker(w, nworkers, 0, cw, lib, barrier, state) for w in range(nworkers)]
    for w in workers:
        w.start()
    bench.run_steps(workers, barrier, state, lib, "resident", 3, passes=args.passes)
    cw.cuda_synchronize()
    res = {"tag": args.tag, "frames": args.frames, "points_per_frame": n}
    vals = []
    for _ in range(2):   # two timed regions: the spread says how much a difference between variants means
        ms = bench.run_steps(workers, barrier, state, lib, "resident", args.steps, passes=args.passes)
        vals.append(round(args.frames * args.passes * args.steps * n / (ms / 1e3) / 1e6, 1))
    res["value"] = max(vals)
    res["values"] = vals
    res["us_per_frame"] = round(1e6 * n / (max(vals) * 1e6), 1)
    if args.e2e:
        bench.run_steps(workers, barrier, state, lib, "e2e", 1, passes=1)
        ms = bench.run_steps(workers, barrier, state, lib, "e2e", 2, passes=2)
        res["e2e"] = round(args.frames * 2 * 2 * n / (ms / 1e3) / 1e6, 1)
    if args.pageable:
        bench.run_steps(workers, barrier, state, lib, "e2e_pageable", 1, passes=1)
        ms = bench.run_steps(workers, barrier, state, lib, "e2e_pageable", 2, passes=2)
        res["pageable"] = round(args.frames * 2 * 2 * n / (ms / 1e3) / 1e6, 1)
    state["stop"] = True
    barrier.wait()
    if args.profile:
        for f in range(2):
            workers[0].frame_chain(device_frames[f]).free()
        cw.cuda_synchronize()
        lib.cwipc_cuda_profile_reset()
        lib.cwipc_cuda_profile_enable(1)
        nprof = min(args.frames, 12)
        for f in range(nprof):
            workers[0].frame_chain(device_frames[f]).free()
        cw.cuda_synchronize()
        lib.cwipc_cuda_profile_enable(0)
        need = lib.cwipc_cuda_profile_report(None, 0)
        buf = ctypes.create_string_buffer(need)
        lib.cwipc_cuda_profile_report(buf, need)
        prof = json.loads(buf.value.decode())
        res["kernels_us"] = {k: round(v["total_ms"] * 1e3 / max(1, v["launches"]), 1) for k, v in sorted(prof.items(), key=lambda kv: -kv[1]["total_ms"])}
        res["kernel_us_per_frame"] = round(sum(v["total_ms"] for v in prof.values()) * 1e3 / nprof, 1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
