#!/usr/bin/env python
"""cwipc_cuda_transform against the host round trip a caller of the reference makes today to move points: get_numpy_matrix,
the matrix product in numpy, cwipc_from_numpy_matrix.

Workloads (synthetic.camera_cloud, 4 cameras): one whole-cloud matrix at 1 M and 8 M points, and a matrix per camera at
1 M and 8 M points, once with each camera's points together (as a capture joins its cameras' clouds) and once shuffled,
so that neighbouring lanes of a warp read different matrices.  The last row gives the same points random tile values and
one matrix for each of the 256 values: the kernel instantiated for 256 matrices, whose launch parameter is 25 KB.

Both arms run in one process and alternate (the order flips every repetition), with the L2 flushed before every call;
two warm-ups, then the median of --reps.  The library call is timed twice: `kernel_us` by CUDA events around the kernel
launch (the library's launch profile), `call_us` by CUDA events around the whole C-ABI call.  The round trip is wall
time up to a device synchronise after the upload.  GB/s is the kernel's 32 B per point (16 read, 16 written) over
kernel_us, and `frac` its share of the HBM bandwidth bench.py uses.  The two arms compute the same formula, so their
outputs must be byte-identical on every row.  The card's name and power limit are read, never set.

    python scripts/bench_transform.py [--reps 9]
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import time

import numpy as np

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)
sys.dont_write_bytecode = True

# (points, per-camera matrices, order)
WORKLOADS = [(1000000, False, "as generated"), (8000000, False, "as generated"), (1000000, True, "grouped"), (1000000, True, "shuffled"),
             (8000000, True, "grouped"), (8000000, True, "shuffled"), (1000000, True, "256 values")]


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True, timeout=30).stdout
        name, power = [f.strip() for f in out.strip().split(",")[:2]]
        return {"name": name, "power_limit": power}
    except Exception as e:  # pragma: no cover
        return {"name": None, "power_limit": None, "error": repr(e)}


def pose(seed):
    """A seeded rotation about a random axis with a translation of up to 2 m: a camera extrinsic."""
    rng = np.random.default_rng(seed)
    axis = rng.normal(size=3)
    axis /= np.linalg.norm(axis)
    a = rng.uniform(0, 2 * np.pi)
    k = np.array([[0, -axis[2], axis[1]], [axis[2], 0, -axis[0]], [-axis[1], axis[0], 0]])
    m = np.eye(4)
    m[:3, :3] = np.eye(3) + np.sin(a) * k + (1 - np.cos(a)) * (k @ k)
    m[:3, 3] = rng.uniform(-2, 2, 3)
    return m


def numpy_round_trip(cw, pc, table):
    """What a caller of the reference does: the points to the host, the formula of cwipc_cuda_transform in float64, back."""
    m = pc.get_numpy_matrix()
    xyz = m[:, :3].astype(np.float64)
    tiles = m[:, 6]
    listed = [t for t in table if t != 0]
    for t, mat in table.items():
        sel = tiles == t if t != 0 else ~np.isin(tiles, listed)
        x, y, z = xyz[sel, 0], xyz[sel, 1], xyz[sel, 2]
        for r in range(3):
            m[sel, r] = (((mat[r, 0] * x + mat[r, 1] * y) + mat[r, 2] * z) + mat[r, 3]).astype(np.float32)
    return cw.cwipc_from_numpy_matrix(m, pc.timestamp())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=9)
    args = ap.parse_args()
    if args.reps < 7:
        ap.error("--reps must be at least 7")
    import cwipc_util_b200 as cw
    from cwipc_util_b200 import synthetic
    from bench import measured_hbm_peak
    lib = cw.util.cwipc_util_dll_load()
    if cw.cuda_device_count() <= 0:
        raise SystemExit("bench_transform.py: no CUDA device")
    peak, peak_src = measured_hbm_peak()

    def library_call(pc, table):
        lib.cwipc_cuda_profile_reset()
        lib.cwipc_cuda_profile_enable(1)
        lib.cwipc_cuda_flush_l2()
        cw.cuda_synchronize()
        t = lib.cwipc_cuda_timer_create()
        lib.cwipc_cuda_timer_start(t)
        out = cw.cwipc_transform(pc, table)
        lib.cwipc_cuda_timer_stop(t)
        cw.cuda_synchronize()
        call_ms = lib.cwipc_cuda_timer_elapsed_ms(t)
        lib.cwipc_cuda_timer_destroy(t)
        lib.cwipc_cuda_profile_enable(0)
        need = lib.cwipc_cuda_profile_report(None, 0)
        buf = ctypes.create_string_buffer(need)
        lib.cwipc_cuda_profile_report(buf, need)
        prof = json.loads(buf.value.decode())
        assert prof["transform_kernel"]["launches"] == 1
        return {"kernel": prof["transform_kernel"]["total_ms"], "call": call_ms}, out

    def round_trip(pc, table):
        lib.cwipc_cuda_flush_l2()
        cw.cuda_synchronize()
        t0 = time.perf_counter()
        out = numpy_round_trip(cw, pc, table)
        cw.cuda_synchronize()
        return {"wall": (time.perf_counter() - t0) * 1e3}, out

    res = {"card": card(), "reps": args.reps, "hbm_peak_GBps": peak, "hbm_peak_source": peak_src, "rows": []}
    print(json.dumps(res["card"]), file=sys.stderr)
    clouds = {}
    for n_req, per_camera, order in WORKLOADS:
        if n_req not in clouds:
            clouds = {n_req: synthetic.camera_cloud(n_req, seed=1)}
        pts = clouds[n_req]
        if order == "grouped":   # each camera's points together, in camera order, as a capture joins them
            pts = pts[np.argsort(pts["tile"], kind="stable")]
        elif order == "shuffled":
            pts = pts[np.random.default_rng(2).permutation(len(pts))]
        elif order == "256 values":
            pts = pts.copy()
            pts["tile"] = np.random.default_rng(3).integers(0, 256, len(pts))
        tiles = sorted(int(t) for t in np.unique(pts["tile"]))
        table = {t: pose(10 + t) for t in tiles} if per_camera else {0: pose(1)}
        pc = cw.cwipc_from_numpy_array(pts, 1)
        arms = {"library": lambda: library_call(pc, table), "round_trip": lambda: round_trip(pc, table)}
        times = {"kernel": [], "call": [], "wall": []}
        outs = {}
        for i in range(args.reps + 2):
            for k in (("library", "round_trip") if i % 2 == 0 else ("round_trip", "library")):
                t, out = arms[k]()
                if i >= 2:
                    for name, ms in t.items():
                        times[name].append(ms)
                outs[k] = out
        a, b = outs["library"].get_numpy_array(), outs["round_trip"].get_numpy_array()
        identical = len(a) == len(b) == len(pts) and bool(np.array_equal(a.view(np.uint8), b.view(np.uint8)))
        med = {k: float(np.median(v)) for k, v in times.items()}
        n = len(pts)
        gbps = 32.0 * n / (med["kernel"] * 1e-3) / 1e9
        row = {"points": n, "matrices": len(table), "order": order, "kernel_us": round(med["kernel"] * 1e3, 2),
               "kernel_range_us": [round(min(times["kernel"]) * 1e3, 2), round(max(times["kernel"]) * 1e3, 2)],
               "call_us": round(med["call"] * 1e3, 2), "GBps": round(gbps, 1), "frac": round(gbps / peak, 4),
               "round_trip_ms": round(med["wall"], 3), "round_trip_range_ms": [round(min(times["wall"]), 3), round(max(times["wall"]), 3)],
               "speedup_vs_round_trip": round(med["wall"] / med["call"], 1), "outputs_identical": identical}
        res["rows"].append(row)
        print(json.dumps(row), file=sys.stderr)
        outs.clear()
        pc.free()
    print(json.dumps(res))
    if not all(r["outputs_identical"] for r in res["rows"]):
        raise SystemExit("bench_transform.py: the two arms' outputs differ")


if __name__ == "__main__":
    main()
