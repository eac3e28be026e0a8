#!/usr/bin/env python
"""cwipc_cuda_icp against the numpy/cKDTree ICP loop of tests/icp_reference.py, on the registration step it serves: each
camera of the 4-camera synthetic cloud (synthetic.camera_cloud) registered against the other three.

Every camera is first moved by a known seeded pose (2-4 degrees about its centre, 2-4 cm) with cwipc_transform, then
cwipc_icp(source = that camera, target = cwipc_tilefilter_masked(pc, ~tile & 0xff), 0.05, max_iterations=30) runs with
open3d's default criteria.  Two sizes: the raw 1 M-point frame, and the frame after cwipc_downsample_pertile(0.005).

Columns: `call_ms` is a host clock around the call, which ends with its own read-back (a device synchronise);
`index_ms` is the device time of the kernels that build the target's search index (bounding box, keys, radix sort,
layout), and `per_iter_ms` the device time of one evaluation (icp_match_kernel + icp_reduce_kernel), both from the
library's launch profile (CUDA events) in a separate call; `ref_s` the reference loop's wall time in the same process.
The recovered matrices must agree: rotation within 1e-6 and the motion of the camera's centre within 1e-5 m.  The
card's name and power limit are read, never set.

--point-to-plane times cwipc_icp_point_to_plane on the same rows instead (normals from KDTreeSearchParamHybrid(normal_radius,
30), normal_radius = 0.01 on the raw frame and 0.02 after the downsample), against tests/icp_plane_reference.py.
`index_ms` then also holds icp_normals_kernel (reported on its own as `normals_ms`), and `per_iter_ms` is
icp_plane_match_kernel + icp_plane_reduce_kernel.

--colored times cwipc_icp_colored (lambda_geometric 0.968) on the same rows, against tests/icp_colored_reference.py fed the
library's normals and gradients (the reference's own are checked in tests/test_gpu_icp_colored.py).  `index_ms` then
also holds icp_normals_kernel and icp_gradients_kernel (reported on their own as `normals_ms` and `gradients_ms`; the
gradients take the 30 nearest points within 2 d = 0.1 m), and `per_iter_ms` is icp_colored_match_kernel +
icp_plane_reduce_kernel.  It then adds the recovery rows: the target is synthetic_cloud(40000) with 2 mm of noise, the
source the z > 0.05 half of a second noisy sampling turned by 3 or 6 degrees about the axis of revolution (y), 1 degree
about x and shifted by 1.5 cm (tests/icp_colored_reference.py: revolution_pair), d = 0.05, normal radius 0.04.  Each
row reports `residual_deg` and `residual_centre_m` of point-to-point, point-to-plane and colored ICP.

    python scripts/bench_icp.py [--reps 5] [--point-to-plane | --colored]
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import time

import numpy as np
from scipy.spatial.transform import Rotation

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)
sys.path.insert(0, os.path.join(REPO, "tests"))
sys.dont_write_bytecode = True

INDEX_KERNELS = ("bbox_octree_kernel", "knn_keygen_kernel", "radix_cluster_kernel", "radix_fused_kernel", "radix_hist_kernel", "radix_onesweep_kernel",
                 "radix_scan_kernel", "knn_layout_kernel")
EVAL_KERNELS = ("icp_match_kernel", "icp_reduce_kernel")
PLANE_EVAL_KERNELS = ("icp_plane_match_kernel", "icp_plane_reduce_kernel")
COLORED_EVAL_KERNELS = ("icp_colored_match_kernel", "icp_plane_reduce_kernel")
NORMAL_RADIUS = {"raw 1 M": 0.01, "downsample_pertile(0.005)": 0.02}


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True, timeout=30).stdout
        name, power = [f.strip() for f in out.strip().split(",")[:2]]
        return {"name": name, "power_limit": power}
    except Exception as e:  # pragma: no cover
        return {"name": None, "power_limit": None, "error": repr(e)}


def pose(seed, centre):
    rng = np.random.default_rng(seed)
    axis = rng.normal(size=3)
    R = Rotation.from_rotvec(np.radians(rng.uniform(2, 4)) * axis / np.linalg.norm(axis)).as_matrix()
    t = rng.normal(size=3)
    T = np.eye(4)
    T[:3, :3] = R
    T[:3, 3] = centre - R @ centre + rng.uniform(0.02, 0.04) * t / np.linalg.norm(t)
    return T


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    mode = ap.add_mutually_exclusive_group()
    mode.add_argument("--point-to-plane", action="store_true", help="time cwipc_icp_point_to_plane instead of cwipc_icp")
    mode.add_argument("--colored", action="store_true", help="time cwipc_icp_colored instead of cwipc_icp, and add the recovery rows")
    args = ap.parse_args()
    import cwipc_util_b200 as cw
    from cwipc_util_b200 import synthetic
    import icp_reference as ref
    import icp_plane_reference as pref
    import icp_colored_reference as cref
    plane, colored = args.point_to_plane, args.colored
    eval_kernels = PLANE_EVAL_KERNELS if plane else COLORED_EVAL_KERNELS if colored else EVAL_KERNELS
    lib = cw.util.cwipc_util_dll_load()
    if cw.cuda_device_count() <= 0:
        raise SystemExit("bench_icp.py: no CUDA device")

    def profiled(fn):
        lib.cwipc_cuda_profile_reset()
        lib.cwipc_cuda_profile_enable(1)
        out = fn()
        cw.cuda_synchronize()
        lib.cwipc_cuda_profile_enable(0)
        need = lib.cwipc_cuda_profile_report(None, 0)
        buf = ctypes.create_string_buffer(need)
        lib.cwipc_cuda_profile_report(buf, need)
        return out, json.loads(buf.value.decode())

    res = {"card": card(), "reps": args.reps, "estimation": "point-to-plane" if plane else "colored" if colored else "point-to-point", "rows": []}
    print(json.dumps(res["card"]), file=sys.stderr)
    raw = cw.cwipc_from_numpy_array(synthetic.camera_cloud(1000000, seed=1), 1)
    for size, pc in (("raw 1 M", raw), ("downsample_pertile(0.005)", cw.cwipc_downsample_pertile(raw, 0.005))):
        for tile in (1, 2, 4, 8):
            cam = cw.cwipc_tilefilter(pc, tile)
            centre = ref.xyz32(cam.get_numpy_array()).astype(np.float64).mean(0)
            P = pose(100 + tile, centre)
            src = cw.cwipc_transform(cam, P)
            tgt = cw.cwipc_tilefilter_masked(pc, ~tile & 0xff)
            if plane:
                call = lambda: cw.cwipc_icp_point_to_plane(src, tgt, 0.05, NORMAL_RADIUS[size], max_iterations=30)
            elif colored:
                call = lambda: cw.cwipc_icp_colored(src, tgt, 0.05, NORMAL_RADIUS[size], max_iterations=30)
            else:
                call = lambda: cw.cwipc_icp(src, tgt, 0.05, max_iterations=30)
            call()  # warm-up
            walls = []
            for _ in range(args.reps):
                cw.cuda_synchronize()
                t0 = time.perf_counter()
                r = call()
                walls.append((time.perf_counter() - t0) * 1e3)
            r, prof = profiled(call)
            normals_ms = prof["icp_normals_kernel"]["total_ms"] if plane or colored else 0.0
            gradients_ms = prof["icp_gradients_kernel"]["total_ms"] if colored else 0.0
            index_ms = sum(prof[k]["total_ms"] for k in INDEX_KERNELS if k in prof) + normals_ms + gradients_ms
            evals = prof[eval_kernels[0]]["launches"]
            per_iter = sum(prof[k]["total_ms"] for k in eval_kernels) / evals
            S, T = ref.xyz32(src.get_numpy_array()), ref.xyz32(tgt.get_numpy_array())
            t0 = time.perf_counter()
            # the library takes the centre of the box the target carries: its own on the raw frame, the whole frame's after
            # cwipc_downsample_pertile (which hands the input's box on)
            origin = pref.box_centre(T if pc is raw else ref.xyz32(raw.get_numpy_array()))
            if plane:
                want = pref.icp_point_to_plane(S, T, 0.05, NORMAL_RADIUS[size], max_iterations=30, origin=origin)
            elif colored:
                want = cref.icp_colored(src.get_numpy_array(), tgt.get_numpy_array(), 0.05, NORMAL_RADIUS[size], max_iterations=30, origin=origin,
                                        normals=cw.cwipc_estimate_normals(tgt, NORMAL_RADIUS[size]),
                                        gradients=cw.cwipc_estimate_color_gradients(tgt, NORMAL_RADIUS[size], 0.1))
            else:
                want = ref.icp(S, T, 0.05, max_iterations=30)
            ref_s = time.perf_counter() - t0
            d = r.matrix - want.matrix
            agree = bool(np.abs(d[:3, :3]).max() < 1e-6 and np.abs(d[:3, :3] @ centre + d[:3, 3]).max() < 1e-5)
            E = r.matrix @ P   # what is left of the known displacement
            row = {"size": size, "camera": tile, "source_points": cam.count(), "target_points": tgt.count(), "iterations": r.iterations,
                   "fitness": round(r.fitness, 6), "inlier_rmse": r.inlier_rmse, "call_ms": round(float(np.median(walls)), 3),
                   "call_range_ms": [round(min(walls), 3), round(max(walls), 3)], "index_ms": round(index_ms, 3), "per_iter_ms": round(per_iter, 3),
                   "evaluations": evals, **({"normals_ms": round(normals_ms, 3)} if plane or colored else {}),
                   **({"gradients_ms": round(gradients_ms, 3)} if colored else {}), "ref_s": round(ref_s, 2), "ref_iterations": want.iterations, "matrices_agree": agree,
                   "residual_deg": float(np.degrees(np.arccos(np.clip((np.trace(E[:3, :3]) - 1) / 2, -1, 1)))),
                   "residual_centre_m": float(np.linalg.norm(E[:3, :3] @ centre + E[:3, 3] - centre))}
            res["rows"].append(row)
            print(json.dumps(row), file=sys.stderr)
    if colored:
        res["recovery"] = []
        for y_degrees in (3.0, 6.0):
            source, target, P = cref.revolution_pair(y_degrees)
            sp, tp = cw.cwipc_from_numpy_array(source, 1), cw.cwipc_from_numpy_array(target, 1)
            centre = ref.move(ref.xyz32(source), np.linalg.inv(P)).astype(np.float64).mean(0)
            row = {"y_degrees": y_degrees, "source_points": sp.count(), "target_points": tp.count()}
            for name, r in (("point-to-point", cw.cwipc_icp(sp, tp, 0.05)), ("point-to-plane", cw.cwipc_icp_point_to_plane(sp, tp, 0.05, 0.04)),
                            ("colored", cw.cwipc_icp_colored(sp, tp, 0.05, 0.04))):
                E = r.matrix @ P
                row[name] = {"iterations": r.iterations, "fitness": round(r.fitness, 6),
                             "residual_deg": float(np.degrees(np.arccos(np.clip((np.trace(E[:3, :3]) - 1) / 2, -1, 1)))),
                             "residual_centre_m": float(np.linalg.norm(E[:3, :3] @ centre + E[:3, 3] - centre))}
            res["recovery"].append(row)
            print(json.dumps(row), file=sys.stderr)
    print(json.dumps(res))
    if not all(r["matrices_agree"] for r in res["rows"]):
        raise SystemExit("bench_icp.py: the library's and the reference's matrices differ")


if __name__ == "__main__":
    main()
