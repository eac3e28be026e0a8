#!/usr/bin/env python
"""bench.py -- headline benchmark of the cwipc filter hot path on B200.

Metric (BASELINE.json): Mpoints/s for downsample + remove_outliers at 1/2/4/8 B200; % of HBM GB/s peak.

Workload (BASELINE.json configs[4], the config the metric is quoted on): a 240-frame sequence of 1M-point
(1000 x 1000) 4-camera synthetic frames, per frame  cwipc_downsample(0.01) -> cwipc_remove_outliers(30, 1.0,
perTile=False), frame-sharded over the GPUs (frame f -> GPU f mod N) with no collective on the data path.
Scaling is STRONG: the same 240 frames at every N (240 / N per GPU).  A step is PASSES (8) passes over the
sequence, so that the timed region of K = 20 steps stays above half a second at 8 GPUs too.

The same run also times BASELINE.json configs[3] on rank 0 (`config4` in the JSON line: one 8M-point cloud,
cwipc_downsample at the five voxel sizes of the sweep and downsample(0.005) -> remove_outliers), the
configuration the north-star HBM-roofline target is stated on.

    python bench.py --gpus 1 --steps 10 --warmup 3            # our arm (CUDA library through its C ABI)
    python bench.py --impl reference --gpus 1 ...             # the reference's CPU path (oracle port, all host cores)
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

`value`   : device-resident inputs, CUDA-event timed (max over worker streams and over ranks).
`e2e`     : same frames from page-locked HOST buffers through cwipc_from_points (H2D inside the timed
            region) and the result read back with cwipc_pointcloud_copy_uncompressed (D2H inside).
`roofline`: dominant kernel of the step (largest total device time in a profiled pass of the same step):
            algorithmic bytes of its launches / their CUDA-event duration, against MEASURED_PEAKS.json.
`cpu_baseline`: the oracle (a single-threaded port of the reference path) timed on a bounded sample.

--dump-outputs DIR writes what the timed `value` path returned in the last pass of its last step, so that two builds can
be compared output for output (the inputs depend only on the arguments):
  DIR/counts_rank<r>.npy   float64 (frames, 2): sequence index of every frame of rank r, points the chain returned for it
  DIR/frame<f>.npy         float32 (points, 7): x, y, z, r, g, b, tile of the chain's result for frame f, for a fixed
                           seeded sample of DUMP_FRAMES frames (rows subsampled with a seed if the files would exceed 64 MB)
"""
from __future__ import annotations

import argparse
import ctypes
import json
import os
import sys
import threading
import time

import numpy as np

# 30 streams per GPU: more hardware queues than the default 8 (must be set before the CUDA context exists)
os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")

REPO = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, REPO)
sys.dont_write_bytecode = True   # the tree may be read-only: the bench writes nothing into it

POINTS_PER_FRAME = int(os.environ.get("BENCH_POINTS", 1000 * 1000))   # BENCH_POINTS: diagnostic only (host-bound or GPU-bound?)
VOXEL = 0.01
K, STDDEV = int(os.environ.get("BENCH_K", 30)), 1.0   # BENCH_K: diagnostic only
SEQUENCE_FRAMES = 240        # configs[4]: the whole sequence, split over the GPUs
PASSES = 8                   # passes over the sequence per step
WORKERS = 30                 # host threads (one CUDA stream each) feeding one GPU; divides the rank's share of the 240 frames at 1, 2 and 4 GPUs
                             # (scripts/ab_value.py on one B200, 16 host cores: 15 threads 8.2-8.5, 24 threads 8.3-8.6, 32 threads 8.6-8.7 Gpoints/s)
HBM_FALLBACK_GBS = 6650.0    # B200_PROFILING.md fallback when MEASURED_PEAKS.json is absent
DUMP_FRAMES = 32             # --dump-outputs: frames written in full (of the rank's share of the sequence)
DUMP_BYTES = 64 << 20        # --dump-outputs: at most this much in all


def log(*a):
    print(*a, file=sys.stderr, flush=True)


# --------------------------------------------------------------------------------------------------
# workload
# --------------------------------------------------------------------------------------------------
def make_frames(first, count, stride):
    """Frames first, first+stride, ...: same geometry, per-frame jitter/outliers seeded by the frame index."""
    from concurrent.futures import ThreadPoolExecutor
    from cwipc_util_b200 import synthetic
    base = synthetic.simulate_cameras(synthetic.synthetic_cloud(POINTS_PER_FRAME), 4)

    def one(j):
        seed = first + j * stride
        return synthetic.add_outliers(synthetic.add_noise(base, 0.002, seed), 0.005, seed)

    cores = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    with ThreadPoolExecutor(max(1, min(8, cores // max(1, int(os.environ.get("LOCAL_WORLD_SIZE", "1")))))) as ex:
        return list(ex.map(one, range(count)))


# --------------------------------------------------------------------------------------------------
# clocks
# --------------------------------------------------------------------------------------------------
class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons of one GPU while the timed region runs."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index = index
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._halt = threading.Event()
        self.armed = threading.Event()      # samples are kept only while the timed region runs
        self.ready = threading.Event()      # NVML initialised (it stalls CUDA calls while it loads)

    def run(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            h = pynvml.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM)
            names = {
                getattr(pynvml, "nvmlClocksEventReasonHwSlowdown", 0x8): "hw_slowdown",
                getattr(pynvml, "nvmlClocksEventReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
                getattr(pynvml, "nvmlClocksEventReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
                getattr(pynvml, "nvmlClocksEventReasonSwPowerCap", 0x4): "sw_power_cap",
            }
            pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM)
            self.ready.set()
            while not self._halt.is_set():
                if not self.armed.is_set():
                    time.sleep(0.005)
                    continue
                self.samples.append(pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM))
                try:
                    mask = pynvml.nvmlDeviceGetCurrentClocksEventReasons(h)
                except Exception:
                    mask = pynvml.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                for bit, name in names.items():
                    if mask & bit:
                        self.reasons.add(name)
                time.sleep(0.01)
        except Exception as e:  # pragma: no cover
            self.reasons.add(f"sampler_error:{type(e).__name__}")
            self.ready.set()

    def stop(self):
        self._halt.set()
        self.join(timeout=2)
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2] if s else None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(s)}


# --------------------------------------------------------------------------------------------------
# our arm
# --------------------------------------------------------------------------------------------------
class Worker(threading.Thread):
    """One host thread = one CUDA stream.  Processes its share of the rank's frames every step."""

    def __init__(self, wid, nworkers, dev, cw, lib, barrier, state):
        super().__init__(daemon=True)
        self.wid, self.nworkers, self.dev, self.cw, self.lib = wid, nworkers, dev, cw, lib
        self.barrier, self.state = barrier, state
        self.error = None
        self.timers = []          # one timer per step
        self.out_points = 0
        self.mid_points = 0
        self.d2h_bytes = 0
        self.last_counts = {}     # frame -> points returned in the last pass (--dump-outputs)
        self.kept = {}            # frame -> result cloud of the last pass, for the frames state["keep"] names

    def frame_chain(self, pc):
        stage = os.environ.get("BENCH_STAGE", "")   # diagnostic only: time one stage of the chain
        if stage == "downsample":
            d = self.cw.cwipc_downsample(pc, VOXEL)
            self.mid_points += d.count()
            return d
        if stage == "outliers":
            return self.cw.cwipc_remove_outliers(self.state["mid_frames"][self.state["device_frames"].index(pc)], K, STDDEV, False)
        d = self.cw.cwipc_downsample(pc, VOXEL)
        o = self.cw.cwipc_remove_outliers(d, K, STDDEV, False)
        self.mid_points += d.count()
        d.free()
        return o

    def run(self):
        try:
            cw, lib, st = self.cw, self.lib, self.state
            cw.cuda_set_device(self.dev)
            mine = list(range(self.wid, len(st["frames"]), self.nworkers))
            while True:
                self.barrier.wait()                      # step start (or shutdown)
                if st["stop"]:
                    return
                mode = st["mode"]
                timer = lib.cwipc_cuda_timer_create()
                self.timers.append(timer)
                self.out_points = 0
                self.mid_points = 0
                self.d2h_bytes = 0
                lib.cwipc_cuda_timer_start(timer)
                # K steps back to back: a worker starts its share of step s+1 as soon as it has finished its share of
                # step s (frames are independent), the timed region is bracketed once, around all K steps
                order = [f for _ in range(st["nsteps"] * st["passes"]) for f in mine]
                last_pass = len(order) - len(mine) if mode == "resident" and st["keep"] is not None else len(order)
                for i, f in enumerate(order):
                    if mode == "resident":
                        o = self.frame_chain(st["device_frames"][f])
                        m = o.count()
                        self.out_points += m
                        if i >= last_pass:
                            self.last_counts[f] = m
                            if f in st["keep"]:
                                self.kept[f] = o     # read back after the timed region
                                continue
                        o.free()
                    else:  # e2e: pinned host -> device -> filters -> pinned host
                        err = ctypes.c_char_p()
                        src = st["host_ptrs"][f] if mode == "e2e" else st["frames"][f].ctypes.data   # e2e_pageable: the caller's own (pageable) numpy memory
                        p = lib.cwipc_from_points(src, POINTS_PER_FRAME * 16, POINTS_PER_FRAME, f, ctypes.byref(err), cw.CWIPC_API_VERSION)
                        if not p:
                            raise RuntimeError(f"cwipc_from_points failed: {err.value}")
                        pc = cw.cwipc_pointcloud_wrapper(p)
                        pc._set_cellsize(st["cellsize"])
                        o = self.frame_chain(pc)
                        nbytes = o.get_uncompressed_size()
                        got = lib.cwipc_pointcloud_copy_uncompressed(o.as_cwipc_p(), st["host_out"][self.wid], nbytes)
                        if got < 0:
                            raise RuntimeError("copy_uncompressed failed")
                        self.out_points += got
                        self.d2h_bytes += nbytes
                        o.free()
                        pc.free()
                lib.cwipc_cuda_timer_stop(timer)
                cw.cuda_synchronize()
                self.barrier.wait()                      # step end
        except Exception as e:  # pragma: no cover
            self.error = e
            try:
                self.barrier.abort()
            except Exception:
                pass


def run_steps(workers, barrier, state, lib, mode, nsteps, passes=None):
    """Run nsteps steps in `mode` inside ONE timed region; returns its device time in ms: from the first worker
    stream's start event to the last one's stop event (host barrier + device synchronize on both sides)."""
    state["mode"] = mode
    state["nsteps"] = nsteps
    state["passes"] = PASSES if passes is None else passes
    barrier.wait()
    barrier.wait()
    for w in workers:
        if w.error:
            raise w.error
    ts = [w.timers[-1] for w in workers]
    ms = max(lib.cwipc_cuda_timer_span_ms(a, b) for a in ts for b in ts)
    for w in workers:
        for t in w.timers:
            lib.cwipc_cuda_timer_destroy(t)
        w.timers = []
    return ms


def dump_outputs(out_dir, workers, rank, world):
    """--dump-outputs (see the module docstring): frame j of this rank is frame rank + j * world of the sequence."""
    counts = {j: m for w in workers for j, m in w.last_counts.items()}
    kept = {j: o for w in workers for j, o in w.kept.items()}
    for w in workers:
        w.kept = {}
    np.save(os.path.join(out_dir, f"counts_rank{rank}.npy"),
            np.array([(rank + j * world, counts[j]) for j in sorted(counts)], np.float64).reshape(-1, 2))
    # 7 float32 per point; every rank's files together stay within DUMP_BYTES (headers and the counts included)
    max_rows = (DUMP_BYTES // world - 16 * len(counts) - 4096 * (len(kept) + 1)) // (7 * 4 * max(1, len(kept)))
    for j in sorted(kept):
        f = rank + j * world
        pts = kept[j].get_numpy_array()
        kept[j].free()
        if len(pts) > max_rows:
            pts = pts[np.sort(np.random.default_rng(f).choice(len(pts), max_rows, replace=False))]
        cols = np.stack([pts[c].astype(np.float32) for c in ("x", "y", "z", "r", "g", "b", "tile")], axis=1)
        np.save(os.path.join(out_dir, f"frame{f:03d}.npy"), cols)


def dist_setup(args):
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        # stdout carries exactly one JSON line: keep NCCL's "NCCL version ..." banner (NCCL_DEBUG=VERSION/INFO) off it
        if os.environ.get("NCCL_DEBUG", "").upper() in ("VERSION", "INFO", "TRACE"):
            os.environ["NCCL_DEBUG_FILE"] = os.environ.get("NCCL_DEBUG_FILE", "/dev/stderr")
        import torch
        import torch.distributed as dist
        torch.cuda.set_device(local)
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl")
        return world, rank, local, dist, torch
    return world, rank, local, None, None


def dist_barrier(dist, torch):
    if dist is not None:
        t = torch.zeros(1, device="cuda")
        dist.all_reduce(t)
        torch.cuda.synchronize()


def dist_reduce(dist, torch, value, op):
    if dist is None:
        return value
    t = torch.tensor([float(value)], dtype=torch.float64, device="cuda")
    dist.all_reduce(t, op=getattr(dist.ReduceOp, op))
    return float(t.item())


def measured_hbm_peak():
    path = os.path.join(REPO, "MEASURED_PEAKS.json")
    try:
        return float(json.load(open(path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return HBM_FALLBACK_GBS, "fallback (B200_PROFILING.md)"


def cpu_baseline_sample(frames, nframes):
    """The oracle (single-threaded port of the reference path) on a bounded sample of the same frames."""
    sys.path.insert(0, os.path.join(REPO, "oracle"))
    import oracle
    from cwipc_util_b200 import synthetic
    cellsize = synthetic.cellsize_of(POINTS_PER_FRAME)
    oracle.load()
    t0 = time.perf_counter()
    for f in range(nframes):
        pts = frames[f % len(frames)]
        ds, cs, _, _ = oracle.downsample(pts, VOXEL, cellsize)
        oracle.remove_outliers(ds, K, STDDEV, False)
    dt = time.perf_counter() - t0
    return nframes * POINTS_PER_FRAME / dt / 1e6, dt


def measure_config4(cw, lib, peak):
    """BASELINE.json configs[3] on one GPU: ONE 8M-point (2828 x 2828) cloud, cwipc_downsample at the five voxel sizes of the
    sweep and downsample(0.005) -> remove_outliers(30, 1.0), device resident, CUDA-event timed around the C-ABI calls with the
    L2 flushed before every call.  Two clouds: `synthetic` is the cloud as cwipc_synthetic generates it (SURVEY.md 8d config 4;
    4-camera tile bits), `jittered` adds 2 mm noise and 0.5 % outliers (scan order no longer voxel-coherent).
    frac = compulsory bytes (16 B per point in + 16 B per point out, per stage) / time / HBM peak."""
    from cwipc_util_b200 import synthetic
    n_req = 2828 * 2828
    out = {"points": n_req, "hbm_peak_GBps": peak, "what": "configs[3]: one 8M-point cloud on one GPU (rank 0), median of 5 after 2 warm-ups, L2 flushed before every call", "clouds": {}}

    def timed(fn, reps=5):
        times, res = [], None
        for i in range(reps + 2):
            lib.cwipc_cuda_flush_l2()
            cw.cuda_synchronize()
            t = lib.cwipc_cuda_timer_create()
            lib.cwipc_cuda_timer_start(t)
            res = fn()
            lib.cwipc_cuda_timer_stop(t)
            cw.cuda_synchronize()
            if i >= 2:
                times.append(lib.cwipc_cuda_timer_elapsed_ms(t))
            lib.cwipc_cuda_timer_destroy(t)
        return float(np.median(times)), res

    def profiled(fn):
        lib.cwipc_cuda_profile_reset()
        lib.cwipc_cuda_profile_enable(1)
        lib.cwipc_cuda_flush_l2()
        r = fn()
        cw.cuda_synchronize()
        lib.cwipc_cuda_profile_enable(0)
        need = lib.cwipc_cuda_profile_report(None, 0)
        buf = ctypes.create_string_buffer(need)
        lib.cwipc_cuda_profile_report(buf, need)
        prof = json.loads(buf.value.decode())
        return r, {k: {"us": round(v["total_ms"] * 1e3, 1), "launches": v["launches"], "GBps": round(v["bytes"] / max(v["total_ms"], 1e-9) / 1e6, 1),
                       "frac": round(v["bytes"] / max(v["total_ms"], 1e-9) / 1e6 / peak, 4)}
                   for k, v in sorted(prof.items(), key=lambda kv: -kv[1]["total_ms"]) if k != "flush_kernel"}

    base = synthetic.simulate_cameras(synthetic.synthetic_cloud(n_req), 4)
    for name in ("synthetic", "jittered"):
        pts = base if name == "synthetic" else synthetic.add_outliers(synthetic.add_noise(base, 0.002, 1), 0.005, 1)
        n = len(pts)
        pc = cw.cwipc_from_numpy_array(pts, 1)
        pc._set_cellsize(synthetic.cellsize_of(n_req))
        rows = []
        for vs in (0.002, 0.005, 0.01, 0.02, 0.05):
            ms, d = timed(lambda: cw.cwipc_downsample(pc, vs))
            v = d.count()
            _, kernels = profiled(lambda: cw.cwipc_downsample(pc, vs))
            rows.append({"voxelsize": vs, "voxels": v, "ms": round(ms, 4), "Mpoints_per_s": round(n / ms / 1e3, 1), "compulsory_GBps": round(16.0 * (n + v) / ms / 1e6, 1),
                         "frac": round(16.0 * (n + v) / ms / 1e6 / peak, 4), "kernels": kernels})
        ms, res = timed(lambda: (lambda d: (d, cw.cwipc_remove_outliers(d, K, STDDEV, False)))(cw.cwipc_downsample(pc, 0.005)))
        d, o = res
        v, m = d.count(), o.count()
        _, kernels = profiled(lambda: cw.cwipc_remove_outliers(cw.cwipc_downsample(pc, 0.005), K, STDDEV, False))
        chain = {"what": "downsample(0.005) -> remove_outliers(30, 1.0, perTile=False)", "voxels": v, "kept": m, "ms": round(ms, 4), "Mpoints_per_s": round(n / ms / 1e3, 1),
                 "frac": round(16.0 * (n + 2 * v + m) / ms / 1e6 / peak, 4), "kernels": kernels}
        # outlier removal of the raw cloud itself (the north star's "8M-point ... outlier removal"): 16 B read per point + survivors written
        for _ in range(2):   # (the first calls at this size grow the library's memory pool)
            cw.cwipc_remove_outliers(pc, K, STDDEV, False).free()
        ms, o = timed(lambda: cw.cwipc_remove_outliers(pc, K, STDDEV, False), reps=3)
        m = o.count()
        _, kernels = profiled(lambda: cw.cwipc_remove_outliers(pc, K, STDDEV, False))
        raw = {"what": "remove_outliers(30, 1.0, perTile=False) of the raw cloud", "kept": m, "ms": round(ms, 4), "Mpoints_per_s": round(n / ms / 1e3, 1),
               "frac": round(16.0 * (n + m) / ms / 1e6 / peak, 4), "kernels": kernels}
        out["clouds"][name] = {"points": n, "downsample": rows, "chain": chain, "remove_outliers_raw": raw}
        pc.free()
    return out


def measure_slab(cw, dist, torch, rank, world):
    """BASELINE.json configs[3], the multi-GPU part: ONE 8M-point synthetic cloud partitioned into x-slabs over the ranks
    (rank r holds the r-th x-quantile of the points, input order kept), filtered by the library's own NCCL protocol
    (csrc/slab.cpp: cwipc_cuda_slab_downsample / _remove_outliers).  All ranks take part; device time of the slowest rank
    (CUDA events on every rank's stream around the collective call, MAX over ranks), median of 3 after 1 warm-up.  The
    downsample result is checked against ONE GPU on the concatenation of the parts: same records, bit for bit."""
    from cwipc_util_b200 import synthetic, util
    lib = util.cwipc_util_dll_load()
    n_req = 2828 * 2828
    pts = synthetic.simulate_cameras(synthetic.synthetic_cloud(n_req), 4)
    n_all = len(pts)
    edges = np.quantile(pts["x"], np.linspace(0, 1, world + 1))
    edges[0], edges[-1] = -np.inf, np.inf
    slab_of = np.clip(np.searchsorted(edges, pts["x"], side="right") - 1, 0, world - 1)
    part = pts[slab_of == rank]
    whole = pts[np.argsort(slab_of, kind="stable")] if rank == 0 else None   # the parts in rank order
    del pts
    uid = None
    if world > 1:
        t = torch.zeros(128, dtype=torch.uint8, device="cuda")
        if rank == 0:
            t = torch.frombuffer(bytearray(util.cuda_comm.unique_id()), dtype=torch.uint8).clone().cuda()
        dist.broadcast(t, src=0)
        uid = bytes(t.cpu().numpy().tobytes())
    comm = util.cuda_comm(uid, world, rank)
    pc = cw.cwipc_from_numpy_array(part, 3)
    pc._set_cellsize(synthetic.cellsize_of(n_req))

    def timed(fn, reps=3, warm=1):
        times, res = [], None
        for i in range(reps + warm):
            lib.cwipc_cuda_flush_l2()
            cw.cuda_synchronize()
            dist_barrier(dist, torch)
            tm = lib.cwipc_cuda_timer_create()
            lib.cwipc_cuda_timer_start(tm)
            res = fn()
            lib.cwipc_cuda_timer_stop(tm)
            cw.cuda_synchronize()
            ms = dist_reduce(dist, torch, lib.cwipc_cuda_timer_elapsed_ms(tm), "MAX")
            lib.cwipc_cuda_timer_destroy(tm)
            if i >= warm:
                times.append(ms)
        return float(np.median(times)), res

    def digest(records):
        """order-independent digest of 16-byte records: sum of mixed words modulo 2^61"""
        w = np.ascontiguousarray(records).view(np.uint64).reshape(-1, 2)
        h = (w[:, 0] * np.uint64(0x9E3779B97F4A7C15) ^ (w[:, 1] + np.uint64(0xC2B2AE3D27D4EB4F))) * np.uint64(0x165667B19E3779F9)
        return int(h.sum(dtype=np.uint64)) & ((1 << 61) - 1) if len(h) else 0

    out = {"what": "configs[3]: one 8M-point synthetic cloud as x-slabs over the ranks, library NCCL protocol (ncclSend/ncclRecv of device buffers), "
                   "max over ranks of the CUDA-event time around the collective call", "points": n_all, "ranks": world, "rows": []}
    ds005 = None
    for vs in (0.002, 0.005, 0.01, 0.02, 0.05):
        ms, d = timed(lambda: comm.downsample(pc, vs))
        v = int(dist_reduce(dist, torch, d.count(), "SUM"))
        out["rows"].append({"op": "downsample", "voxelsize": vs, "voxels": v, "ms": round(ms, 4), "Mpoints_per_s": round(n_all / ms / 1e3, 1)})
        if vs == 0.005:
            ds005 = d
    # bit-identity with one GPU: digests of the ranks' pieces add up (mod 2^61) to the digest of the single-GPU result
    local = digest(ds005.get_numpy_array())
    if dist is not None:
        parts = [torch.zeros(1, dtype=torch.int64, device="cuda") for _ in range(world)]
        dist.all_gather(parts, torch.tensor([local], dtype=torch.int64, device="cuda"))
        total = sum(int(p.item()) for p in parts) & ((1 << 61) - 1)
    else:
        total = local
    if rank == 0:
        whole_pc = cw.cwipc_from_numpy_array(whole, 3)
        whole_pc._set_cellsize(synthetic.cellsize_of(n_req))
        single = cw.cwipc_downsample(whole_pc, 0.005)
        v_slabs = [r["voxels"] for r in out["rows"] if r["voxelsize"] == 0.005][0]
        out["downsample_0.005_vs_one_gpu"] = {"voxels_one_gpu": single.count(), "voxels_slabs": v_slabs,
                                              "records_identical": bool(single.count() == v_slabs and digest(single.get_numpy_array()) == total)}
        single.free()
        whole_pc.free()
    ms, o = timed(lambda: comm.remove_outliers(ds005, K, STDDEV, False))
    m_in = int(dist_reduce(dist, torch, ds005.count(), "SUM"))
    out["rows"].append({"op": "remove_outliers of the downsample(0.005) result", "points": m_in, "kept": int(dist_reduce(dist, torch, o.count(), "SUM")), "ms": round(ms, 4),
                        "Mpoints_per_s": round(m_in / ms / 1e3, 1)})
    # (three warm-ups: the first calls at this size grow the library's memory pool by several hundred MB)
    ms, o = timed(lambda: comm.remove_outliers(pc, K, STDDEV, False), reps=3, warm=3)
    out["rows"].append({"op": "remove_outliers of the raw cloud", "points": n_all, "kept": int(dist_reduce(dist, torch, o.count(), "SUM")), "ms": round(ms, 4),
                        "Mpoints_per_s": round(n_all / ms / 1e3, 1)})
    comm.free()
    return out


def run_ours(args):
    # stdout carries exactly ONE JSON line: everything else that libraries print there (e.g. NCCL's version banner)
    # is sent to stderr by pointing fd 1 at fd 2 for the duration of the run
    sys.stdout.flush()
    json_fd = os.dup(1)
    os.dup2(2, 1)
    world, rank, local, dist, torch = dist_setup(args)
    # Host threads: each worker spends most of its time waiting for a count readback; the library polls briefly and
    # then naps between polls (csrc/runtime.cu: stream_sync), so many threads per GPU also work on few cores per GPU.
    cores = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    if args.workers <= 0:
        args.workers = WORKERS if cores >= world * 16 else 15   # 30 threads with 16 cores or more per rank, else 15
        if cores < world * 8:
            # e.g. 8 ranks on a 32-core node: fewer, lazier waiters (measured at 8 GPUs: 10 threads napping 60 us
            # gave 42.6 Gpoints/s, 15 napping 20 us 39.7, 10 polling 36.5)
            args.workers = 10
            os.environ.setdefault("CWIPC_CUDA_SPIN_US", "10")
            os.environ.setdefault("CWIPC_CUDA_SLEEP_US", "60")
    import cwipc_util_b200 as cw
    from cwipc_util_b200 import synthetic
    lib = cw.util.cwipc_util_dll_load()
    if cw.cuda_device_count() <= 0:
        raise SystemExit("bench.py: libcwipc_util_cuda sees no CUDA device (there is no CPU fallback)")
    dev = local if cw.cuda_device_count() > local else 0
    cw.cuda_set_device(dev)
    # frame f of the 240-frame sequence goes to GPU f mod N (strong scaling); --frames-per-gpu overrides for diagnostics
    nframes = args.frames_per_gpu if args.frames_per_gpu > 0 else len(range(rank, args.sequence_frames, world))
    cellsize = synthetic.cellsize_of(POINTS_PER_FRAME)

    t0 = time.perf_counter()
    frames = make_frames(rank, nframes, world)          # frame f of the sequence goes to GPU f mod N
    log(f"[rank {rank}] generated {nframes} frames in {time.perf_counter() - t0:.1f}s")

    # device-resident copies (for `value`) and page-locked host copies (for `e2e`)
    device_frames, host_ptrs = [], []
    for f, pts in enumerate(frames):
        pc = cw.cwipc_from_numpy_array(pts, f)
        pc._set_cellsize(cellsize)
        device_frames.append(pc)
        hp = lib.cwipc_cuda_host_alloc(POINTS_PER_FRAME * 16)
        ctypes.memmove(hp, pts.ctypes.data, POINTS_PER_FRAME * 16)
        host_ptrs.append(hp)
    if os.environ.get("BENCH_STAGE", "") == "outliers":
        state_mid = [cw.cwipc_downsample(pc, VOXEL) for pc in device_frames]
    else:
        state_mid = []
    nworkers = args.workers
    host_out = [lib.cwipc_cuda_host_alloc(POINTS_PER_FRAME * 16) for _ in range(nworkers)]
    state = {"frames": frames, "device_frames": device_frames, "host_ptrs": host_ptrs, "host_out": host_out, "cellsize": cellsize, "stop": False, "mode": "resident", "mid_frames": state_mid,
             "keep": None}
    barrier = threading.Barrier(nworkers + 1)
    workers = [Worker(w, nworkers, dev, cw, lib, barrier, state) for w in range(nworkers)]
    for w in workers:
        w.start()

    # ---- warm-up (both paths), then the timed regions ----
    sampler = ClockSampler(dev)
    sampler.start()
    sampler.ready.wait(timeout=30)
    run_steps(workers, barrier, state, lib, "resident", args.warmup)
    run_steps(workers, barrier, state, lib, "e2e", max(1, args.warmup // 2), passes=1)
    cw.cuda_synchronize()
    dist_barrier(dist, torch)

    if args.dump_outputs:
        state["keep"] = set(np.random.default_rng(0).choice(nframes, min(DUMP_FRAMES, nframes), replace=False).tolist())
    sampler.armed.set()
    launches0 = cw.cuda_kernel_launches()
    resident_ms = run_steps(workers, barrier, state, lib, "resident", args.steps)
    launches = cw.cuda_kernel_launches() - launches0
    out_points = sum(w.out_points for w in workers) // args.steps      # per step
    mid_points = sum(w.mid_points for w in workers) // args.steps
    state["keep"] = None
    dist_barrier(dist, torch)
    e2e_ms = run_steps(workers, barrier, state, lib, "e2e", args.steps)
    d2h_bytes = sum(w.d2h_bytes for w in workers)
    sampler.armed.clear()
    clocks = sampler.stop()
    dist_barrier(dist, torch)
    # the path an UNCHANGED reference caller takes: cwipc_from_points from its own pageable memory (python/cwipc/util.py
    # passes ctypes / numpy buffers), one step of one pass
    run_steps(workers, barrier, state, lib, "e2e_pageable", 1, passes=1)     # warm-up: every thread's staging ring gets allocated here
    pageable_ms = run_steps(workers, barrier, state, lib, "e2e_pageable", 1, passes=1)
    dist_barrier(dist, torch)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, workers, rank, world)

    # ---- roofline: the same frames once more on ONE stream with events around every launch, so that the
    # per-kernel durations are not inflated by the other streams' kernels sharing the SMs ----
    state["stop"] = True
    barrier.wait()
    prof = {}
    if rank == 0:
        nprof = min(nframes, 12)
        for f in range(2):                                # warm the main thread's stream, pools and workspace
            o = workers[0].frame_chain(device_frames[f])
            o.free()
        cw.cuda_synchronize()
        lib.cwipc_cuda_profile_reset()
        lib.cwipc_cuda_profile_enable(1)
        for f in range(nprof):
            o = workers[0].frame_chain(device_frames[f])
            o.free()
        cw.cuda_synchronize()
        lib.cwipc_cuda_profile_enable(0)
        need = lib.cwipc_cuda_profile_report(None, 0)
        buf = ctypes.create_string_buffer(need)
        lib.cwipc_cuda_profile_report(buf, need)
        prof = json.loads(buf.value.decode())

    # ---- aggregate over ranks: time = max over ranks, work = sum ----
    total_ms = dist_reduce(dist, torch, resident_ms, "MAX")
    total_e2e_ms = dist_reduce(dist, torch, e2e_ms, "MAX")
    launches_all = dist_reduce(dist, torch, launches, "SUM")
    d2h_all = dist_reduce(dist, torch, d2h_bytes, "SUM")
    total_pageable_ms = dist_reduce(dist, torch, pageable_ms, "MAX")
    frames_all = int(dist_reduce(dist, torch, nframes, "SUM"))            # the whole sequence
    points_per_step = frames_all * PASSES * POINTS_PER_FRAME
    value = points_per_step * args.steps / (total_ms / 1e3) / 1e6
    e2e_value = points_per_step * args.steps / (total_e2e_ms / 1e3) / 1e6
    pageable_value = frames_all * POINTS_PER_FRAME / (total_pageable_ms / 1e3) / 1e6

    slab = measure_slab(cw, dist, torch, rank, world) if not args.skip_config4 else None   # every rank takes part
    if rank != 0:
        dist_barrier(dist, torch)      # rank 0 times the single-GPU part of configs[3] meanwhile
        return
    peak, peak_src = measured_hbm_peak()
    config4 = measure_config4(cw, lib, peak) if not args.skip_config4 else None
    if config4 is not None:
        config4["slabs"] = slab
    dist_barrier(dist, torch)
    roofline = None
    if prof:
        name, rec = max(prof.items(), key=lambda kv: kv[1]["total_ms"])
        achieved = rec["bytes"] / (rec["total_ms"] / 1e3) / 1e9 if rec["total_ms"] > 0 else 0.0
        traffic, issue = None, None
        try:
            tj = json.load(open(os.path.join(REPO, "profiles", "traffic.json")))
            traffic = tj.get(name)
            winst = tj.get("_warp_instructions", {}).get(name)
            if winst and rec["total_ms"] > 0:
                # instruction-issue roofline of the same launches: warp instructions per launch (ncu smsp__inst_executed.sum)
                # over the measured launch time, against 148 SMs x 4 schedulers x 1 instruction per clock at the max SM clock
                per_s = winst / (rec["total_ms"] / 1e3 / max(1, rec["launches"]))
                peak_issue = 148 * 4 * 1.965e9
                issue = {"warp_inst_per_launch": winst, "achieved_Ginst_per_s": round(per_s / 1e9, 1), "peak_Ginst_per_s": round(peak_issue / 1e9, 1),
                         "frac": round(per_s / peak_issue, 4)}
        except Exception:
            pass
        step_kernel_ms = sum(r["total_ms"] for r in prof.values())
        kernels = {}
        for k, v in sorted(prof.items(), key=lambda kv: -kv[1]["total_ms"]):
            gbs = v["bytes"] / max(v["total_ms"], 1e-9) / 1e6
            kernels[k] = {"launches_per_frame": round(v["launches"] / nprof, 2), "us_per_launch": round(v["total_ms"] * 1e3 / max(1, v["launches"]), 2),
                          "GBps": round(gbs, 1), "frac": round(gbs / peak, 4), "share": round(v["total_ms"] / step_kernel_ms, 3)}
        roofline = {"bound": "hbm", "kernel": name, "achieved": round(achieved, 1), "peak": peak, "unit": "GB/s", "frac": round(achieved / peak, 4),
                    "traffic": traffic, "traffic_source": "static: dram__bytes_read.sum + dram__bytes_write.sum per launch from the latest ncu --set full capture (profiles/traffic.json), not measured in this run",
                    "issue": issue, "peak_source": peak_src, "launches": rec["launches"], "avg_launch_us": round(rec["total_ms"] * 1e3 / max(1, rec["launches"]), 2),
                    "algorithmic_bytes_per_launch": int(rec["bytes"] / max(1, rec["launches"])), "share_of_step_kernel_time": round(rec["total_ms"] / step_kernel_ms, 3),
                    "how": f"{nprof} of the step's frames replayed on one stream, CUDA events around every launch (cwipc_cuda_profile_*)",
                    "note": "the kNN kernels are instruction-issue bound (exact top-(k+1) selection over ~300 candidates per query), not HBM bound: "
                            "their HBM fraction is reported as required, their issue utilisation is in profiles/",
                    "kernels": kernels}
        # whole-op roofline on compulsory bytes (SURVEY.md §8d): 16 B in + 16 B out per stage
        # downsample: 16 N in + 16 V out; remove_outliers: 16 V in + 16 M out   (per rank and step)
        compulsory = 16.0 * (nframes * PASSES * POINTS_PER_FRAME + 2 * mid_points + out_points)
        roofline["op_compulsory_GBps_per_gpu"] = round(compulsory / (resident_ms / args.steps / 1e3) / 1e9, 1)
        roofline["op_compulsory_frac"] = round(roofline["op_compulsory_GBps_per_gpu"] / peak, 4)

    cpu_mpts, cpu_dt = cpu_baseline_sample(frames, args.cpu_frames)
    line = {
        "metric": "Mpoints/s for downsample+remove_outliers at 1/2/4/8 B200; % of HBM GB/s peak",
        "value": round(value, 1), "unit": "Mpoints/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": round(total_ms / args.steps, 3), "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "f32 keys/distances, int64 fixed-point sums, f64 statistics", "data": "synthetic",
        "config": {"workload": f"configs[4]: {frames_all}-frame sequence of 1M-point 4-camera synthetic frames, per frame cwipc_downsample(0.01) -> cwipc_remove_outliers(30,1.0,perTile=False); "
                               f"frame f on GPU f mod N (strong scaling: the same {frames_all} frames at every N), no collective; a step = {PASSES} passes over the sequence",
                   "points_per_frame": POINTS_PER_FRAME, "sequence_frames": frames_all, "passes_per_step": PASSES, "frames_per_gpu": nframes,
                   "host_threads_per_gpu": nworkers, "host_cores": cores, "host_wait": "poll %s us then nap %s us" % (os.environ.get("CWIPC_CUDA_SPIN_US", "20"), os.environ.get("CWIPC_CUDA_SLEEP_US", "20")),
                   "l2": f"inputs larger than L2 ({nframes} x 16 MB per GPU per pass, each frame touched once per pass)",
                   "parallelism": f"frames x{world}"},
        "e2e": {"value": round(e2e_value, 1), "unit": "Mpoints/s", "h2d_bytes_per_step": points_per_step * 16, "d2h_bytes_per_step": int(d2h_all / max(1, args.steps)),
                "ms_per_step": round(total_e2e_ms / args.steps, 3), "host_memory": "page-locked (cwipc_cuda_host_alloc)",
                "pageable": {"value": round(pageable_value, 1), "unit": "Mpoints/s", "what": "the same chain with cwipc_from_points reading the caller's pageable numpy memory, as an unchanged "
                             "python/cwipc/util.py caller supplies it; one pass over the sequence", "ms": round(total_pageable_ms, 3)}},
        "config4": config4,
        "gpu_launches": int(launches_all),
        "clocks": clocks,
        "roofline": roofline,
        "cpu_baseline": {"value": round(cpu_mpts, 3), "unit": "Mpoints/s", "cores": 1, "kind": "port",
                         "sample": f"{args.cpu_frames} of the same frames through oracle/cwipc_oracle.c (downsample 0.01 + remove_outliers 30/1.0), {cpu_dt:.1f}s, single thread"},
        "out_points_per_step": int(out_points),
        "timed_region_ms": round(total_ms, 3), "e2e_timed_region_ms": round(total_e2e_ms, 3),
    }
    sys.stdout.flush()
    os.write(json_fd, (json.dumps(line) + "\n").encode())


# --------------------------------------------------------------------------------------------------
# reference arm: the reference's CPU path (oracle port: the reference itself needs PCL and cannot be built here)
# --------------------------------------------------------------------------------------------------
def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if rank != 0:
        return  # rank 0 alone runs the CPU arm
    sys.path.insert(0, os.path.join(REPO, "oracle"))
    import oracle
    from cwipc_util_b200 import synthetic
    oracle.load()
    cores = os.cpu_count() or 1
    nthreads = max(1, cores)
    per_step = nthreads  # one frame per host thread per step: a bounded sample of the 8 x 240-frame step
    frames = make_frames(0, min(per_step, 16), 1)
    cellsize = synthetic.cellsize_of(POINTS_PER_FRAME)

    def one(i):
        pts = frames[i % len(frames)]
        ds, cs, _, _ = oracle.downsample(pts, VOXEL, cellsize)
        oracle.remove_outliers(ds, K, STDDEV, False)

    from concurrent.futures import ThreadPoolExecutor
    with ThreadPoolExecutor(nthreads) as ex:
        for _ in range(args.warmup):
            list(ex.map(one, range(per_step)))
        t0 = time.perf_counter()
        for _ in range(args.steps):
            list(ex.map(one, range(per_step)))   # ctypes releases the GIL: frames run on all cores
        dt = time.perf_counter() - t0
    value = per_step * args.steps * POINTS_PER_FRAME / dt / 1e6
    line = {
        "impl": "reference",
        "metric": "Mpoints/s for downsample+remove_outliers at 1/2/4/8 B200; % of HBM GB/s peak",
        "value": round(value, 3), "unit": "Mpoints/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": round(dt / args.steps * 1e3, 3), "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "f32/f64 (CPU)", "data": "synthetic",
        "config": {"workload": "configs[4]: 1M-point 4-camera synthetic frames, per frame cwipc_downsample(0.01) -> cwipc_remove_outliers(30,1.0,perTile=False)",
                   "points_per_frame": POINTS_PER_FRAME, "frames_per_step": per_step, "parallelism": f"{nthreads} host threads, one frame each"},
        "cpu_baseline": {"value": round(value, 3), "unit": "Mpoints/s", "cores": nthreads, "kind": "port",
                         "sample": f"{per_step} frames per step (one per host thread) through oracle/cwipc_oracle.c; the reference itself needs PCL and cannot be built here"},
        "e2e": {"value": round(value, 3), "unit": "Mpoints/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


def main():
    global PASSES
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--sequence-frames", type=int, default=SEQUENCE_FRAMES)
    ap.add_argument("--frames-per-gpu", type=int, default=0, help="diagnostics: this many frames on every GPU instead of its share of the sequence")
    ap.add_argument("--skip-config4", action="store_true", help="diagnostics: leave out the 8M-point configs[3] measurement")
    ap.add_argument("--passes", type=int, default=PASSES, help="diagnostics: passes over the sequence per step (the contract value is 8)")
    ap.add_argument("--workers", type=int, default=0, help="host threads per GPU (0 = choose from the core count)")
    ap.add_argument("--cpu-frames", type=int, default=24)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the timed path returned in its last step to DIR/*.npy (float32/float64, at most 64 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the results of our arm (--impl ours)")
    if args.dump_outputs:
        os.makedirs(args.dump_outputs, exist_ok=True)
    PASSES = max(1, args.passes)
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
