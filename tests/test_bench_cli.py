"""bench.py on the CPU: the reference arm (the oracle on the host cores) prints exactly one JSON line with the keys
its readers use; our arm refuses to run without a GPU instead of falling back.  On the GPU: --dump-outputs writes what
the timed chain returns for the bench's own frames."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def run_bench(*args, **env):
    e = dict(os.environ, BENCH_POINTS="20000")
    e.update(env)
    return subprocess.run([sys.executable, os.path.join(REPO, "bench.py"), *args], capture_output=True, text=True, env=e, timeout=600)


def test_reference_arm_prints_one_json_line():
    r = run_bench("--impl", "reference", "--gpus", "1", "--steps", "2", "--warmup", "1")
    assert r.returncode == 0, r.stderr
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "Mpoints/s" and d["higher_is_better"] is True
    assert d["value"] > 0 and d["steps"] == 2 and d["n_gpus"] == 1
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "Mpoints/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"]


def test_reference_arm_other_ranks_exit_quietly():
    r = run_bench("--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "0", RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_our_arm_fails_loudly_without_a_gpu():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    r = run_bench("--steps", "1", "--warmup", "3")
    assert r.returncode != 0
    assert r.stdout.strip() == ""          # no JSON line that could be mistaken for a measurement
    assert "no CUDA device" in (r.stderr + r.stdout) or "CUDA" in r.stderr


def test_bad_arguments_are_refused():
    assert run_bench("--steps", "0").returncode == 2
    assert run_bench("--impl", "reference", "--dump-outputs", "unused").returncode == 2


@pytest.mark.gpu
def test_dump_outputs_are_what_the_chain_returns(cw, tmp_path):
    """Every frame's count and, for the sampled frames, the points of downsample(0.01) -> remove_outliers(30, 1.0) of
    that frame, recomputed here from the same seeds (at the bench's own frame size: smaller frames are coarser than the voxel)."""
    from cwipc_util_b200 import synthetic
    n, frames = 1000 * 1000, 4
    out = tmp_path / "dump"
    r = run_bench("--steps", "2", "--warmup", "3", "--frames-per-gpu", str(frames), "--passes", "2", "--workers", "2", "--cpu-frames", "1",
                  "--skip-config4", "--dump-outputs", str(out), BENCH_POINTS=str(n))
    assert r.returncode == 0, r.stderr[-3000:]
    assert json.loads(r.stdout)["steps"] == 2
    counts = np.load(out / "counts_rank0.npy")
    assert counts.dtype == np.float64 and counts.shape == (frames, 2) and list(counts[:, 0]) == list(range(frames))
    assert sorted(os.listdir(out)) == ["counts_rank0.npy"] + [f"frame{f:03d}.npy" for f in range(frames)]
    base = synthetic.simulate_cameras(synthetic.synthetic_cloud(n), 4)
    for f in range(frames):
        pc = cw.cwipc_from_numpy_array(synthetic.add_outliers(synthetic.add_noise(base, 0.002, f), 0.005, f), f)
        pc._set_cellsize(synthetic.cellsize_of(n))
        want = cw.cwipc_remove_outliers(cw.cwipc_downsample(pc, 0.01), 30, 1.0, False).get_numpy_array()
        got = np.load(out / f"frame{f:03d}.npy")
        assert got.dtype == np.float32 and counts[f, 1] == len(want) > 0
        assert np.array_equal(got, np.stack([want[c].astype(np.float32) for c in ("x", "y", "z", "r", "g", "b", "tile")], axis=1))
