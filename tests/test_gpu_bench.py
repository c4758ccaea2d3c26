"""bench.py on the GPU: the one-line JSON carries every key of the contract (structure only, no thresholds), and
--dump-outputs writes the same outputs on every run."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench(*args):
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + list(args), capture_output=True, text=True,
                         timeout=900, cwd=ROOT)
    assert res.returncode == 0, res.stderr[-3000:]
    lines = [l for l in res.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, res.stdout[-2000:]
    return json.loads(lines[0])


def _dumped(path):
    return {f[:-4]: np.load(os.path.join(path, f)) for f in sorted(os.listdir(path))}


def test_default_arm_json_contract(tmp_path):
    d = _bench("--steps", "6000", "--warmup", "3", "--mix", "100", "--no-cpu-baseline",
               "--dump-outputs", str(tmp_path / "out"))
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
              "vs_baseline", "dtype", "data", "config", "clocks", "e2e", "gpu_launches", "roofline", "cpu_baseline"):
        assert k in d, k
    assert d["n_gpus"] == 1 and d["steps"] == 6000 and d["scaling"] == "weak" and d["dtype"] == "u8"
    assert d["config"]["workload"].startswith("C2") and "model" not in d["config"]
    import argparse
    import bench
    assert d["config"] == bench.static_config(argparse.Namespace(workload="c2", envs_per_gpu=None, hardness="none"), 1)
    rs = d["run_stats"]
    # --steps 6000 times exactly 6,000 steps (~0.2 s): one region, its time over 6,000 is the reported step time
    assert rs["blocks"] == 1 and rs["timed_steps_total"] == 6000 and rs["timed_region_ms"] >= 150
    assert abs(rs["timed_region_ms"] / 6000 - d["ms_per_step"]) <= 1e-9 * d["ms_per_step"]
    assert abs(d["value"] - 4096 * 6000 / (rs["timed_region_ms"] * 1e-3)) <= 1e-6 * d["value"]
    assert d["gpu_launches"] == rs["launches_per_step"] * 6000 and d["value"] > 0
    assert d["clocks"]["samples"] >= 5
    r = d["roofline"]
    assert r["bound"] == "hbm" and r["unit"] == "GB/s" and abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-9
    assert r["traffic"] is None or (r["traffic"] > 0 and r["dram_frac"] > 0)
    e = d["e2e"]
    assert e["value"] > 0 and e["h2d_bytes_per_step"] == 4 * 4096 and e["d2h_bytes_per_step"] == 20 * 4096
    assert {"numpy_obs", "aux5_scaled_float", "aux5_uint8"} <= set(e["variants"])
    assert set(d["clocks"]) >= {"sm_mhz", "sm_max_mhz", "reasons"}
    assert {"rgb_only", "float_chw", "a2c_pass", "reference_run_config"} <= set(d["secondary"])
    # --dump-outputs: what the caller of the last timed step receives, a seeded row sample of the 4,096-env batch
    out = _dumped(tmp_path / "out")
    assert set(out) == {"obs_rgb", "obs_goal_rgb", "obs_depth", "last_action_reward", "reward", "done"}
    assert sum(os.path.getsize(tmp_path / "out" / (k + ".npy")) for k in out) <= 64_000_000
    assert all(a.dtype in (np.float32, np.float64) for a in out.values())
    rows = out["obs_rgb"].shape[0]
    assert 0 < rows < 4096 and out["obs_rgb"].shape[1:] == (84, 84, 3) and out["obs_depth"].shape[1:] == (84, 84, 1)
    assert out["obs_goal_rgb"].shape == out["obs_rgb"].shape and out["last_action_reward"].shape == (4096, 5)
    assert out["reward"].shape == out["done"].shape == (4096,) and set(np.unique(out["done"])) <= {0.0, 1.0}
    for k in ("obs_rgb", "obs_goal_rgb", "obs_depth"):
        assert out[k].min() >= 0 and out[k].max() <= 255 and np.array_equal(out[k], np.round(out[k])) and out[k].any()


@pytest.mark.parametrize("workload", ["c2", "c5"])
def test_dump_outputs_repeat_exactly(tmp_path, workload):
    """Two runs with the same arguments step the same envs through the same states: the dumped outputs are equal bit for
    bit, so two builds of the project can be compared output for output."""
    args = ["--workload", workload, "--steps", "7", "--warmup", "3"]
    args += ["--quick", "--mix", "50"] if workload == "c2" else []
    runs = []
    for k in range(2):
        assert _bench(*args, "--dump-outputs", str(tmp_path / str(k)))["value"] > 0
        runs.append(_dumped(tmp_path / str(k)))
    a, b = runs
    assert set(a) == set(b) and len(a) >= 5
    same = lambda x, y: x.dtype == y.dtype and x.shape == y.shape and x.tobytes() == y.tobytes()
    differ = [k for k in a if not same(a[k], b[k])]
    assert not differ, differ
