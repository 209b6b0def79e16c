"""The bench line the driver parses: one JSON object on the last stdout line with the keys of the measurement contract
(metric / value / roofline / e2e / gpu_launches / clocks), produced by a short run of the real bench on a small batch."""
import json
import os
import subprocess
import sys

import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _dumped(out_dir):
    import numpy as np
    arrays = {f[:-4]: np.load(os.path.join(out_dir, f)) for f in os.listdir(out_dir)}
    assert all(a.dtype in (np.float32, np.float64) for a in arrays.values())
    assert sum(a.nbytes for a in arrays.values()) <= 64_000_000
    return arrays


def test_bench_line_has_the_contract_keys(tmp_path):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "8", "--warmup", "3", "--envs-per-gpu", "4096",
                          "--no-cpu-baseline", "--no-ppo", "--dump-outputs", str(tmp_path)], capture_output=True, text=True,
                         timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.strip().splitlines() if l.startswith("{")]
    assert len(lines) == 1, "exactly one JSON line"
    d = json.loads(lines[0])
    for key in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
                "dtype", "data", "config", "roofline", "e2e", "gpu_launches", "clocks"):
        assert key in d, key
    assert d["n_gpus"] == 1 and d["steps"] == 8 and d["warmup"] == 3 and d["higher_is_better"] is True and d["scaling"] == "weak"
    assert d["vs_baseline"] is None and d["data"] == "synthetic" and d["gpu_launches"] == 8 and "workload" in d["config"]
    assert d["value"] > 0 and abs(d["value"] - 4096 / (d["ms_per_step"] * 1e-3)) < 1e-6 * d["value"]
    r = d["roofline"]
    assert r["bound"] == "hbm" and r["unit"] == "GB/s" and r["peak"] > 0 and abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-9
    e = d["e2e"]
    assert e["value"] > 0 and e["h2d_bytes_per_step"] == 4096 and e["d2h_bytes_per_step"] == 4096 * 5
    assert e["with_obs"]["d2h_bytes_per_step"] == 4096 * (5 + 5 * 14 * 4)
    assert set(d["clocks"]) >= {"sm_mhz", "sm_max_mhz", "reasons"}
    # --dump-outputs: the last timed step's (obs, reward, done, info), one row per env
    arrays = _dumped(tmp_path)
    assert arrays["obs"].shape == (4096, 5, 14) and arrays["reward_f64"].dtype.name == "float64"
    assert {"reward", "done", "J_val", "num_assigned", "is_valid_action", "avg_p_dmg", "avg_p_final", "env_id"} <= set(arrays)
    assert all(len(a) == 4096 for a in arrays.values())
    assert abs(arrays["reward"] - arrays["reward_f64"]).max() <= 1e-5 * max(1.0, abs(arrays["reward_f64"]).max())


def test_ppo_bench_times_exactly_the_requested_iterations(tmp_path):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "c4", "--steps", "2", "--warmup", "3",
                          "--envs-per-gpu", "1024", "--dump-outputs", str(tmp_path)], capture_output=True, text=True,
                         timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    d = json.loads(out.stdout.strip().splitlines()[-1])
    assert d["metric"] == "ppo_samples_per_sec" and d["steps"] == 2
    arrays = _dumped(tmp_path)
    assert {"loss_actor", "loss_critic", "entropy"} <= set(arrays) and arrays["policy_params"].shape == (419267,)
