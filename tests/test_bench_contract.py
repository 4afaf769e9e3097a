"""bench.py prints ONE JSON line with the keys the driver reads (CPU: the reference arm; GPU: the native arm)."""
import json
import os
import subprocess
import sys

import pytest

from conftest import REPO

BASE_KEYS = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
             "vs_baseline", "dtype", "data", "config", "e2e", "gpu_launches"}


def _run(*args):
    out = subprocess.run([sys.executable, "bench.py", *args], cwd=REPO, capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-1500:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, out.stdout[-500:]
    return json.loads(lines[0])


def test_reference_arm_line():
    d = _run("--impl", "reference", "--steps", "3", "--warmup", "3", "--workload", "cfg5")
    assert d["impl"] == "reference" and BASE_KEYS <= d.keys()
    assert d["value"] > 0 and d["unit"] == "env-steps/s" and d["higher_is_better"] is True and d["vs_baseline"] is None
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["config"]["workload"] == "cfg5" and d["gpu_launches"] == 0


@pytest.mark.gpu
def test_native_arm_line():
    d = _run("--steps", "30", "--warmup", "3", "--workload", "cfg2", "--no-extra")
    assert BASE_KEYS | {"roofline", "cpu_baseline", "clocks"} <= d.keys() and "impl" not in d
    # a 65,536-env shard: the 30 bound steps of the gc_step_many call run inside one kernel, and the same loop is
    # reported with one launch per step beside it
    if os.environ.get("GC_B200_STEP_MANY_FUSED", "1")[:1] == "0":
        pytest.skip("the one-launch path is switched off in this environment")
    assert d["gpu_launches"] == 1 and d["steps_per_launch"] == 30 and d["separate_launches"]["gpu_launches"] == 30
    assert 0 < d["separate_launches"]["value"] < d["value"] and d["episode_stats"]["consistent"]
    assert d["n_gpus"] == 1 and d["scaling"] == "weak" and d["data"] == "synthetic"
    r = d["roofline"]
    assert r["bound"] == "hbm" and r["unit"] == "GB/s" and abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-9
    # (the many-step kernel reads state and t once per launch: 29 - 7 bytes per env-step)
    assert r["bytes_per_env_step"] == 22.0 and r["algorithmic_bytes_per_step"] == 22 * 65536
    assert r["algorithmic_bytes_per_launch"] == 30 * 22 * 65536
    e = d["e2e"]
    assert e["h2d_bytes_per_step"] == 4 * 65536 and e["d2h_bytes_per_step"] == 13 * 65536 and 0 < e["value"] < d["value"]
    assert d["clocks"]["sm_max_mhz"] and not {"hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown"} & set(d["clocks"]["reasons"])
    assert d["cpu_baseline"]["kind"] == "port" and d["config"]["workload"] == "cfg2"


@pytest.mark.gpu
def test_dump_outputs_hold_the_last_timed_step(tmp_path):
    """--dump-outputs writes what the timed path computed in its last step, as float arrays: on cfg2 (65,536 envs,
    all of them in the sample) it equals the oracle stepped through the warmup and timed steps of the bench's
    seeded action ring."""
    import numpy as np
    import torch
    import bench
    from oracle import oracle as O
    warmup, steps = 5, 30
    d = _run("--steps", str(steps), "--warmup", str(warmup), "--workload", "cfg2", "--no-extra", "--no-cpu-baseline",
             "--no-side", "--dump-outputs", str(tmp_path))
    assert d["steps"] == steps and d["warmup"] == warmup
    out = {p.stem: np.load(p) for p in tmp_path.glob("*.npy")}
    assert set(out) == {"cellular_" + k for k in ("env_ids", "state", "reward", "terminated", "truncated", "unsafe",
                                                   "count", "time_step", "tabular_state")}
    assert all(a.dtype in (np.float32, np.float64) for a in out.values())
    assert sum(p.stat().st_size for p in tmp_path.iterdir()) <= 64 << 20
    b, = bench.build_batches("cfg2", torch.device("cuda", 0), 0)
    n, ring = b["n"], [a[:, :b["n"]].cpu().numpy() for a in b["ring"]]
    b["env"].close()
    assert (out["cellular_env_ids"] == np.arange(n)).all()
    ora = O.OracleEnv(n_envs=n, seed=0)
    for i in range(warmup + steps):
        ora.step(ring[i % len(ring)])
    assert (out["cellular_state"] == ora.state).all() and (out["cellular_tabular_state"] == ora.index).all()
    assert (out["cellular_time_step"] == warmup + steps).all() and (out["cellular_time_step"] == ora.t).all()
    assert (out["cellular_unsafe"] == ora.unsafe).all() and (out["cellular_count"] == ora.count).all()
    assert not out["cellular_terminated"].any() and not out["cellular_truncated"].any()
    np.testing.assert_allclose(out["cellular_reward"], ora.reward, rtol=1e-6, atol=1e-7)
