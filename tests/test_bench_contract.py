"""bench.py's bookkeeping, checked on the CPU: the roofline numerator is SURVEY 8d's algorithmic FLOP count, the
workloads are BASELINE.json's configurations, the reference arm prints the contract's keys (it runs the oracle
port on the host cores; no GPU involved) and --dump-outputs keeps to its budget; on the GPU, --dump-outputs end to
end."""
import importlib.util
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench():
    spec = importlib.util.spec_from_file_location("bench_module", os.path.join(ROOT, "bench.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def test_algorithmic_flops_are_the_surveys():
    """SURVEY 8d: F = 2 (n M_e + M_s); EB-CADRL net 245,300 MAC per entity + 132,000 per state -> 8.11 MFLOP at n = 16,
    14.98 at n = 30; SARL baseline 62,050 + 33,500 -> 0.6875 MFLOP at n = 5 (a17)."""
    b = _bench()
    eb, _ = b.value_net_weights(fixture="weights_ebcadrl.npz")
    sarl, _ = b.value_net_weights(fixture="weights_sarl_baseline.npz")
    assert b.flops_per_eval(eb, 16) == 2 * (16 * 245300 + 132000) == 8113600
    assert b.flops_per_eval(eb, 30) == 2 * (30 * 245300 + 132000)
    assert b.flops_per_eval(sarl, 5) == 2 * (5 * 62050 + 33500) == 687500


def test_workloads_are_the_baseline_configs():
    b = _bench()
    shape, cfg = b.workload("cfg2")                       # BASELINE configs[1]: 10 typed humans + 3 walls, 4096 episodes
    assert (shape.H, shape.Smax, b.WORKLOADS["cfg2"][4], cfg.with_agent_type, cfg.robot_kinematics) == (10, 6, 4096, True, "holonomic")
    shape, cfg = b.workload("cfg3")                       # configs[2]: unicycle robot, 16,384 episodes
    assert (shape.H, shape.Smax, b.WORKLOADS["cfg3"][4], cfg.robot_kinematics) == (5, 0, 16384, "unicycle")
    shape, cfg = b.workload("cfg4")                       # configs[3]: 20 humans + 10 walls, 8,192 episodes per GPU
    assert (shape.H, shape.num_walls, b.WORKLOADS["cfg4"][4]) == (20, 10, 8192)
    base = json.load(open(os.path.join(ROOT, "BASELINE.json")))
    assert len(base["configs"]) == 5 and "4096" in base["configs"][1] and "16384" in base["configs"][2]
    peaks = b.measured_peaks()
    assert peaks["hbm_gbs"] > 0 and peaks["tensor_tflops"] > 0


def test_reference_arm_prints_the_contract_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                         capture_output=True, text=True, timeout=600, env=dict(os.environ, RANK="0", WORLD_SIZE="1"))
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads([l for l in out.stdout.splitlines() if l.startswith("{")][-1])
    assert line["impl"] == "reference" and line["metric"] == "agent_steps_per_sec" and line["higher_is_better"] is True
    assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["cores"] == (os.cpu_count() or 1)
    assert line["e2e"] == {"value": line["value"], "unit": line["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert line["config"]["workload"] == "cfg2_h10_typed_3walls" and line["value"] > 0
    # rank > 0 of a torchrun launch exits 0 without work
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                         capture_output=True, text=True, timeout=120, env=dict(os.environ, RANK="1", WORLD_SIZE="2"))
    assert out.returncode == 0 and not [l for l in out.stdout.splitlines() if l.startswith("{")]


def test_dump_outputs_keeps_the_same_rows_within_the_budget(tmp_path):
    b = _bench()
    rng = np.random.default_rng(1)
    n = 1000
    arrays = {"values": rng.random((n, 81), dtype=np.float32), "reward": rng.random(n),
              "argmax": rng.integers(0, 81, n, dtype=np.int32), "done": (rng.random(n) < 0.1).astype(np.uint8)}

    def written(d):
        return {f[:-4]: np.load(os.path.join(d, f)) for f in os.listdir(d)}

    b.dump_outputs(str(tmp_path / "whole"), arrays)
    whole = written(str(tmp_path / "whole"))
    assert set(whole) == set(arrays) | {"episode_index"}
    assert all(v.dtype in (np.float32, np.float64) for v in whole.values())
    assert np.array_equal(whole["episode_index"], np.arange(n))
    for k, v in arrays.items():
        assert np.array_equal(whole[k], v) and whole[k].dtype == (v.dtype if k in ("values", "reward") else np.float64)

    budget = 100_000
    for name in ("a", "b"):
        b.dump_outputs(str(tmp_path / name), arrays, budget=budget)
    a, a2 = written(str(tmp_path / "a")), written(str(tmp_path / "b"))
    assert sum(os.path.getsize(str(tmp_path / "a" / f)) for f in os.listdir(str(tmp_path / "a"))) <= budget
    idx = a["episode_index"].astype(np.int64)
    assert 0 < len(idx) < n and np.all(np.diff(idx) > 0)
    for k, v in arrays.items():
        assert np.array_equal(a[k], v[idx]) and np.array_equal(a[k], a2[k])


@pytest.mark.gpu
def test_dump_outputs_repeat_and_follow_steps(tmp_path):
    """The same arguments dump the same outputs bit for bit; one more timed step dumps a later state."""
    b = _bench()

    def run(steps, name):
        d = str(tmp_path / name)
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--episodes", "512", "--steps", str(steps),
                              "--warmup", "3", "--no-cpu-baseline", "--sustained-seconds", "0", "--dump-outputs", d],
                             capture_output=True, text=True, timeout=600, env=dict(os.environ, RANK="0", WORLD_SIZE="1"))
        assert out.returncode == 0, out.stderr[-2000:]
        assert json.loads([l for l in out.stdout.splitlines() if l.startswith("{")][-1])["steps"] == steps
        return {f[:-4]: np.load(os.path.join(d, f)) for f in os.listdir(d)}

    first, again, later = run(2, "first"), run(2, "again"), run(3, "later")
    assert set(first) == set(b.DUMPED) | {"episode_index"}
    assert first["values"].shape == (512, 81) and np.array_equal(first["episode_index"], np.arange(512))
    for k, v in first.items():
        assert v.dtype in (np.float32, np.float64) and np.isfinite(v).all(), k
        assert np.array_equal(v, again[k]), k
    assert not np.array_equal(first["hum_pv"], later["hum_pv"])
