"""GPU: bench.py keeps its contract (one JSON line; metric / roofline / cpu_baseline / e2e / clocks / gpu_launches)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT

pytestmark = pytest.mark.gpu


def test_bench_line_contract_on_a_small_batch():
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "20", "--warmup", "3", "--envs", "8192", "--cpu-steps", "5", "--extra-steps", "10"],
                         capture_output=True, text=True, timeout=600)
    assert res.returncode == 0, res.stderr[-2000:]
    lines = [l for l in res.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, res.stdout
    d = json.loads(lines[0])
    assert d["metric"] == "BlueROV2 6DoF env-steps/sec" and d["unit"] == "env-steps/s" and d["higher_is_better"] is True
    assert d["n_gpus"] == 1 and d["steps"] == 20 and d["warmup"] == 3 and d["scaling"] == "weak" and d["vs_baseline"] is None
    assert d["dtype"] == "f32" and d["data"] == "synthetic" and "workload" in d["config"]
    assert d["value"] > 0 and d["gpu_launches"] == 20 * d["config"]["stream_groups"]
    assert d["config"]["stream_groups"] == 1 and d["single_launch_per_step"]["value"] > 0    # batches this small are not split
    r = d["roofline"]
    assert r["unit"] == "TFLOP/s" and abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-9 and r["hbm"]["unit"] == "GB/s"
    assert r["executed_frac"] < r["frac"]
    c = d["cpu_baseline"]
    assert c["kind"] == "port" and c["cores"] >= 1 and c["value"] > 0
    e = d["e2e"]
    assert e["value"] > 0 and e["h2d_bytes_per_step"] == 8192 * 8 * 4 and e["d2h_bytes_per_step"] == 8192 * (9 * 4 + 1)
    assert "sm_mhz" in d["clocks"] and "reasons" in d["clocks"]
    assert c["as_shipped_rk45_pid_port_one_core"] > 0 and c["legacy_auv_step_port_one_core"] > 0
    r5 = d["extra"]["config5_rollout"]   # config 5 rides along at every N
    assert r5["value"] > 0 and 0 < r5["env_share"] < 1
    assert r["executed_flop_per_env_step"] > 0
    assert r5["two_stream_groups"]["value"] > 0 and r5["two_stream_groups"]["launches_per_step"] == 4


def test_bench_line_with_stream_groups():
    """--stream-groups G: the environments of a rank as G independent blocks (vec_tools.EnvBlocks); G launches per step."""
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "20", "--warmup", "3", "--envs", "65536", "--stream-groups", "2",
                          "--no-cpu", "--no-extra"], capture_output=True, text=True, timeout=600)
    assert res.returncode == 0, res.stderr[-2000:]
    d = json.loads([l for l in res.stdout.splitlines() if l.strip()][-1])
    assert d["config"]["stream_groups"] == 2 and d["gpu_launches"] == 40 and d["value"] > 0 and d["steps"] == 20
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "20", "--warmup", "3", "--envs", "131072", "--no-cpu", "--no-extra"],
                         capture_output=True, text=True, timeout=600)
    assert res.returncode == 0, res.stderr[-2000:]
    d = json.loads([l for l in res.stdout.splitlines() if l.strip()][-1])
    tried = d["config"]["stream_groups_tried_ms_per_step"]                                    # default: calibrated choice
    assert set(tried) == {"1", "2", "4", "8"} and d["config"]["stream_groups"] == int(min(tried, key=tried.get))
    assert d["gpu_launches"] == 20 * d["config"]["stream_groups"] and d["single_launch_per_step"]["ms_per_step"] == tried["1"]


def test_bench_dump_outputs_repeat_bit_for_bit(tmp_path):
    """--dump-outputs DIR: obs / reward / done / state after the last timed step, for a fixed sample of the environments;
    the same arguments give the same arrays bit for bit, one more timed step gives others."""
    def run(d, steps):
        res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", str(steps), "--warmup", "3", "--envs", "100000",
                              "--no-cpu", "--no-extra", "--dump-outputs", str(d)], capture_output=True, text=True, timeout=600)
        assert res.returncode == 0, res.stderr[-2000:]
        assert json.loads([l for l in res.stdout.splitlines() if l.strip()][-1])["steps"] == steps
        return {f[:-len(".npy")]: np.load(os.path.join(d, f)) for f in os.listdir(d)}
    a, b, c = run(tmp_path / "a", 20), run(tmp_path / "b", 20), run(tmp_path / "c", 21)
    assert sorted(a) == ["done", "env_index", "obs", "reward", "state"]
    k = 65536   # 100 000 environments: a sample
    assert a["obs"].shape == (k, 9) and a["state"].shape == (k, 12) and a["reward"].shape == a["done"].shape == a["env_index"].shape == (k,)
    assert all(v.dtype == np.float32 for n, v in a.items() if n != "env_index")
    assert np.array_equal(a["env_index"], np.unique(a["env_index"])) and 0 <= a["env_index"][0] and a["env_index"][-1] < 100000
    assert np.isin(a["done"], (0, 1)).all()
    for name in a:
        assert np.array_equal(a[name], b[name], equal_nan=True), name
    assert not np.array_equal(a["state"], c["state"], equal_nan=True)
