"""CPU: host-side logic that needs no GPU - 3DoF / legacy constants against the
reference's golden values, struct layouts against the header, the sharding
arithmetic, and the episode-statistics reduction over a 2-rank gloo group."""
import ctypes as C
import os
import subprocess
import sys
import textwrap

import numpy as np
import pytest

from conftest import ROOT, load_golden
from marinevehiclereinforcementlearning_b200 import _lib
from marinevehiclereinforcementlearning_b200.distributed import shard_range


@pytest.fixture(scope="module")
def lib():
    if not os.path.exists(_lib.LIB_PATH):
        _lib.build()
    return _lib.load()


def test_rov3_native_and_python_constants(lib):
    from marinevehiclereinforcementlearning_b200.rov3 import Rov3Constants
    g = load_golden("rov3")
    p = _lib.MvrlRov3Params()
    assert lib.mvrl_rov3_default_params(C.byref(p)) == 0
    q = Rov3Constants().to_struct()
    assert np.abs(np.array(p.Ainv).reshape(4, 3) - g["Ainv3"]).max() < 1e-14
    assert np.array_equal(np.array(q.Ainv).reshape(4, 3), g["Ainv3"])
    for name, _ in _lib.MvrlRov3Params._fields_:
        a, b = getattr(p, name), getattr(q, name)
        a, b = (np.array(a), np.array(b)) if hasattr(a, "__len__") else (np.array([a]), np.array([b]))
        assert np.abs(a - b).max() <= 1e-13 * max(1.0, np.abs(b).max()), name
    assert C.sizeof(_lib.MvrlRov3Params) == (27 + 9 + 9 + 12 + 15) * 8


def test_auv_native_constants_and_layout(lib):
    p = _lib.MvrlAuvParams()
    assert lib.mvrl_auv_default_params(C.byref(p)) == 0
    # tag_00.../verySimpleAuv.py:110-132
    assert (p.m, p.Izz, p.maxForce, p.maxMoment) == (11.4, 0.16, 150., 20.)
    assert p.Xuu == -18.18 * 2.21 and p.Yvv == -21.66 * 4.87 and p.Xu == -4.03 * 2.21 and p.Yv == -6.22 * 4.87
    assert (p.xMin, p.xMax, p.yMin, p.yMax) == (-1., 1., -1., 1.)
    assert C.sizeof(_lib.MvrlAuvParams) == (17 + 96) * 8 + 8 and C.sizeof(_lib.MvrlAuvBuffers) == 16 * 8
    assert p.variant == 0 and p.n_waypoints == 0
    assert C.sizeof(_lib.MvrlAuvConfig) == 4 + 4 + 8 + 8 + 8 + 4 * 4


LEGACY_WITHOUT_GPU = textwrap.dedent("""
    import ctypes as C, sys
    sys.path.insert(0, %r)
    import numpy as np, pytest, torch
    from marinevehiclereinforcementlearning_b200 import _lib
    assert not torch.cuda.is_available()
    lib = _lib.load()
    p = _lib.MvrlAuvParams()
    lib.mvrl_auv_default_params(C.byref(p))
    cfg = _lib.MvrlAuvConfig(dtype=0, max_steps=250, dt=0.02)
    h = C.c_void_p()
    assert lib.mvrl_auv_create(C.byref(h), C.byref(p), C.byref(cfg)) == -3
    from marinevehiclereinforcementlearning_b200.tag_00_Dec2023_simpleControlTurbulence import flowGenerator
    with pytest.raises(RuntimeError):
        flowGenerator.ReconstructedFlow.from_base_field(np.zeros((4, 3, 3, 3)))
    from marinevehiclereinforcementlearning_b200 import dynamicsModel_BlueROV2_Heavy_3DoF as m3
    with pytest.raises(RuntimeError):
        m3.BlueROV2Heavy3DoF(np.zeros(3)).derivs(0.0, np.zeros(6))
    print("legacy without gpu ok")
""")


def test_legacy_create_without_gpu_fails_loudly(lib):
    """Checked in a fresh interpreter that sees no CUDA device (CUDA_VISIBLE_DEVICES=""), so it runs on GPU machines too."""
    res = subprocess.run([sys.executable, "-c", LEGACY_WITHOUT_GPU % ROOT], env=dict(os.environ, CUDA_VISIBLE_DEVICES=""),
                         capture_output=True, text=True, timeout=600)
    assert res.returncode == 0 and "legacy without gpu ok" in res.stdout, res.stdout[-2000:] + res.stderr[-2000:]


def test_shard_range_partitions_every_env_once():
    for total, world in ((1 << 20, 8), (1000, 3), (7, 8), (262144, 4)):
        blocks = [shard_range(total, r, world) for r in range(world)]
        assert blocks[0][0] == 0 and blocks[-1][1] == total
        assert all(blocks[r][1] == blocks[r + 1][0] for r in range(world - 1))
        sizes = [hi - lo for lo, hi in blocks]
        assert max(sizes) - min(sizes) <= 1


def test_pdcontroller_matches_reference_law():
    from marinevehiclereinforcementlearning_b200.tag_00_Dec2023_simpleControlTurbulence.verySimpleAuv import PDController
    import torch
    obs = np.array([[0.5, -0.2, 0.9, 0, 0, 0, 0, 0, 0, 0, 0], [0.4, -0.1, 0.7, 0, 0, 0, 0, 0, 0, 0, 0]], dtype=float)
    pd = PDController(0.02)
    a0, s0 = pd.predict(obs[0])
    a1, _ = pd.predict(obs[1])
    assert np.allclose(a0, [0.5, -0.2, 0.9]) and np.array_equal(s0, obs[0])
    want = np.clip(obs[1, :3] + (obs[1, :3] - obs[0, :3]) / 0.02 * np.array([0.05, 0.05, 0.01]), -1, 1)
    assert np.allclose(a1, want)
    pdt = PDController(0.02)
    pdt.predict(torch.as_tensor(obs[0:1]))
    at, _ = pdt.predict(torch.as_tensor(obs[1:2]))
    assert np.allclose(at.numpy()[0], want)


WORKER = textwrap.dedent("""
    import os, sys
    sys.path.insert(0, %r)
    import torch, torch.distributed as dist
    from marinevehiclereinforcementlearning_b200.distributed import reduce_episode_stats, shard_range
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    dist.init_process_group("gloo", init_method="tcp://127.0.0.1:%%s" %% os.environ["MASTER_PORT"], rank=rank, world_size=world)
    lo, hi = shard_range(1000, rank, world)
    # per-rank accumulators as the step kernels leave them: episodes, sum len, sum ret, min, max, nonfinite, 0, 0
    s = torch.tensor([hi - lo, 250.0 * (hi - lo), 2.0 * (hi - lo) * (rank + 1), -1.0 - rank, 5.0 + rank, rank, 0, 0], dtype=torch.float64)
    out = reduce_episode_stats(s)
    assert out["episodes"] == 1000 and out["mean_length"] == 250.0, out
    assert out["min_return"] == -2.0 and out["max_return"] == 6.0 and out["nonfinite"] == 1, out
    assert abs(out["mean_return"] - (2.0 * 500 * 1 + 2.0 * 500 * 2) / 1000) < 1e-12, out
    dist.destroy_process_group()
    print("rank %%d ok" %% rank)
""")


def test_episode_stats_allreduce_gloo_world2(tmp_path):
    script = tmp_path / "worker.py"
    script.write_text(WORKER % ROOT)
    port = str(29500 + os.getpid() % 2000)
    procs = []
    for r in range(2):
        env = dict(os.environ, RANK=str(r), WORLD_SIZE="2", MASTER_ADDR="127.0.0.1", MASTER_PORT=port)
        procs.append(subprocess.Popen([sys.executable, str(script)], env=env, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True))
    for r, p in enumerate(procs):
        out, _ = p.communicate(timeout=240)
        assert p.returncode == 0, out
        assert "rank %d ok" % r in out


def test_bench_reference_arm_prints_one_contract_line():
    """bench.py --impl reference (the CPU arm the driver runs first): exactly one JSON line on stdout with the
    contract's keys, whatever libraries write to stdout / stderr meanwhile."""
    import json
    import subprocess
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    res = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--steps", "3", "--warmup", "3"],
                         capture_output=True, text=True, timeout=600)
    assert res.returncode == 0, res.stderr[-2000:]
    lines = [l for l in res.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, res.stdout
    d = json.loads(lines[0])
    for key in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
                "dtype", "data", "config", "impl", "cpu_baseline", "e2e", "gpu_launches"):
        assert key in d, key
    assert d["impl"] == "reference" and d["gpu_launches"] == 0 and d["value"] > 0
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_bench_refuses_zero_steps_and_dumps_of_other_paths(tmp_path):
    """--steps is the number of timed steps (0 is an error); --dump-outputs writes the rov6 GPU path's outputs and is refused
    for the other paths instead of being ignored."""
    for extra in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", str(tmp_path / "d")],
                  ["--workload", "auv", "--dump-outputs", str(tmp_path / "d")]):
        res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + extra, capture_output=True, text=True, timeout=120)
        assert res.returncode == 2 and "error" in res.stderr and not res.stdout.strip(), extra
    assert not (tmp_path / "d").exists()


def test_bench_merges_shard_episode_statistics():
    """bench.py's config-4 leg steps the batch as several env objects (vec_tools.EnvShards): their episode statistics are
    reported as one record - sums, episode-weighted means, extremes; shards without a finished episode carry NaNs."""
    import math
    sys.path.insert(0, ROOT)
    import bench
    nan = float("nan")
    a = {"episodes": 10, "mean_length": 5.0, "mean_return": -2.0, "min_return": -7.0, "max_return": 1.0, "nonfinite": 0}
    b = {"episodes": 30, "mean_length": 9.0, "mean_return": 2.0, "min_return": -3.0, "max_return": 4.0, "nonfinite": 2}
    idle = {"episodes": 0, "mean_length": nan, "mean_return": nan, "min_return": nan, "max_return": nan, "nonfinite": 0}
    assert bench.merge_episode_stats([a]) is a
    m = bench.merge_episode_stats([a, idle, b])
    assert m["episodes"] == 40 and m["nonfinite"] == 2 and m["min_return"] == -7.0 and m["max_return"] == 4.0
    assert abs(m["mean_length"] - 8.0) < 1e-12 and abs(m["mean_return"] - 1.0) < 1e-12
    e = bench.merge_episode_stats([idle, idle])
    assert e["episodes"] == 0 and math.isnan(e["mean_length"]) and math.isnan(e["min_return"])


class _FakeStream:
    """Stands in for torch.cuda.Stream on a box without a GPU: records what it was made to wait for."""
    def __init__(self, device=None):
        self.device, self.waited = device, []

    def wait_stream(self, other):
        self.waited.append(other)


def _fake_cuda(monkeypatch):
    import contextlib
    import torch
    cur = {"s": _FakeStream("caller")}

    @contextlib.contextmanager
    def use(s):
        prev, cur["s"] = cur["s"], s
        try:
            yield
        finally:
            cur["s"] = prev
    monkeypatch.setattr(torch.cuda, "Stream", _FakeStream)
    monkeypatch.setattr(torch.cuda, "current_stream", lambda device=None: cur["s"])
    monkeypatch.setattr(torch.cuda, "stream", use)
    return cur


def test_env_blocks_host_logic_with_fake_streams(monkeypatch):
    """vec_tools.EnvBlocks / EnvShards, host side only (the CUDA part is tests/test_vec_tools_gpu.py): the blocks tile the
    batch once, start on multiples of `align`, every block's step is queued on ITS stream, the block streams wait for the
    caller's stream at the fork and the caller's stream waits for every block stream at the join."""
    from marinevehiclereinforcementlearning_b200 import vec_tools
    cur = _fake_cuda(monkeypatch)
    caller = cur["s"]

    class Env:
        num_envs, device = 10007, "cuda:0"

        def __init__(self):
            self.calls = []

        def step_range_async(self, first, count):
            self.calls.append((first, count, cur["s"]))

    for n, groups, align in [(10007, 3, 2), (131072, 8, 2), (131072, 3, 128), (130, 8, 128), (5, 1, 2), (7, 7, 1)]:
        env = Env()
        env.num_envs = n
        b = vec_tools.EnvBlocks(env, groups, align)
        assert 1 <= len(b) <= groups and len(b.streams) == len(b.blocks)
        covered = []
        for lo, cnt in b.blocks:
            assert lo % align == 0 and cnt > 0
            covered += list(range(lo, lo + cnt))
        assert covered == list(range(n))                       # every environment once, in order
        with pytest.raises(RuntimeError):
            b.step_async()                                     # not forked
        with b:
            assert all(s.waited == [caller] for s in b.streams)
            b.step_async()
            b.step_async()
        assert caller.waited[-len(b):] == b.streams            # joined
        assert [(lo, cnt) for lo, cnt, _ in env.calls] == b.blocks * 2
        assert [s for _, _, s in env.calls] == b.streams * 2    # block g always on stream g
        assert [(lo, cnt, s) for lo, cnt, s in b] == [(lo, cnt, s) for (lo, cnt), s in zip(b.blocks, b.streams)]
        with pytest.raises(RuntimeError):
            b.step_async()                                     # joined again
    with pytest.raises(TypeError):
        vec_tools.EnvBlocks(object(), 2)
    with pytest.raises(ValueError):
        vec_tools.EnvBlocks(Env(), 0)

    class Shard:
        device = "cuda:0"

        def __init__(self):
            self.on = []

        def step_async(self):
            self.on.append(cur["s"])

    parts = [Shard() for _ in range(3)]
    sh = vec_tools.EnvShards(parts)
    assert len(sh) == 3 and [e for e, _ in sh] == parts
    with pytest.raises(RuntimeError):
        sh.step_async()
    with sh:
        sh.step_async()
    assert [p.on for p in parts] == [[s] for s in sh.streams] and caller.waited[-3:] == sh.streams
    with pytest.raises(ValueError):
        vec_tools.EnvShards([])
