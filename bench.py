#!/usr/bin/env python
"""Benchmark of the batched BlueROV2 6DoF env step (BASELINE.json metric:
"BlueROV2 6DoF env-steps/sec ... (1M envs); % of FP pipe peak").

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--scaling weak|strong] [--dump-outputs DIR]

Workload (config 3 of BASELINE.json, SURVEY.md 8(d)): BlueROV2 Heavy 6DoF,
fp32, 1 048 576 environments PER GPU (weak scaling: the path shards by
environment with no data-path collective), direct thruster-rpm actions
~U(-3500, 3500) (seed 1234 + rank), dt = 0.2 s as nSub = 8 fixed RK4 sub-steps,
maxSteps = 250 with auto-reset.  One "step" = one pass of the fused step kernel
over the whole batch: every environment advances by one env step.  The pass is
G launches, one per block of environments (vec_tools.EnvBlocks: the blocks are
independent, each steps as its own chain on its own stream, like the reference's
SubprocVecEnv workers); G is the fastest of 1 / 2 / 4 / 8 in a 40-step calibration
run unless --stream-groups fixes it, the line says which (config.stream_groups)
and carries the one-launch-per-step figure of the same run beside the headline
(single_launch_per_step).  Prints ONE JSON line (rank 0).

Next to the headline the line carries (all measured in the same run, a few seconds in total):
  "strong"  (N > 1) the config as written - 1 048 576 environments IN TOTAL, N / G per GPU (`--scaling strong`
            makes that the headline instead);
  "extra"   short legs of the other configurations: set-point (the reference's Gym semantics) / force modes, fp64,
            n_sub 1 and 4, config 2 (4096 envs fp64), config 4 (legacy auv_step, over calibrated vec_tools.EnvShards),
            the 3DoF env, config 5 (rollout collection: fused actor kernel + env step, at every N, with the
            episode-statistics all-reduce; the PyTorch-policy baseline and the two-block form beside it), and at N = 1
            the single-GPU rates of the 1/2, 1/4, 1/8, 1/16 shards of the 1 Mi batch.

`--impl reference` times the reference's CPU implementation of the same path:
the reference is pure Python (no compiled artefact can be built from it and
/root/reference does not exist on the GPU box), so this arm runs the C port of
it (oracle/mvrl_oracle.c, pinned to vectors produced by the unmodified
reference) on all host threads, on a bounded sample of the same workload.
"""
import argparse
import glob
import json
import os
import re
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True   # the benchmark writes nothing into the tree it runs from (which may be read-only)

import numpy as np  # noqa: E402

METRIC = "BlueROV2 6DoF env-steps/sec"
UNIT = "env-steps/s"
ENVS_PER_GPU = 1 << 20
ENVS_TOTAL_STRONG = 1 << 20
N_SUB = 8
DT = 0.2
MAX_STEPS = 250
CPU_SAMPLE_ENVS = 32768
# SURVEY.md 8(d): algorithmic work of one 6DoF env step, direct-rpm mode
FLOP_PER_ENV_STEP = 1600 * N_SUB + 60          # FMA = 2, other fp ops = 1, libm calls not counted
BYTES_PER_ENV_STEP_F32 = 177                   # state r/w, action r, obs/reward/done w, counter r/w
NOMINAL_FP32_TFLOPS = 148 * 128 * 2 * 1.965e9 / 1e12


def kernel_stats():
    """What the built kernels execute, counted from their SASS by tools/kernel_stats.py at build() time
    (marinevehiclereinforcementlearning_b200/kernel_stats.json; counted here when that file is missing or older than the
    library, without writing it: the tree may be read-only)."""
    path = os.path.join(ROOT, "marinevehiclereinforcementlearning_b200", "kernel_stats.json")
    lib = os.environ.get("MVRL_LIB") or os.path.join(ROOT, "marinevehiclereinforcementlearning_b200", "libmvrl.so")
    try:
        if os.environ.get("MVRL_LIB") or not os.path.exists(path) or os.path.getmtime(path) < os.path.getmtime(lib):
            sys.path.insert(0, os.path.join(ROOT, "tools"))
            import kernel_stats as ks
            return ks.collect(lib)
        return json.load(open(path))
    except Exception as e:   # cuobjdump missing etc.: the line then says so instead of carrying a stale constant
        return {"error": str(e), "kernels": {}}


def ncu_traffic(kernel_regex):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the newest committed `ncu --set full` summary whose
    kernel name matches; (bytes, file) or (None, None)."""
    best = (None, None)
    files = sorted(glob.glob(os.path.join(ROOT, "profiles", "*_ncu_full_summary.txt")),
                   key=lambda f: (int((re.search(r"/r(\d+)_", f) or [0, 0])[1]), os.path.basename(f)))
    unit = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}
    for f in files:
        for block in open(f).read().split("----"):
            name = re.search(r"Kernel Name = (.*)", block)
            rd = re.search(r"dram__bytes_read.sum = ([\d.]+) (\w+)", block)
            wr = re.search(r"dram__bytes_write.sum = ([\d.]+) (\w+)", block)
            grid = re.search(r"launch__grid_size = (\d+)", block)
            if name and rd and wr and re.search(kernel_regex, name.group(1)) and grid and int(grid.group(1)) >= 4096:
                best = (float(rd.group(1)) * unit[rd.group(2)] + float(wr.group(1)) * unit[wr.group(2)], os.path.relpath(f, ROOT))
    return best


ACTION_SCALE = {"rpm": 3500.0, "force": 40.0, "setpoint": 1.0}
ACTION_DIM = {"rpm": 8, "force": 6, "setpoint": 6}
# SURVEY.md 8(d): derivative = 360 flop (rpm) / 610 (PID set-point; force mode has the allocation but no PID: 538)
DERIV_FLOP = {"rpm": 360, "force": 538, "setpoint": 610}


def flop_per_env_step(mode, n_sub):
    return (4 * DERIV_FLOP[mode] + 160) * n_sub + 60


def bytes_per_env_step(mode, w):
    b = 12 * w * 2 + ACTION_DIM[mode] * w + 9 * w + w + 1 + 8          # state r/w, action r, obs/reward/done w, counter r/w
    if mode == "setpoint":
        b += 13 * w * 2 + 6 * w * 2 + 6 * w                            # PID state r/w, set-point r/w, path r
    return b


def workload_name(envs, mode="rpm", dtype="f32", n_sub=N_SUB):
    return ("rov6_step %s: BlueROV2 Heavy 6DoF, %d envs/GPU, %s actions U(-%g,%g), dt=%.1f as nSub=%d RK4, "
            "maxSteps=%d auto-reset" % (dtype, envs, mode, ACTION_SCALE[mode], ACTION_SCALE[mode], DT, n_sub, MAX_STEPS))


# --------------------------------------------------------------------------
# The contract is ONE JSON line on stdout.  Libraries write there too (NCCL prints its version banner on the first
# collective), so file descriptor 1 is pointed at stderr for the whole run and the line goes to the saved descriptor.
_REAL_STDOUT = None


def capture_stdout():
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.dup(1)
        os.dup2(2, 1)


def emit(line):
    text = (json.dumps(line) + "\n").encode()
    sys.stdout.flush()
    if _REAL_STDOUT is None:
        os.write(1, text)
    else:
        os.write(_REAL_STDOUT, text)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.lines, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append((time.time(), line.strip()))

    def stop(self, t0, t1):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, smax, reasons, power = [], [], set(), []
        for ts, line in self.lines:
            f = [x.strip() for x in line.split(",")]
            if len(f) < 9:
                continue
            if t0 - 0.05 <= ts <= t1 + 0.15:
                try:
                    sm.append(float(f[1])); smax.append(float(f[2])); power.append(float(f[3]))
                except ValueError:
                    continue
                for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                    if val.lower().startswith("active"):
                        reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no sample inside the timed region"], "samples": 0}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(smax)), "reasons": sorted(reasons),
                "samples": len(sm), "power_w_max": max(power)}


def bind_to_gpu_numa_node(index):
    """Pin this rank's host threads (and with them its first-touch / pinned allocations) to the CPUs of the NUMA node the
    GPU hangs off: the e2e leg moves 76 MB per step between host memory and the GPU, and with one rank per GPU the
    cross-socket hop otherwise becomes the limiter.  Returns the node, or None when the topology is not exposed."""
    try:
        import torch
        pr = torch.cuda.get_device_properties(index)
        bdf = "%04x:%02x:%02x.0" % (pr.pci_domain_id, pr.pci_bus_id, pr.pci_device_id)
        node = int(open("/sys/bus/pci/devices/%s/numa_node" % bdf).read())
        if node < 0:
            return None
        cpus = set()
        for part in open("/sys/devices/system/node/node%d/cpulist" % node).read().strip().split(","):
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        cpus &= os.sched_getaffinity(0)
        if not cpus:
            return None
        os.sched_setaffinity(0, cpus)
        return node
    except Exception:
        return None


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return json.load(open(p)), "measured (MEASURED_PEAKS.json)"
    return {"hbm_gbs": 6650.0}, "fallback (B200_PROFILING.md)"


# --------------------------------------------------------------------------
def host_threads():
    """All the host threads this process may use (torchrun exports OMP_NUM_THREADS=1, which must not throttle the CPU arm)."""
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


def cpu_port_rate(n_envs, n_steps, threads=0, seed=1234):
    """env-steps/s of the C port of the reference's step loop on the host."""
    from oracle import c_oracle as c
    from oracle import oracle_np as o
    threads = threads or host_threads()
    env = c.Rov6EnvC(n_envs, mode=o.MODE_RPM, max_steps=MAX_STEPS, n_sub=N_SUB, dt=DT, auto_reset=True, seed=seed, threads=threads)
    env.reset()
    rng = np.random.default_rng(seed)
    acts = rng.uniform(-3500.0, 3500.0, (4, n_envs, 8))
    env.step(acts[0])  # warm-up (thread pool, page faults)
    t0 = time.perf_counter()
    for k in range(n_steps):
        env.step(acts[k % 4])
    dt = time.perf_counter() - t0
    return n_envs * n_steps / dt, dt, threads


def python_port_rate(seconds=3.0):
    """env-steps/s of the numpy restatement stepped ONE environment at a time -
    the shape of the reference's own loop (per-env Python/numpy, one core)."""
    from oracle import oracle_np as o
    env = o.Rov6EnvOracle(1, mode=o.MODE_RPM, max_steps=10 ** 9, n_sub=N_SUB, dt=DT)
    env.reset(initial_setpoint=np.zeros(6))
    rng = np.random.default_rng(0)
    n, t0 = 0, time.perf_counter()
    while time.perf_counter() - t0 < seconds:
        env.step(rng.uniform(-3500, 3500, (1, 8)))
        n += 1
    return n / (time.perf_counter() - t0)


def as_shipped_port_rate(seconds=2.0):
    """env-steps/s of the reference's env step AS SHIPPED (6DoF.py:545-557: scipy RK45, rtol = atol = 1e-3,
    max_step = dt, stateful PID inside the right-hand side, fixed set-point) with the numpy port of its derivs, one core."""
    from scipy.integrate import solve_ivp
    from oracle import oracle_np as o
    p = o.Rov6Params()
    ctrl = o.pid6_new_state(1)
    sp = np.array([[0.5, -0.3, 0.2, 0., 0., 1.0]])
    y, t, n, t0 = np.zeros(12), 0.0, 0, time.perf_counter()
    while time.perf_counter() - t0 < seconds:
        res = solve_ivp(lambda tt, yy: o.derivs6_pid(p, tt, yy[None], ctrl, sp)[0], (t, t + DT), y, method="RK45", t_eval=[t + DT],
                        max_step=DT, rtol=1e-3, atol=1e-3)
        y, t, n = res.y[:, -1], t + DT, n + 1
        y[3:6] %= 2 * np.pi
    return n / (time.perf_counter() - t0)


def legacy_port_rate(seconds=2.0):
    """env-steps/s of the legacy AuvEnv.step (verySimpleAuv.py:264-410) as the numpy port steps it, ONE environment at a
    time like the reference, synthetic flow field of config 4 (256 time levels), one core."""
    from oracle import oracle_np as o
    ltm = np.load(os.path.join(ROOT, "tests", "golden", "golden_legacy.npz"))["ltm"]
    rng = np.random.default_rng(7)
    flow = o.FlowOracle(ltm[None] + 0.05 * rng.standard_normal((256,) + ltm.shape))
    flow.scale(11., 1.0, 2.0, translate=(-1.65, -1.1))
    env = o.AuvEnvOracle(1, flow, noiseMagCoeffs=0.1, noiseMagActuation=0.1, auto_reset=True, seed=1)
    env.reset()
    n, t0 = 0, time.perf_counter()
    while time.perf_counter() - t0 < seconds:
        env.step(rng.uniform(-1, 1, (1, 3)))
        n += 1
    return n / (time.perf_counter() - t0)


def run_reference(args, rank, world):
    if rank != 0:
        return
    n_envs = CPU_SAMPLE_ENVS
    from oracle import c_oracle as c
    from oracle import oracle_np as o
    threads = host_threads()
    env = c.Rov6EnvC(n_envs, mode=o.MODE_RPM, max_steps=MAX_STEPS, n_sub=N_SUB, dt=DT, auto_reset=True, seed=1234, threads=threads)
    env.reset()
    rng = np.random.default_rng(1234)
    acts = rng.uniform(-3500.0, 3500.0, (4, n_envs, 8))
    for k in range(args.warmup):
        env.step(acts[k % 4])
    t0 = time.perf_counter()
    for k in range(args.steps):
        env.step(acts[k % 4])
    t_total = time.perf_counter() - t0
    value = n_envs * args.steps / t_total
    sample = ("%d envs x 1 env step per bench step (nSub=%d RK4), all host threads; a SAMPLE of the %d-env workload - the metric is "
              "throughput per env-step, so the rate carries over" % (n_envs, N_SUB, ENVS_PER_GPU))
    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": 1e3 * t_total / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic", "impl": "reference",
            "config": {"workload": workload_name(ENVS_PER_GPU), "sample_envs": n_envs, "l2": "n/a (CPU arm)"},
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    emit(line)


# --------------------------------------------------------------------------
# timing helpers shared by every leg
def _barrier(world):
    import torch
    import torch.distributed as dist
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()


def _max_over_ranks(x, dev, world):
    import torch
    import torch.distributed as dist
    t = torch.tensor([x], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t[0])


def timed_launches(dev, world, one_step, steps, warmup, graph=True, clocks=False, blocks=None):
    """W untimed calls of one_step(k), then EXACTLY `steps` timed ones (replayed as ONE CUDA graph unless graph=False)
    between barrier + synchronize on both sides; CUDA events on the launching stream; returns (ms max over ranks, clocks).
    blocks = vec_tools.EnvBlocks: one_step(k) queues step k of every block on the block's own stream; the block streams
    fork from the timed stream after the start event and re-join it before the stop event (parallel branches of the
    same graph), so every environment still takes exactly `steps` steps inside the timed region."""
    import contextlib
    import torch

    def issue(count):
        with (blocks if blocks is not None else contextlib.nullcontext()):
            for k in range(count):
                one_step(k)

    issue(warmup)
    _barrier(world)
    g = None
    if graph:
        g = torch.cuda.CUDAGraph()
        side = torch.cuda.Stream(device=dev)
        side.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(side):
            with torch.cuda.graph(g, stream=side):
                issue(steps)
        torch.cuda.current_stream(dev).wait_stream(side)
        g.replay()   # warm-up replay
        _barrier(world)
    sampler = None
    if clocks:
        sampler = ClockSampler(dev.index)
        sampler.start()
        time.sleep(0.25)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    _barrier(world)
    t0 = time.time()
    e0.record()
    if g is not None:
        g.replay()
    else:
        issue(steps)
    e1.record()
    _barrier(world)
    t1 = time.time()
    ms = _max_over_ranks(e0.elapsed_time(e1), dev, world)
    return ms, (sampler.stop(t0, t1) if sampler else None)


def rov6_leg(dev, rank, world, n, mode="rpm", dtype="f32", n_sub=N_SUB, steps=50, warmup=5, env_id0=None, max_steps=MAX_STEPS,
             fast=0, stats=True, graph=True, clocks=False, keep=False, groups=1):
    """One timed leg of the fused 6DoF step: n environments on this rank; returns rate per GPU (n / max-over-ranks time).
    groups > 1 (0 = pick the fastest of 1 / 2 / 4 / 8 by a short calibration run): the environments are stepped as
    `groups` independent blocks (vec_tools.EnvBlocks -> mvrl_rov6_step_range), each block a chain of launches on its own
    stream - the analogue of the reference's SubprocVecEnv workers, which step their environments without waiting for each other (legacy/script_0_checkScaling.py:23-40).  Every environment still takes exactly
    `steps` steps; a block's prologue / epilogue then overlaps the other blocks' RK4 loops instead of idling the SMs."""
    import torch
    from marinevehiclereinforcementlearning_b200 import BlueROV2Heavy6DoFVecEnv
    tdtype = torch.float64 if dtype == "f64" else torch.float32
    na = ACTION_DIM[mode]
    env = BlueROV2Heavy6DoFVecEnv(n, action_mode=mode, dtype=tdtype, device=dev, dt=DT, maxSteps=max_steps, n_sub=n_sub, seed=1234,
                                  env_id0=rank * n if env_id0 is None else env_id0, auto_reset=True, fast_math=bool(fast),
                                  record_terminal_obs=False, collect_stats=stats)
    env.reset()
    gen = torch.Generator(device=dev).manual_seed(1234 + rank)
    n_act = 4  # rotating action batches
    acts = [(torch.rand((na, env.ld), generator=gen, device=dev, dtype=tdtype) * 2 - 1) * ACTION_SCALE[mode] for _ in range(n_act)]
    # stagger episode phase like a long-running job: env i starts at iStep = i % maxSteps
    env._istep.copy_((torch.arange(env.ld, device=dev) % max_steps).to(torch.int32))

    def one_step(k):
        env._bufs.action = acts[k % n_act].data_ptr()
        env.step_async()
    from marinevehiclereinforcementlearning_b200.vec_tools import EnvBlocks

    def blocked(g):
        if g <= 1:
            return None, one_step
        eb = EnvBlocks(env, g)

        def blocked_step(k):
            env._bufs.action = acts[k % n_act].data_ptr()
            eb.step_async()
        return eb, blocked_step
    tried = None
    if groups == 0:   # auto: a short calibration run of each candidate (same kernels, same environments), the fastest is timed
        tried = {}
        for g in ((1, 2, 4, 8) if n >= 65536 else (1,)):
            eb, f = blocked(g)
            tried[g] = timed_launches(dev, world, f, min(steps, 40), 3, graph=graph, blocks=eb)[0] / min(steps, 40)
        groups = min(tried, key=tried.get)   # the times are maxima over the ranks: every rank makes the same choice
    blocks, step_fn = blocked(groups)
    ms, clk = timed_launches(dev, world, step_fn, steps, warmup, graph=graph, clocks=clocks, blocks=blocks)
    w = 8 if dtype == "f64" else 4
    touched = n * bytes_per_env_step(mode, w) + n_act * na * env.ld * w
    out = {"envs_per_gpu": n, "action_mode": mode, "dtype": dtype, "n_sub": n_sub, "steps": steps, "ms_per_step": ms / steps,
           "rate_per_gpu": n / (ms / steps * 1e-3), "stream_groups": len(blocks) if blocks is not None else 1,
           "stream_groups_tried_ms_per_step": tried,
           "l2": "larger than L2" if touched > 126e6 else "working set %.0f MB is L2-resident (what stepping a shard of this size is)" % (touched / 1e6)}
    if clk is not None:
        out["clocks"] = clk
    if stats:
        out["episode_stats"] = env.episode_stats(reset=True)  # K5; all-reduced over NCCL when world > 1 (off the timed path)
    if keep:
        out["env"], out["acts"] = env, acts
    else:
        env._bufs.action = env._action.data_ptr()
    return out


def leg_summary(leg, fp_peak):
    flop = flop_per_env_step(leg["action_mode"], leg["n_sub"])
    return {"value": leg["rate_per_gpu"], "unit": UNIT + " per GPU", "ms_per_step": leg["ms_per_step"], "envs_per_gpu": leg["envs_per_gpu"],
            "steps": leg["steps"], "algorithmic_flop_per_env_step": flop, "frac_of_fp_peak": leg["rate_per_gpu"] * flop / 1e12 / fp_peak,
            "stream_groups": leg["stream_groups"], "stream_groups_tried_ms_per_step": leg["stream_groups_tried_ms_per_step"], "l2": leg["l2"]}


def merge_episode_stats(stats):
    """Episode statistics of several shards as one (sums, weighted means, extremes)."""
    if len(stats) == 1:
        return stats[0]
    ep = sum(st["episodes"] for st in stats)
    out = {"episodes": ep, "nonfinite": sum(st.get("nonfinite", 0) for st in stats)}
    for k in ("mean_length", "mean_return"):
        out[k] = (sum(st[k] * st["episodes"] for st in stats if st["episodes"]) / ep) if ep else float("nan")
    live = [st for st in stats if st["episodes"]]
    out["min_return"] = min(st["min_return"] for st in live) if live else float("nan")
    out["max_return"] = max(st["max_return"] for st in live) if live else float("nan")
    return out


def auv_leg(dev, rank, world, n=262144, steps=50, warmup=5, field="modes", graph=True, clocks=False, groups=1):
    """Config 4: legacy AuvEnv, fp32, synthetic turbulence field [2000, 41, 61] scaled like verySimpleAuv.py:104,
    a ~ U(-1, 1)^3, noiseMag* = 0.1.  One step = one auv_step launch over the batch - or, groups > 1 (0 = the fastest of
    1 / 2 / 4 / 8 by a short calibration run), one launch per shard: the batch as `groups` env objects with consecutive env_id0,
    each stepping as a chain on its own stream (vec_tools.EnvShards; the reference's SubprocVecEnv workers)."""
    import torch
    from marinevehiclereinforcementlearning_b200 import AuvVecEnv
    from marinevehiclereinforcementlearning_b200.tag_00_Dec2023_simpleControlTurbulence import flowGenerator
    from marinevehiclereinforcementlearning_b200.vec_tools import EnvShards
    ltm = np.load(os.path.join(ROOT, "tests", "golden", "golden_legacy.npz"))["ltm"]   # the reference's ltm.npy (41 x 61 x 3)
    flow = flowGenerator.ReconstructedFlow.synthetic(lt_mean=ltm, nt=2000, seed=7, sigma=0.05, kind=field, dtype=torch.float32, device=dev)
    flow.scale(11., 1.0, 2.0, translate=(-1.65, -1.1))

    def make(g):
        per = -(-n // g)
        envs, fns = [], []
        gen = torch.Generator(device=dev).manual_seed(1234 + rank)
        for lo in range(0, n, per):
            e = AuvVecEnv(min(per, n - lo), flow, seed=1234, env_id0=rank * n + lo, noiseMagCoeffs=0.1, noiseMagActuation=0.1, auto_reset=True,
                          dtype=torch.float32, record_terminal_obs=False)
            e.reset()
            acts = [torch.rand((3, e.ld), generator=gen, device=dev) * 2 - 1 for _ in range(8)]
            envs.append(e)
            fns.append(acts)
        if g == 1:
            def one_step(k):
                envs[0]._bufs.action = fns[0][k % 8].data_ptr()
                envs[0].step_async()
            return envs, None, one_step
        shards = EnvShards(envs)

        def sharded_step(k):
            for e, acts in zip(envs, fns):
                e._bufs.action = acts[k % 8].data_ptr()
            shards.step_async()
        return envs, shards, sharded_step
    tried = None
    if groups == 0:
        tried = {}
        for g in (1, 2, 4, 8):
            _, sh, f = make(g)
            tried[g] = timed_launches(dev, world, f, min(steps, 40), 5, graph=graph, blocks=sh)[0] / min(steps, 40)
        groups = min(tried, key=tried.get)
    envs, shards, step_fn = make(groups)
    ms, clk = timed_launches(dev, world, step_fn, steps, warmup, graph=graph, clocks=clocks, blocks=shards)
    rate = n / (ms / steps * 1e-3)
    # state 6 r/w, action 3 r, obs 11 w, reward w, mults 11 r, target 2 r, err_o 3 r/w, ring 30 r + 3 w, return r/w, done 1, istep 8
    nbytes = (12 + 3 + 11 + 1 + 11 + 2 + 6 + 33 + 2) * 4 + 9
    peaks, peak_src = measured_peaks()
    return {"value": rate, "unit": UNIT + " per GPU", "ms_per_step": ms / steps, "envs_per_gpu": n, "steps": steps, "field": field,
            "stream_groups": len(envs), "stream_groups_tried_ms_per_step": tried,
            "hbm_gbs": rate * nbytes / 1e9, "frac_of_hbm_peak": rate * nbytes / 1e9 / peaks["hbm_gbs"], "bytes_per_env_step": nbytes,
            "gathered_bytes_per_env_step_from_l2": 64, "peak_source": peak_src, "clocks": clk,
            "episode_stats": merge_episode_stats([e.episode_stats() for e in envs]),
            "l2": "40 MB field is L2-resident by design; per-env arrays (87 MB / step) rotate through 8 action batches"}


def rov3_leg(dev, rank, world, n, mode, n_sub=N_SUB, steps=50, warmup=5, clocks=False):
    """Config 1's model at scale: BlueROV2 Heavy 3DoF env, fp32, setpoint = the reference's Gym semantics, rpm = 4 thruster rpm."""
    import torch
    from marinevehiclereinforcementlearning_b200 import BlueROV2Heavy3DoFVecEnv
    na, scale = (4, 3500.0) if mode == "rpm" else (3, 1.0)
    env = BlueROV2Heavy3DoFVecEnv(n, action_mode=mode, dtype=torch.float32, device=dev, dt=DT, maxSteps=MAX_STEPS, n_sub=n_sub,
                                  seed=1234, env_id0=rank * n, auto_reset=True, record_terminal_obs=False)
    env.reset()
    gen = torch.Generator(device=dev).manual_seed(1234 + rank)
    acts = [(torch.rand((na, env.ld), generator=gen, device=dev) * 2 - 1) * scale for _ in range(8)]
    env._istep.copy_((torch.arange(env.ld, device=dev) % MAX_STEPS).to(torch.int32))

    def one_step(k):
        env._bufs.action = acts[k % 8].data_ptr()
        env.step_async()
    ms, clk = timed_launches(dev, world, one_step, steps, warmup, clocks=clocks)
    return {"value": n / (ms / steps * 1e-3), "unit": UNIT + " per GPU", "ms_per_step": ms / steps, "envs_per_gpu": n, "steps": steps,
            "action_mode": mode, "n_sub": n_sub, "clocks": clk, "episode_stats": env.episode_stats()}


def rollout_leg(dev, rank, world, n=131072, T=128, rollouts=2, n_sub=N_SUB, clocks=False, policy="fused", groups=1):
    """Config 5: rollout collection over the 6DoF env in the reference's Gym semantics (PID set-point actions) with the
    policy of legacy/main_00_sbl.py:100-105 (MLP 9-128-128-128-6, GELU) + Gaussian head; T-step rollouts replayed as one
    CUDA graph, episode statistics all-reduced once per rollout (K5, NCCL when N > 1).
    policy = "fused": the actor is ONE tensor-core kernel (mvrl_policy_act) on the env's own buffers and the env writes
    observation / reward / done straight into the rollout buffers, so a rollout step is two launches.
    policy = "torch": the same network as PyTorch library calls (cuBLASLt TF32 GEMMs with fused bias + GELU, elementwise
    sampling kernels) - the baseline the fused actor replaces."""
    import torch
    from marinevehiclereinforcementlearning_b200 import BlueROV2Heavy6DoFVecEnv, MlpGaussianPolicy
    torch.backends.cuda.matmul.allow_tf32 = True
    env = BlueROV2Heavy6DoFVecEnv(n, action_mode="setpoint", dtype=torch.float32, device=dev, n_sub=n_sub, seed=1234,
                                  env_id0=rank * n, auto_reset=True, record_terminal_obs=False)
    env.reset()
    pol = MlpGaussianPolicy(9, 6, device=dev, seed=1234)
    ld = env.ld
    buf_obs = torch.empty((T + 1, 9, ld), device=dev)
    buf_act = torch.empty((T, 6, ld), device=dev)
    buf_logp = torch.empty((T, ld), device=dev)
    buf_rew = torch.empty((T, ld), device=dev)
    buf_done = torch.empty((T, ld), dtype=torch.uint8, device=dev)
    own = (env._bufs.obs, env._bufs.action, env._bufs.reward, env._bufs.done)

    if policy == "fused":
        buf_obs[0].copy_(env._obs)

        import ctypes as C
        from marinevehiclereinforcementlearning_b200 import _lib

        def policy_step(t, lo=0, cnt=n):
            if cnt == n:
                pol.act_into(buf_obs[t], buf_act[t], n, logp=buf_logp[t], env_id0=rank * n, step=t)
            else:   # environments [lo, lo + cnt) of the same rows: the C entry point takes plain pointers
                o = 4 * lo
                _lib.check(pol.lib.mvrl_policy_act(pol._h, cnt, ld, C.c_void_p(buf_obs[t].data_ptr() + o), C.c_void_p(buf_act[t].data_ptr() + o),
                                                   C.c_void_p(buf_logp[t].data_ptr() + o), None, None, pol.seed & (2 ** 64 - 1), rank * n + lo, t, 0,
                                                   _lib.current_stream(dev)))

        def env_step(t, lo=0, cnt=n):   # the step kernel reads the actor's output and writes the next rollout row: no copies
            env._bufs.action, env._bufs.obs = buf_act[t].data_ptr(), buf_obs[t + 1].data_ptr()
            env._bufs.reward, env._bufs.done = buf_rew[t].data_ptr(), buf_done[t].data_ptr()
            if cnt == n:
                env.step_async()
            else:
                env.step_range_async(lo, cnt)

        # groups > 1: the environments are split into independent blocks, each block a chain (actor, env step) x T on its
        # own stream - one block's actor (tensor core / XU pipe) runs beside another block's env step (FMA pipe)
        eb = None
        if groups > 1:
            from marinevehiclereinforcementlearning_b200.vec_tools import EnvBlocks
            eb = EnvBlocks(env, groups, align=128)           # whole actor tiles
        blocks = eb.blocks if eb is not None else [(0, n)]

        def rollout():
            if eb is None:
                for t in range(T):
                    policy_step(t)
                    env_step(t)
            else:
                with eb:
                    for lo, cnt, s in eb:
                        with torch.cuda.stream(s):
                            for t in range(T):
                                policy_step(t, lo, cnt)
                                env_step(t, lo, cnt)
            buf_obs[0].copy_(buf_obs[T])   # the next rollout starts where this one ended
        launches_per_step = 2 * len(blocks)
    else:
        Wt = [w.to(dev).T.contiguous() for w in pol.weights]         # [in, out]
        b1 = [b.to(dev) for b in pol.biases]
        obs_nk = env._obs.T                          # [ld, 9] strided view of the SoA observation buffer: cuBLAS reads it in place
        std = pol.log_std.exp().reshape(1, 6).to(dev)
        logp_const = pol.logp_const

        def policy_step(t):
            buf_obs[t].copy_(env._obs)
            h = obs_nk
            for i in range(3):    # batch-major activations [N, k]; bias + GELU fused into the GEMM epilogue (cuBLASLt)
                h = torch._addmm_activation(b1[i], h, Wt[i], use_gelu=True)
            mean = torch.tanh(torch.addmm(b1[3], h, Wt[3]))
            eps = torch.randn_like(mean)
            act = torch.addcmul(mean, eps, std).clamp_(-1., 1.)
            buf_logp[t].copy_((eps * eps).sum(1).mul_(-0.5).add_(logp_const))
            buf_act[t].copy_(act.T)             # back to the env's feature-major action layout

        def env_step(t):
            env._bufs.action = buf_act[t].data_ptr()
            env.step_async()
            buf_rew[t].copy_(env._reward)
            buf_done[t].copy_(env._done)

        def rollout():
            for t in range(T):
                policy_step(t)
                env_step(t)
        launches_per_step = None
    rollout()
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    side = torch.cuda.Stream(device=dev)
    side.wait_stream(torch.cuda.current_stream(dev))
    with torch.cuda.stream(side):
        with torch.cuda.graph(graph, stream=side):
            rollout()
    torch.cuda.current_stream(dev).wait_stream(side)
    holder = {}

    def one_rollout(k):
        graph.replay()
        holder["s"] = env.episode_stats()     # K5: device accumulators -> all-reduce (NCCL) -> host, once per rollout
    ms, clk = timed_launches(dev, world, one_rollout, rollouts, 1, graph=False, clocks=clocks)
    # share of the env step: the same T env steps alone (the actor's last outputs as actions), as one graph
    g2 = torch.cuda.CUDAGraph()
    side.wait_stream(torch.cuda.current_stream(dev))
    with torch.cuda.stream(side):
        with torch.cuda.graph(g2, stream=side):
            for t in range(T):
                env_step(t)
    torch.cuda.current_stream(dev).wait_stream(side)
    ms_env, _ = timed_launches(dev, world, lambda k: g2.replay(), rollouts, 1, graph=False)
    env._bufs.obs, env._bufs.action, env._bufs.reward, env._bufs.done = own
    per_step = ms / (rollouts * T)
    dims = [9, 128, 128, 128, 6]
    return {"value": n * T * rollouts / (ms * 1e-3), "unit": UNIT + " per GPU (policy included)", "ms_per_step": per_step, "envs_per_gpu": n,
            "rollout_len": T, "rollouts": rollouts, "policy_impl": policy, "launches_per_step": launches_per_step, "stream_groups": max(1, groups),
            "env_share": (ms_env / (rollouts * T)) / per_step,
            "env_us_per_step": 1e3 * ms_env / (rollouts * T), "policy_and_bookkeeping_us_per_step": 1e3 * (per_step - ms_env / (rollouts * T)),
            "flop_per_env_step": {"env": flop_per_env_step("setpoint", n_sub), "policy": 2 * sum(dims[i] * dims[i + 1] for i in range(4))},
            "policy": (("MLP 9-128-128-128-6 GELU + Gaussian head as one kernel: warp-level mma.sync bf16 (fp32 accumulate), activations in "
                        "registers, weights in shared memory, Philox sampling (csrc/mvrl_policy.cu, MVRL_POLICY_MMA_SYNC=1)")
                       if os.environ.get("MVRL_POLICY_MMA_SYNC", "0") == "1" else
                       ("MLP 9-128-128-128-6 GELU + Gaussian head as one kernel: tcgen05.mma (bf16 operands through shared-memory descriptors, "
                        "fp32 accumulators in tensor memory, biases added by the tensor core), 128-environment tiles, 4 in flight per SM, "
                        "Philox sampling (csrc/mvrl_policy.cu)")) if policy == "fused" else
                      "MLP 9-128-128-128-6 GELU + Gaussian head, PyTorch (cuBLASLt TF32 GEMMs with fused bias + GELU): library code",
            "stats_allreduce": "episode statistics (8 doubles) all-reduced once per rollout, inside the timed region" if world > 1 else "single rank: no collective",
            "clocks": clk, "episode_stats": holder.get("s")}


DUMP_SAMPLE_ENVS = 65536


def dump_outputs(out_dir, env):
    """--dump-outputs: what env.step() hands its caller after the last timed step - obs [k, 9], reward [k], done [k] (0 / 1) -
    and the state behind it (systemState [k, 12]), in the env's dtype, for the environments listed in env_index.npy: all of
    them, or a fixed sample of DUMP_SAMPLE_ENVS drawn with seed 0 (at most 13 MB in all).  The environments, their actions
    and the number of steps they take are fixed by the arguments, so two builds run with the same arguments compare file
    for file."""
    import torch
    n = env.num_envs
    idx = np.arange(n) if n <= DUMP_SAMPLE_ENVS else np.sort(np.random.default_rng(0).choice(n, DUMP_SAMPLE_ENVS, replace=False))
    sel = torch.as_tensor(idx, device=env.device)
    arrays = {"obs": env.state, "reward": env._reward[:n], "done": env._done[:n].to(env.dtype), "state": env.systemState}
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.index_select(0, sel).cpu().numpy())
    np.save(os.path.join(out_dir, "env_index.npy"), idx.astype(np.float64))


# --------------------------------------------------------------------------
def run_ours(args, rank, local_rank, world):
    import torch
    from marinevehiclereinforcementlearning_b200 import _lib
    from marinevehiclereinforcementlearning_b200.distributed import shard_range

    dev = torch.device("cuda", local_rank)
    numa_node = bind_to_gpu_numa_node(local_rank) if args.bind_numa else None
    strong = args.scaling == "strong"
    if strong:
        lo, hi = shard_range(ENVS_TOTAL_STRONG, rank, world)
        n, id0 = hi - lo, lo
    else:
        n, id0 = args.envs, rank * args.envs
    mode, n_sub = args.action_mode, args.n_sub
    w = 8 if args.dtype == "f64" else 4
    na = ACTION_DIM[mode]
    leg = rov6_leg(dev, rank, world, n, mode, args.dtype, n_sub, args.steps, args.warmup, env_id0=id0, max_steps=args.max_steps,
                   fast=args.fast_math, stats=not args.no_stats, graph=bool(args.graph), clocks=True, keep=True, groups=max(0, args.stream_groups))
    env, acts = leg["env"], leg["acts"]
    if args.dump_outputs and rank == 0:   # before the e2e leg below steps the same environments further
        dump_outputs(args.dump_outputs, env)
    ms_per_step = leg["ms_per_step"]
    n_total = ENVS_TOTAL_STRONG if strong else world * n
    value = n_total / (ms_per_step * 1e-3)

    # ---- end to end through the public API with HOST buffers -----------------
    # BlueROV2Heavy6DoFVecEnv.step_host -> mvrl_rov6_step_host: pinned host [N, 8] actions in, pinned host
    # obs [N, 9] / reward [N] / done [N] out, every step; upload / step / download pipelined over chunks.
    h_act = [a[:, :n].T.contiguous().cpu().pin_memory() for a in acts[:2]]          # [N, A] like a VecEnv caller
    env._bufs.action = env._action.data_ptr()

    def e2e_step(k):
        env.step_host(h_act[k % 2], chunks=args.e2e_chunks)                # returns when the host tensors are complete

    e2e_steps = max(3, min(args.steps, 50))
    for k in range(3):
        e2e_step(k)
    _barrier(world)
    w0 = time.perf_counter()
    for k in range(e2e_steps):
        e2e_step(k)
    _barrier(world)
    e2e_s = _max_over_ranks(time.perf_counter() - w0, dev, world)
    e2e_value = n_total * e2e_steps / e2e_s
    h2d = n * na * w
    d2h = n * (9 * w + 1)     # obs + done; the reward is identically 0 and is not shipped (the host array is zero-filled once)
    e2e_pieces = _lib.load().mvrl_host_chunk_count(n, args.e2e_chunks)
    del env, acts, h_act, leg["env"], leg["acts"]

    fp32_peak = _lib.measure_fma_peak(_lib.F32, local_rank)   # K6, measured now on this GPU (every rank: keeps the ranks in step)
    fp64_peak = _lib.measure_fma_peak(_lib.F64, local_rank, iters=1024)
    fp_peak = fp64_peak if args.dtype == "f64" else fp32_peak

    # ---- the other configurations, a few seconds in total ---------------------------------------------------
    extra, strong_leg = {}, None
    if not args.no_extra:
        xs, xw = args.extra_steps, 5
        if world > 1 and not strong:   # config 3 as written: 1 Mi environments IN TOTAL
            lo, hi = shard_range(ENVS_TOTAL_STRONG, rank, world)
            sl = rov6_leg(dev, rank, world, hi - lo, mode, args.dtype, n_sub, max(xs, 200), xw, env_id0=lo, stats=False, groups=max(0, args.stream_groups))
            sv = ENVS_TOTAL_STRONG / (sl["ms_per_step"] * 1e-3)
            strong_leg = {"value": sv, "unit": UNIT, "envs_total": ENVS_TOTAL_STRONG, "envs_per_gpu": hi - lo, "ms_per_step": sl["ms_per_step"],
                          "stream_groups": sl["stream_groups"], "stream_groups_tried_ms_per_step": sl["stream_groups_tried_ms_per_step"],
                          "steps": sl["steps"], "efficiency_vs_one_gpu_with_all_envs": sv / (value / world) / world,
                          "note": "one GPU stepping all 1 Mi environments = the per-GPU rate of the weak headline (value / n_gpus)", "l2": sl["l2"]}
        if world == 1 and (mode, args.dtype, n_sub, n) == ("rpm", "f32", N_SUB, ENVS_PER_GPU):
            big = ENVS_PER_GPU
            extra["setpoint_f32"] = leg_summary(rov6_leg(dev, rank, world, big, "setpoint", "f32", N_SUB, xs, xw, stats=False, groups=0), fp32_peak)
            extra["force_f32"] = leg_summary(rov6_leg(dev, rank, world, big, "force", "f32", N_SUB, xs, xw, stats=False, groups=0), fp32_peak)
            extra["rpm_f64"] = leg_summary(rov6_leg(dev, rank, world, big, "rpm", "f64", N_SUB, xs, xw, stats=False, groups=0), fp64_peak)
            extra["setpoint_f64"] = leg_summary(rov6_leg(dev, rank, world, big // 4, "setpoint", "f64", N_SUB, max(10, xs // 4), 3, stats=False), fp64_peak)
            extra["rpm_f32_nsub1"] = leg_summary(rov6_leg(dev, rank, world, big, "rpm", "f32", 1, xs, xw, stats=False), fp32_peak)
            extra["rpm_f32_nsub4"] = leg_summary(rov6_leg(dev, rank, world, big, "rpm", "f32", 4, xs, xw, stats=False), fp32_peak)
            extra["config2_4096_envs_f64_rpm"] = leg_summary(rov6_leg(dev, rank, world, 4096, "rpm", "f64", N_SUB, 4 * xs, xw, stats=False), fp64_peak)
            extra["single_gpu_shards_rpm_f32"] = {}
            for div in (2, 4, 8, 16):
                sl = rov6_leg(dev, rank, world, big // div, "rpm", "f32", N_SUB, 4 * xs, xw, stats=False, groups=0)
                extra["single_gpu_shards_rpm_f32"][str(big // div)] = {"value": sl["rate_per_gpu"], "ms_per_step": sl["ms_per_step"],
                                                                       "stream_groups": sl["stream_groups"],
                                                                       "stream_groups_tried_ms_per_step": sl["stream_groups_tried_ms_per_step"],
                                                                       "relative_to_1Mi_launch": sl["rate_per_gpu"] / (value / world), "l2": sl["l2"]}
            extra["config4_auv_262144_envs"] = auv_leg(dev, rank, world, 262144, 4 * xs, xw, groups=0)
            extra["rov3_setpoint_f32"] = rov3_leg(dev, rank, world, big, "setpoint", steps=xs, warmup=xw)
            extra["rov3_rpm_f32"] = rov3_leg(dev, rank, world, big, "rpm", steps=xs, warmup=xw)
        extra["config5_rollout"] = rollout_leg(dev, rank, world, 131072, args.rollout_len, rollouts=2, policy="fused")
        tl = rollout_leg(dev, rank, world, 131072, args.rollout_len, rollouts=2, policy="torch")
        extra["config5_rollout"]["pytorch_policy_baseline"] = {k: tl[k] for k in ("value", "ms_per_step", "env_share", "policy_and_bookkeeping_us_per_step", "policy")}
        r2g = rollout_leg(dev, rank, world, 131072, args.rollout_len, rollouts=2, policy="fused", groups=2)
        extra["config5_rollout"]["two_stream_groups"] = {k: r2g[k] for k in ("value", "ms_per_step", "launches_per_step", "stream_groups")}
        if world > 1:
            extra["config5_rollout"]["value_all_gpus"] = extra["config5_rollout"]["value"] * world

    if rank == 0:
        peaks, peak_src = measured_peaks()
        per_gpu_rate = n / (ms_per_step * 1e-3)
        flop, nbytes = flop_per_env_step(mode, n_sub), bytes_per_env_step(mode, w)
        ach_tflops = per_gpu_rate * flop / 1e12
        ach_gbs = per_gpu_rate * nbytes / 1e9
        ks = kernel_stats()
        kname = "rov6_step_%s_%s" % ("f64" if args.dtype == "f64" else "f32x2", mode)
        kst = ks.get("kernels", {}).get(kname)
        executed = (kst["flop_per_env_per_substep"] * n_sub + kst["flop_per_env_outside_loop"]) if kst else None
        traffic, traffic_src = (None, None)
        if (args.dtype, n) == ("f32", ENVS_PER_GPU) and n_sub == N_SUB:
            traffic, traffic_src = ncu_traffic(r"rov6_step_kernel<F2, %d" % {"rpm": 0, "force": 1, "setpoint": 2}[mode])
        roofline = {"bound": "fp64" if args.dtype == "f64" else "fp32", "achieved": ach_tflops, "peak": fp_peak, "unit": "TFLOP/s",
                    "frac": ach_tflops / fp_peak, "traffic": traffic,
                    "traffic_source": "dram__bytes_read.sum + dram__bytes_write.sum of one launch, ncu --set full: %s" % traffic_src,
                    "peak_source": "FMA-chain microbenchmark (mvrl_measure_fma_peak: operands from uniform registers) run on this GPU in this "
                    "process; nominal fp32 %.1f. With three distinct register operands FFMA sustains only 0.61 inst/clk/SMSP "
                    "(45.7 TFLOP/s, tools/ffma_regs.cu)" % NOMINAL_FP32_TFLOPS,
                    "fp32_peak_tflops": fp32_peak, "fp64_peak_tflops": fp64_peak, "flop_per_env_step": flop,
                    # what the shipped kernel executes, counted from its SASS at build time (tools/kernel_stats.py): folding / hoisting /
                    # anchored trig make it fewer flops than the frozen algorithmic count, hence frac ~ 1
                    "executed_flop_per_env_step": executed,
                    "executed_frac": (per_gpu_rate * executed / 1e12 / fp_peak) if executed else None,
                    "executed_source": ("SASS of %s: %d instructions per RK4 sub-step and thread (%d FMA-pipe, %d ALU-pipe), loop body %d bytes"
                                        % (kst["function"][:60], kst["loop_instructions_per_trip"], kst["loop_fma_pipe_instructions"],
                                           kst["loop_alu_pipe_instructions"], kst["loop_bytes"])) if kst else ks.get("error"),
                    "hbm": {"achieved": ach_gbs, "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": ach_gbs / peaks["hbm_gbs"],
                            "bytes_per_env_step": nbytes, "peak_source": peak_src}}
        cpu = None
        if not args.no_cpu and world == 1:   # the CPU baseline is reported at N = 1 only
            rate, secs, used = cpu_port_rate(CPU_SAMPLE_ENVS, args.cpu_steps)
            cpu = {"value": rate, "unit": UNIT, "cores": used, "kind": "port",
                   "sample": "%d envs x %d env steps of the same workload, C port of the reference loop, %d threads, %.1f s" %
                             (CPU_SAMPLE_ENVS, args.cpu_steps, used, secs),
                   # the reference-shaped loops next to it (BASELINE.md section 3), one core each, numpy ports of the reference code
                   "python_port_one_core": python_port_rate(2.0),
                   "as_shipped_rk45_pid_port_one_core": as_shipped_port_rate(2.0),
                   "legacy_auv_step_port_one_core": legacy_port_rate(2.0),
                   "variants": "python_port = the reference's forceModel / solve / J under the same RK4 x 8, one env at a time (its own loop "
                               "shape); as_shipped = env.step with scipy RK45 (rtol = atol = 1e-3) and the stateful PID, fixed set-point "
                               "(6DoF.py:545-557); legacy = AuvEnv.step (verySimpleAuv.py:264-410) with the config-4 field"}
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong" if strong else "weak", "vs_baseline": None,
                "dtype": args.dtype, "data": "synthetic",
                "config": {"workload": workload_name(n, mode, args.dtype, n_sub), "envs_per_gpu": n, "envs_total": n_total, "n_sub": n_sub,
                           "action_mode": mode, "fast_math": bool(args.fast_math), "cuda_graph": bool(args.graph),
                           # independent blocks of environments as chains of launches on their own streams (vec_tools.EnvBlocks): every
                           # environment takes exactly `steps` steps in the timed region, a block's k-th step waits for its own (k-1)-th only
                           "stream_groups": leg["stream_groups"], "stream_groups_tried_ms_per_step": leg["stream_groups_tried_ms_per_step"],
                           "two_envs_per_thread_ffma2": os.environ.get("MVRL_NO_X2", "0") != "1" and args.dtype == "f32", "parallelism": "env-sharded x%d, no collective on the step path" % world,
                           "l2": leg["l2"] + " (+ 4 rotating action batches)"},
                "roofline": roofline, "cpu_baseline": cpu,
                "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "steps": e2e_steps,
                        "chunks": e2e_pieces, "host_numa_node": numa_node, "gpu_launches_per_step": 3 * e2e_pieces,
                        "path": "BlueROV2Heavy6DoFVecEnv.step_host (mvrl_rov6_step_host): pinned host [N,8] actions -> pinned host obs/reward/done, "
                                "chunked H2D / transpose / fused step / transpose / D2H pipeline (obs by copy engine, done stored into the pinned host array by the transpose kernel; the always-zero reward does not travel)"},
                "gpu_launches": args.steps * leg["stream_groups"], "clocks": leg.get("clocks"), "episode_stats": leg.get("episode_stats")}
        tried = leg["stream_groups_tried_ms_per_step"]
        if tried and 1 in tried:   # the same workload with ONE launch per step (stream_groups = 1), from the calibration run
            line["single_launch_per_step"] = {"value": n_total / (tried[1] * 1e-3), "unit": UNIT, "ms_per_step": tried[1], "steps": min(args.steps, 40)}
        if strong_leg is not None:
            line["strong"] = strong_leg
        if extra:
            line["extra"] = extra
        emit(line)


def run_secondary(args, rank, local_rank, world):
    """--workload auv | rov3 | rollout: the secondary configuration as the headline of its own line."""
    import torch
    dev = torch.device("cuda", local_rank)
    if args.workload == "auv":
        n = args.envs if args.envs != ENVS_PER_GPU else 262144
        r = auv_leg(dev, rank, world, n, args.steps, args.warmup, field=args.field, graph=bool(args.graph), clocks=True, groups=max(0, args.stream_groups))
        metric, dtype = "legacy AuvEnv env-steps/sec", "f32"
        cfg = {"workload": "auv_step fp32: legacy verySimpleAuv, %d envs/GPU, field [2000,41,61,2] (%s), a~U(-1,1)^3" % (n, args.field),
               "cuda_graph": bool(args.graph), "stream_groups": r["stream_groups"], "stream_groups_tried_ms_per_step": r["stream_groups_tried_ms_per_step"], "smem_staged_gather": os.environ.get("MVRL_AUV_NO_STAGE", "0") != "1", "l2": r["l2"]}
        extra = {"roofline": {"bound": "hbm", "achieved": r["hbm_gbs"], "peak": r["hbm_gbs"] / r["frac_of_hbm_peak"], "unit": "GB/s",
                              "frac": r["frac_of_hbm_peak"], "traffic": None, "bytes_per_env_step": r["bytes_per_env_step"],
                              "gathered_bytes_per_env_step_from_l2": 64, "peak_source": r["peak_source"]}}
        launches = args.steps * r["stream_groups"]
    elif args.workload == "rov3":
        mode = "rpm" if args.action_mode == "rpm" else "setpoint"
        r = rov3_leg(dev, rank, world, args.envs, mode, args.n_sub, args.steps, args.warmup, clocks=True)
        metric, dtype = "BlueROV2 3DoF env-steps/sec", "f32"
        cfg = {"workload": "rov3_step fp32: BlueROV2 Heavy 3DoF, %d envs/GPU, %s actions, dt=%.1f as nSub=%d RK4, maxSteps=%d auto-reset"
                           % (args.envs, mode, DT, args.n_sub, MAX_STEPS)}
        extra, launches = {}, args.steps
    else:
        n = args.envs if args.envs != ENVS_PER_GPU else 131072
        rollouts = max(2, args.steps // args.rollout_len)
        r = rollout_leg(dev, rank, world, n, args.rollout_len, rollouts, args.n_sub, clocks=True, policy=args.policy, groups=max(1, args.stream_groups))
        metric, dtype = "6DoF rollout collection env-steps/sec (policy included)", "f32 env; policy bf16 operands / fp32 accumulate (fused) or TF32 (torch)"
        cfg = {"workload": "rollout: 6DoF set-point env + MLP 9-128-128-128-6 GELU Gaussian policy, %d envs/GPU, %d-step rollouts, "
                           "nSub=%d, CUDA-graph replay, stats all-reduce per rollout" % (n, args.rollout_len, args.n_sub)}
        extra = {k: r[k] for k in ("env_share", "env_us_per_step", "policy_and_bookkeeping_us_per_step", "flop_per_env_step", "policy", "policy_impl",
                                   "launches_per_step", "stats_allreduce", "stream_groups")}
        launches = rollouts * args.rollout_len
    if rank == 0:
        line = {"metric": metric, "value": world * r["value"], "unit": UNIT, "n_gpus": world, "steps": r.get("steps", launches), "warmup": args.warmup,
                "ms_per_step": r["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": dtype,
                "data": "synthetic", "config": cfg, "gpu_launches": launches, "clocks": r.get("clocks"), "episode_stats": r.get("episode_stats")}
        line.update(extra)
        emit(line)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=1000)
    ap.add_argument("--warmup", type=int, default=50)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="weak: --envs environments per GPU (headline); strong: 1 048 576 environments in total, sharded over the GPUs")
    ap.add_argument("--envs", type=int, default=ENVS_PER_GPU, help="environments per GPU")
    ap.add_argument("--fast-math", type=int, default=0)
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-extra", action="store_true", help="skip the short legs of the other configurations (the `extra` / `strong` keys)")
    ap.add_argument("--extra-steps", type=int, default=50, help="timed steps of each 1 Mi-env extra leg")
    ap.add_argument("--cpu-steps", type=int, default=100)
    ap.add_argument("--e2e-chunks", type=int, default=0, help="pieces of the host-buffer pipeline; 0 = the library's default")
    ap.add_argument("--action-mode", default="rpm", choices=["rpm", "force", "setpoint"], help="default rpm = BASELINE config 3")
    ap.add_argument("--dtype", default="f32", choices=["f32", "f64"])
    ap.add_argument("--n-sub", type=int, default=N_SUB)
    ap.add_argument("--workload", default="rov6", choices=["rov6", "rov3", "auv", "rollout"],
                    help="rov6 = BASELINE config 3 (the metric); rov3 = the 3DoF env at scale; auv = config 4; rollout = config 5")
    ap.add_argument("--field", default="modes", choices=["modes", "noise"], help="auv: synthetic turbulence stand-in")
    ap.add_argument("--rollout-len", type=int, default=128)
    ap.add_argument("--policy", default="fused", choices=["fused", "torch"], help="rollout: the fused tensor-core actor or the PyTorch baseline")
    ap.add_argument("--max-steps", type=int, default=MAX_STEPS, help="episode length (diagnostics; default = the reference's 250)")
    ap.add_argument("--graph", type=int, default=1, help="1: the K timed launches are replayed as one CUDA graph; 0: K separate launches")
    ap.add_argument("--bind-numa", type=int, default=1, help="1: bind each rank to the CPUs of its GPU's NUMA node (host buffers of the e2e leg)")
    ap.add_argument("--stream-groups", type=int, default=0,
                    help="step the environments of a rank as this many independent blocks, each a chain of launches on its own stream "
                         "(vec_tools.EnvBlocks); 1 = one launch per step; 0 (default) = rov6: the fastest of 1 / 2 / 4 / 8 by a short calibration run, rollout: 1")
    ap.add_argument("--no-stats", action="store_true", help="diagnostics: do not accumulate episode statistics in the step kernel")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one returned (obs, reward, done) and the state as DIR/<name>.npy, "
                         "for rank 0's environments or a fixed sample of %d of them (rov6 workload)" % DUMP_SAMPLE_ENVS)
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.workload != "rov6"):
        ap.error("--dump-outputs writes the outputs of the rov6 workload's GPU path (--impl ours --workload rov6)")
    args.warmup = max(args.warmup, 3)
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
    capture_stdout()
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    import torch
    import torch.distributed as dist
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    try:
        if args.workload == "rov6":
            run_ours(args, rank, local_rank, world)
        else:
            run_secondary(args, rank, local_rank, world)
    finally:
        if world > 1:
            dist.destroy_process_group()


if __name__ == "__main__":
    main()
