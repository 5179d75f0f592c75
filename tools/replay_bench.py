"""Cost of the device replay buffer (vec_tools.ReplayBuffer: replay_add_kernel, replay_sample_kernel) against a PyTorch
restatement of the same semantics, and its share of a SAC-shaped collection loop.

    python tools/replay_bench.py [--out profiles/replay_b200.json]

* add, at 131 072 and 1 Mi environments, for the 6DoF shapes (obs 9, act 6) and the AUV shapes (obs 11, act 3), fp32, a
  buffer of 2^23 transitions (64 / 8 slots).  The inputs are env-shaped feature-major buffers [k, ld] with random contents
  and 1 / 64 of the environments done.  The PyTorch restatement: clone of the staging row, torch.where against the terminal
  observations, transposed copies into slot `pos` (index_copy_ with the device-side pos), staging refresh, pos update on the
  device.  Before timing, three adds of each from the same state are compared bitwise (storage, staging row, pos and number of adds).
* sample, B = 256, 4096, 65 536 from the full 6DoF-shaped buffer at 131 072 environments, against torch.randint for slot and
  environment plus the five advanced-indexing gathers and dones * (1 - timeouts).
  Both sides of both comparisons run as CUDA graphs of --calls calls, timed with CUDA events, the two alternating round by
  round; the figure is device time per call (median of the rounds).  At 131 072 environments the env buffers an add reads
  (about 13 MB) stay in the 126 MB L2 from one call to the next, as they do in a collection loop right after the env step
  wrote them; every add writes a new slot.  At 1 Mi environments the working set exceeds L2.
* bytes: what the algorithm moves, computed from the shapes (add: read staging, obs, action, reward, done; write obs,
  next_obs, action, reward, done, timeout, staging; sample: the gathered rows and the outputs), and the ratio of bytes / time
  to the 7.7 TB/s data-sheet HBM rate of a B200 - a fraction of the data-sheet rate, not a measured peak.
* loop: 131 072 environments of the 6DoF set-point env, T = 128 steps, bf16 squashed head, each variant one CUDA graph:
  act + step; act + step + add; act + step + add + sample(4096).  The variants alternate round by round; env-steps/s from
  the median round.

Prints one JSON line (with the device name, power limit and max SM clock, from a read-only nvidia-smi query) and writes it to
--out."""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

HBM_DATASHEET = 7.7e12


def gpu_info(index):
    try:
        q = subprocess.run(["nvidia-smi", "-i", str(index), "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=60).stdout.strip()
        name, power, clock = [s.strip() for s in q.split(",")]
        return {"nvidia_smi_name": name, "power_limit": power, "sm_max_clock": clock}
    except Exception as e:   # the timing does not depend on it; say why it is missing
        return {"nvidia_smi_error": str(e)}


class EnvBuffers:
    """The env attributes ReplayBuffer reads, filled with random values (feature-major [k, ld], as the envs hold them)."""

    def __init__(self, torch, n, obs_dim, act_dim, dev, seed=0):
        g = torch.Generator(device=dev).manual_seed(seed)
        self.num_envs, self.lenObs, self.lenAction, self.dtype, self.device = n, obs_dim, act_dim, torch.float32, dev
        self.ld, self.auto_reset = (n + 31) // 32 * 32, True
        r = lambda k: torch.rand((k, self.ld), generator=g, device=dev)
        self._obs, self._terminal_obs, self._action = r(obs_dim), r(obs_dim), r(act_dim)
        self._reward = torch.rand(self.ld, generator=g, device=dev)
        self._done = (torch.rand(self.ld, generator=g, device=dev) < 1 / 64).to(torch.uint8)


class TorchReplay:
    """The same add / sample semantics in PyTorch operations (what a user would write without the kernels)."""

    def __init__(self, torch, buf):
        self.t, self.b = torch, buf
        self.st = {k: getattr(buf, k).clone() for k in buf._STATE}

    def add(self, env):
        t, st, n = self.t, self.st, self.b.n_envs
        obs_t = st["last_obs"][:, :n].clone()
        nxt = t.where(env._done[:n].bool(), env._terminal_obs[:, :n], env._obs[:, :n])
        pos = st["cursor"][0:1]
        st["observations"].index_copy_(0, pos, obs_t.T.unsqueeze(0))
        st["next_observations"].index_copy_(0, pos, nxt.T.unsqueeze(0))
        st["actions"].index_copy_(0, pos, env._action[:, :n].T.unsqueeze(0))
        st["rewards"].index_copy_(0, pos, env._reward[:n].unsqueeze(0))
        st["dones"].index_copy_(0, pos, env._done[:n].unsqueeze(0))
        st["timeouts"].index_fill_(0, pos, 0)
        st["last_obs"].copy_(env._obs)
        st["cursor"][1:2].add_(1)
        st["cursor"][0:1].copy_(t.remainder(pos + 1, self.b.buffer_size))

    def sample(self, batch, size):
        t, st, dev = self.t, self.st, self.b.device
        slot = t.randint(0, size, (batch,), device=dev)
        env = t.randint(0, self.b.n_envs, (batch,), device=dev)
        dones = st["dones"][slot, env].float() * (1 - st["timeouts"][slot, env].float())
        return (st["observations"][slot, env], st["actions"][slot, env], st["next_observations"][slot, env], dones[:, None],
                st["rewards"][slot, env][:, None])


def graph_of(torch, fn, calls):
    fn()
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for _ in range(calls):
            fn()
    g.replay()
    torch.cuda.synchronize()
    return g


def time_alternating(torch, graphs, calls, rounds):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    times = {k: [] for k in graphs}
    for _ in range(rounds):
        for name, g in graphs.items():
            e0.record()
            g.replay()
            e1.record()
            e1.synchronize()
            times[name].append(e0.elapsed_time(e1) * 1e3 / calls)
    return {k: statistics.median(v) for k, v in times.items()}


def bench_add(torch, dev, n, obs_dim, act_dim, calls, rounds):
    from marinevehiclereinforcementlearning_b200 import ReplayBuffer
    env = EnvBuffers(torch, n, obs_dim, act_dim, dev)
    buf = ReplayBuffer(2 ** 23, env, seed=0)
    buf.on_reset(env)
    ref = TorchReplay(torch, buf)
    for _ in range(3):
        buf.add(env)
        ref.add(env)
    torch.cuda.synchronize()
    same = all(torch.equal(getattr(buf, k), ref.st[k]) for k in buf._STATE if k != "cursor") and torch.equal(buf.cursor[:2], ref.st["cursor"][:2])
    graphs = {"kernel": graph_of(torch, lambda: buf.add(env), calls), "torch": graph_of(torch, lambda: ref.add(env), calls)}
    us = time_alternating(torch, graphs, calls, rounds)
    nbytes = n * (4 * (obs_dim + obs_dim + act_dim + 1) + 1 + 4 * (3 * obs_dim + act_dim + 1) + 2)
    return {"num_envs": n, "obs_dim": obs_dim, "act_dim": act_dim, "slots": buf.buffer_size, "outputs_bitwise_equal": same,
            "kernel_us": us["kernel"], "torch_us": us["torch"], "speedup": us["torch"] / us["kernel"], "bytes": nbytes,
            "kernel_fraction_of_datasheet_hbm": nbytes / (us["kernel"] * 1e-6) / HBM_DATASHEET,
            "torch_fraction_of_datasheet_hbm": nbytes / (us["torch"] * 1e-6) / HBM_DATASHEET}


def bench_sample(torch, dev, n, batches, calls, rounds):
    from marinevehiclereinforcementlearning_b200 import ReplayBuffer
    env = EnvBuffers(torch, n, 9, 6, dev)
    buf = ReplayBuffer(2 ** 23, env, seed=0)
    buf.on_reset(env)
    for _ in range(buf.buffer_size + 1):
        buf.add(env)
    ref = TorchReplay(torch, buf)
    size = buf.size()
    out = []
    for B in batches:
        graphs = {"kernel": graph_of(torch, lambda: buf.sample(B), calls), "torch": graph_of(torch, lambda: ref.sample(B, size), calls)}
        us = time_alternating(torch, graphs, calls, rounds)
        nbytes = B * (2 * 4 * (9 + 9 + 6 + 1) + 2 + 4)
        out.append({"batch": B, "kernel_us": us["kernel"], "torch_us": us["torch"], "speedup": us["torch"] / us["kernel"], "bytes": nbytes,
                    "kernel_fraction_of_datasheet_hbm": nbytes / (us["kernel"] * 1e-6) / HBM_DATASHEET})
    return {"num_envs": n, "slots": buf.buffer_size, "batches": out}


def bench_loop(torch, dev, n, T, rounds):
    from marinevehiclereinforcementlearning_b200 import BlueROV2Heavy6DoFVecEnv, ReplayBuffer, SquashedGaussianPolicy
    env = BlueROV2Heavy6DoFVecEnv(n, action_mode="setpoint", dtype=torch.float32, device=dev, seed=3, auto_reset=True)
    env.reset()
    pol = SquashedGaussianPolicy(9, 6, device=dev, seed=1, action_noise_std=0.1, precision="bf16")
    buf = ReplayBuffer(2 ** 23, env, seed=0)
    buf.on_reset(env)

    def loop(add, sample):
        for t in range(T):
            pol.act(env, step=t)
            env.step_async()
            if add:
                buf.add(env)
            if sample:
                buf.sample(4096)

    variants = {"act_step": (False, False), "act_step_add": (True, False), "act_step_add_sample4096": (True, True)}
    graphs = {}
    for name, (a, s) in variants.items():
        loop(a, s)
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            loop(a, s)
        g.replay()
        graphs[name] = g
    torch.cuda.synchronize()
    us = time_alternating(torch, graphs, T, rounds)
    return {"num_envs": n, "T": T, "head": "squashed bf16", **{k + "_env_steps_per_s": n / (v * 1e-6) for k, v in us.items()},
            **{k + "_us_per_step": v for k, v in us.items()}}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "replay_b200.json"))
    ap.add_argument("--device", default="cuda:0")
    ap.add_argument("--rounds", type=int, default=15)
    ap.add_argument("--calls", type=int, default=50)
    ap.add_argument("--steps", type=int, default=128)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("replay_bench needs a CUDA device")
    dev = torch.device(args.device)
    res = {"what": "device replay buffer (SB3 ReplayBuffer semantics) vs a PyTorch restatement; fp32", "device": gpu_info(dev.index or 0),
           "torch": torch.__version__, "rounds": args.rounds, "calls_per_graph": args.calls,
           "hbm_datasheet_bytes_per_s": HBM_DATASHEET,
           "add": [bench_add(torch, dev, n, o, a, args.calls, args.rounds) for n in (131072, 1 << 20) for o, a in ((9, 6), (11, 3))],
           "sample": bench_sample(torch, dev, 131072, (256, 4096, 65536), args.calls, args.rounds),
           "loop": bench_loop(torch, dev, 131072, args.steps, args.rounds)}
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
