"""Cost of the squashed Gaussian head (SB3 SAC / TQC Actor) against the fixed-std head of the fused rollout actor, and of
the fp32 precision against the bf16 one.

    python tools/policy_heads_bench.py [--out profiles/<name>.json]

* Actor kernel time: mvrl_policy_act for the fixed head, the squashed head and the squashed head with action noise, each
  in both precisions (bf16, the default, and fp32: the "_fp32" entries), at 131 072 and 1 Mi environments (6DoF shapes:
  obs 9, act 6), next to "torch_fp32": the same network and squashed head evaluated by PyTorch in fp32 (no TF32,
  nn.GELU(), SB3's sample and log-prob) on the same feature-major buffers.  CUDA events around blocks of launches (one
  CUDA graph per block); the variants alternate block by block in one process, so that clock and neighbour drift hit
  all alike; 1000 timed launches per variant and size after a warm-up.  Inputs are L2-resident (38 MB of observations
  at 1 Mi), as in a rollout, where the step kernel has just written them.
* Rollout: T = 128 steps of (actor, env.step_async) on the 6DoF set-point env's own buffers at 131 072 environments,
  captured as one CUDA graph per fused variant and replayed alternately; env-steps/s with the policy included.

Prints one JSON line (with the device name, power limit and max SM clock, read with a read-only nvidia-smi query) and
writes it to --out when given."""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_info(index):
    try:
        q = subprocess.run(["nvidia-smi", "-i", str(index), "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=60).stdout.strip()
        name, power, clock = [s.strip() for s in q.split(",")]
        return {"nvidia_smi_name": name, "power_limit": power, "sm_max_clock": clock}
    except Exception as e:   # the timing does not depend on it; say why it is missing
        return {"nvidia_smi_error": str(e)}


def make_policies(dev, seed=1234):
    from marinevehiclereinforcementlearning_b200 import MlpGaussianPolicy, SquashedGaussianPolicy
    pols = {}
    for prec, suffix in (("bf16", ""), ("fp32", "_fp32")):
        pols["fixed" + suffix] = MlpGaussianPolicy(9, 6, device=dev, seed=seed, precision=prec)
        pols["squashed" + suffix] = SquashedGaussianPolicy(9, 6, device=dev, seed=seed, precision=prec)
        pols["squashed_noise" + suffix] = SquashedGaussianPolicy(9, 6, device=dev, seed=seed, action_noise_std=0.1, precision=prec)
    return pols


class TorchFp32Actor:
    """The squashed actor as PyTorch evaluates it for SB3 in fp32: Linear + nn.GELU() x 3, mu / log_std heads, log_std
    clamped to [-20, 2], a = tanh(mu + exp(log_std) eps) with torch.randn noise, the log-prob with the tanh Jacobian; reads
    and writes the same feature-major buffers as the fused actor (the transposes are part of its cost)."""

    def __init__(self, pol):
        import torch
        p = {k: v.to(pol.device) for k, v in pol.state_dict().items()}
        self.layers = [(p["latent_pi.%d.weight" % i], p["latent_pi.%d.bias" % i]) for i in (0, 2, 4)]
        self.mu, self.ls = (p["mu.weight"], p["mu.bias"]), (p["log_std.weight"], p["log_std.bias"])
        self.gelu = torch.nn.GELU()

    def act_into(self, obs_fm, act_fm, n, logp=None, step=None):
        import torch
        h = obs_fm[:, :n].T
        for W, b in self.layers:
            h = self.gelu(torch.nn.functional.linear(h, W, b))
        mu = torch.nn.functional.linear(h, *self.mu)
        log_std = torch.nn.functional.linear(h, *self.ls).clamp(-20.0, 2.0)
        std = log_std.exp()
        u = mu + std * torch.randn_like(mu)
        a = torch.tanh(u)
        act_fm[:, :n] = a.T
        if logp is not None:
            lp = torch.distributions.Normal(mu, std, validate_args=False).log_prob(u).sum(1) - torch.log(1.0 - a * a + 1e-6).sum(1)
            logp[:n] = lp


def actor_times(dev, pols, n, rounds, block, warmup):
    """us per launch of each head: median and min over `rounds` blocks of `block` launches.  A block is one CUDA graph of
    `block` launches: a launch from Python costs about as much host time as the kernel runs at 131 072 environments."""
    import torch
    ld = n
    obs = torch.rand((9, ld), device=dev) * 2 - 1
    act, logp = torch.empty((6, ld), device=dev), torch.empty((ld,), device=dev)
    side = torch.cuda.Stream(device=dev)
    graphs = {}
    for name, p in pols.items():
        for k in range(warmup):
            p.act_into(obs, act, n, logp=logp, step=k)
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        side.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(side):
            with torch.cuda.graph(g, stream=side):
                for k in range(block):
                    p.act_into(obs, act, n, logp=logp, step=k)
        torch.cuda.current_stream(dev).wait_stream(side)
        g.replay()
        graphs[name] = g
    torch.cuda.synchronize()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(rounds * len(pols))]
    order = []
    i = 0
    for r in range(rounds):
        for name, g in graphs.items():
            e0, e1 = ev[i]
            e0.record()
            g.replay()
            e1.record()
            order.append((name, i))
            i += 1
    torch.cuda.synchronize()
    per = {name: [] for name in pols}
    for name, j in order:
        per[name].append(1e3 * ev[j][0].elapsed_time(ev[j][1]) / block)
    return {name: {"us_median": statistics.median(v), "us_min": min(v), "launches": rounds * block} for name, v in per.items()}


def rollout_rates(dev, pols, n, T, replays, rounds):
    """env-steps/s of T-step rollouts (actor + 6DoF set-point step, one CUDA graph per head), heads alternated."""
    import torch
    from marinevehiclereinforcementlearning_b200 import BlueROV2Heavy6DoFVecEnv
    env = BlueROV2Heavy6DoFVecEnv(n, action_mode="setpoint", dtype=torch.float32, device=dev, seed=1234, auto_reset=True, record_terminal_obs=False)
    env.reset()
    logp = torch.empty((T, env.ld), device=dev)
    graphs = {}
    side = torch.cuda.Stream(device=dev)
    for name, p in pols.items():
        def rollout(p=p):
            for t in range(T):
                p.act(env, logp=logp[t], step=t)
                env.step_async()
        rollout()
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        side.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(side):
            with torch.cuda.graph(g, stream=side):
                rollout()
        torch.cuda.current_stream(dev).wait_stream(side)
        g.replay()
        graphs[name] = g
    torch.cuda.synchronize()
    per = {name: [] for name in graphs}
    for r in range(rounds):
        for name, g in graphs.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(replays):
                g.replay()
            e1.record()
            e1.synchronize()
            per[name].append(e0.elapsed_time(e1) * 1e-3 / (replays * T))   # s per step
    assert bool(torch.isfinite(env.systemState).all()) and bool(torch.isfinite(logp[:, :n]).all())
    return {name: {"env_steps_per_s": n / statistics.median(v), "us_per_step_median": 1e6 * statistics.median(v),
                   "us_per_step_min": 1e6 * min(v)} for name, v in per.items()}


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--device", type=int, default=0)
    ap.add_argument("--rounds", type=int, default=20, help="alternation rounds (actor and rollout)")
    ap.add_argument("--block", type=int, default=50, help="actor launches per timed block")
    ap.add_argument("--warmup", type=int, default=50)
    ap.add_argument("--rollout-len", type=int, default=128)
    ap.add_argument("--replays", type=int, default=4, help="rollout graph replays per timed block")
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    args = ap.parse_args()
    import torch
    from marinevehiclereinforcementlearning_b200 import _lib
    _lib.require_cuda()
    dev = torch.device("cuda", args.device)
    torch.cuda.set_device(dev)
    torch.backends.cuda.matmul.allow_tf32 = False   # the PyTorch baseline in true fp32
    pols = make_policies(dev)
    timed = dict(pols, torch_fp32=TorchFp32Actor(pols["squashed"]))
    res = {"tool": "policy_heads_bench", "device": torch.cuda.get_device_name(dev), **gpu_info(args.device),
           "obs_dim": 9, "act_dim": 6, "actor_us_per_launch": {}, "rollout": {}}
    for n in (131072, 1 << 20):
        t = actor_times(dev, timed, n, args.rounds, args.block, args.warmup)
        med = lambda k: t[k]["us_median"]
        t["squashed_over_fixed"] = med("squashed") / med("fixed") - 1.0
        t["squashed_noise_over_fixed"] = med("squashed_noise") / med("fixed") - 1.0
        for k in ("fixed", "squashed", "squashed_noise"):
            t[k + "_fp32_over_bf16"] = med(k + "_fp32") / med(k)
        t["torch_fp32_over_squashed_fp32"] = med("torch_fp32") / med("squashed_fp32")
        res["actor_us_per_launch"][str(n)] = t
    n = 131072
    res["rollout"] = {"envs": n, "T": args.rollout_len, "env": "BlueROV2Heavy6DoFVecEnv set-point fp32",
                      **rollout_rates(dev, pols, n, args.rollout_len, args.replays, args.rounds)}
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
