"""Time ``CriticTarget`` (one critic_target_kernel launch) against SB3 SAC / sb3_contrib TQC's target block restated in
PyTorch (fp32, TF32 off), eager and captured in a CUDA graph, with CUDA events; the three are alternated over several
rounds and the median per call is reported.  In the same run the kernel's target is checked against the PyTorch
restatement fed the kernel's eps, within the tolerance of tests/test_critic_target_gpu.py.

    python tools/critic_target_bench.py --out profiles/critic_target_b200.json

Writes one JSON file: the card's name and power limit, then one row per (shape, variant, batch size)."""
import argparse
import json
import math
import os
import statistics
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from marinevehiclereinforcementlearning_b200 import CriticTarget, SquashedGaussianPolicy  # noqa: E402
from marinevehiclereinforcementlearning_b200.vec_tools import ReplayBufferSamples  # noqa: E402

DEV = "cuda"
SHAPES = [(9, 6), (11, 3)]
VARIANTS = [("tqc", 2, 25, 2), ("tqc", 5, 25, 2), ("sac", 2, 1, 0)]
SIZES = [256, 4096, 65536]
GAMMA, ALPHA, TOL = 0.99, 0.2, 5e-5


def linear(g, fan_in, fan_out):
    return (torch.randn(fan_out, fan_in, generator=g) / math.sqrt(fan_in)).to(DEV), (torch.rand(fan_out, generator=g) * 0.6 - 0.3).to(DEV)


def networks(obs_dim, act_dim, n_critics, n_out, seed=0):
    g = torch.Generator().manual_seed(seed)
    actor = {}
    for i, fan_in in zip((0, 2, 4), (obs_dim, 128, 128)):
        actor["latent_pi.%d.weight" % i], actor["latent_pi.%d.bias" % i] = linear(g, fan_in, 128)
    actor["mu.weight"], actor["mu.bias"] = linear(g, 128, act_dim)
    actor["log_std.weight"], actor["log_std.bias"] = linear(g, 128, act_dim)
    critic = {}
    for i in range(n_critics):
        for j, fan_in, fan_out in ((0, obs_dim + act_dim, 128), (2, 128, 128), (4, 128, 128), (6, 128, n_out)):
            critic["qf%d.%d.weight" % (i, j)], critic["qf%d.%d.bias" % (i, j)] = linear(g, fan_in, fan_out)
    return actor, critic


def torch_target(actor, critic, batch, ent_coef, kind, n_critics, drop, eps=None, with_logp=False):
    """SB3's block in PyTorch fp32: action_log_prob (th.randn for eps unless given), the critics, sort / min, the tail."""
    gelu = torch.nn.functional.gelu
    x = batch.next_observations
    h = x
    for j in (0, 2, 4):
        h = gelu(torch.nn.functional.linear(h, actor["latent_pi.%d.weight" % j], actor["latent_pi.%d.bias" % j]))
    mu = torch.nn.functional.linear(h, actor["mu.weight"], actor["mu.bias"])
    ls = torch.clamp(torch.nn.functional.linear(h, actor["log_std.weight"], actor["log_std.bias"]), -20.0, 2.0)
    std = ls.exp()
    u = mu + std * (torch.randn_like(mu) if eps is None else eps)
    a = torch.tanh(u)
    logp = (-((u - mu) ** 2) / (2 * std * std) - ls - math.log(math.sqrt(2 * math.pi))).sum(1) - torch.log(1 - a * a + 1e-6).sum(1)
    xa = torch.cat([x, a], 1)
    qs = []
    for i in range(n_critics):
        q = xa
        for j in (0, 2, 4):
            q = gelu(torch.nn.functional.linear(q, critic["qf%d.%d.weight" % (i, j)], critic["qf%d.%d.bias" % (i, j)]))
        qs.append(torch.nn.functional.linear(q, critic["qf%d.6.weight" % i], critic["qf%d.6.bias" % i]))
    q = torch.stack(qs, 1)
    if kind == "tqc":
        q, _ = torch.sort(q.reshape(q.shape[0], -1))
        q = q[:, :n_critics * (q.shape[1] // n_critics - drop)]
    else:
        q, _ = torch.min(torch.cat(qs, 1), dim=1, keepdim=True)
    target = batch.rewards + (1 - batch.dones) * GAMMA * (q - ent_coef * logp.reshape(-1, 1))
    return (target, logp) if with_logp else target


def time_calls(fn, reps):
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    for _ in range(reps):
        fn()
    e.record()
    e.synchronize()
    return s.elapsed_time(e) * 1e3 / reps   # us per call


def card():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=60).stdout.strip().splitlines()[0]
    except Exception as exc:   # the card's name from torch is still recorded
        q = "nvidia-smi unavailable: %s" % exc
    return name, q


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--min-ms", type=float, default=20.0, help="GPU time per timed window")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this benchmark measures the GPU and has nothing to report without one")
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    name, smi = card()
    rows = []
    for obs_dim, act_dim in SHAPES:
        for kind, n_critics, n_q, drop in VARIANTS:
            actor_sd, critic_sd = networks(obs_dim, act_dim, n_critics, n_q)
            pol = SquashedGaussianPolicy(obs_dim, act_dim, device=DEV, precision="fp32").load_state_dict(actor_sd, share=True)
            tgt = CriticTarget(pol, kind=kind, n_critics=n_critics, n_quantiles=n_q, top_quantiles_to_drop_per_net=drop, gamma=GAMMA)
            tgt.load_state_dict(critic_sd, share=True)
            alpha = torch.tensor([ALPHA], device=DEV)
            for b in SIZES:
                g = torch.Generator(device=DEV).manual_seed(b)
                obs = torch.rand((b, obs_dim), generator=g, device=DEV) * 2 - 1
                batch = ReplayBufferSamples(obs, None, obs, (torch.rand((b, 1), generator=g, device=DEV) < 0.3).float(),
                                            torch.rand((b, 1), generator=g, device=DEV) * 2 - 1)
                # agreement in this run: the kernel against the PyTorch restatement fed the kernel's eps
                eps = torch.empty((b, act_dim), device=DEV)
                y = tgt(batch, alpha, eps=eps)
                ref, logp = torch_target(actor_sd, critic_sd, batch, alpha, kind, n_critics, drop, eps=eps, with_logp=True)
                lp_scale = max(1.0, float(logp.abs().max()))
                err = float((y - ref).abs().max()) / (TOL * max(1.0, float(ref.abs().max())) + GAMMA * ALPHA * 4 * TOL * act_dim * lp_scale)
                assert err <= 1.0, (obs_dim, act_dim, kind, n_critics, b, err)
                kern = lambda: tgt(batch, alpha)
                eager = lambda: torch_target(actor_sd, critic_sd, batch, alpha, kind, n_critics, drop)
                side = torch.cuda.Stream()
                side.wait_stream(torch.cuda.current_stream())
                with torch.cuda.stream(side):
                    for _ in range(3):
                        eager()
                torch.cuda.current_stream().wait_stream(side)
                graph = torch.cuda.CUDAGraph()
                with torch.cuda.graph(graph):
                    eager()
                fns = {"kernel": kern, "torch_eager": eager, "torch_graph": graph.replay}
                reps = {}
                for k, fn in fns.items():   # warm-up and a window of at least --min-ms
                    t = time_calls(fn, 3)
                    reps[k] = max(10, int(args.min_ms * 1e3 / max(t, 1.0)))
                times = {k: [] for k in fns}
                for _ in range(args.rounds):
                    for k, fn in fns.items():
                        times[k].append(time_calls(fn, reps[k]))
                row = {"obs_dim": obs_dim, "act_dim": act_dim, "kind": kind, "n_critics": n_critics, "n_quantiles": n_q, "drop": drop,
                       "batch": b, "rel_err_vs_torch_fp32": err}
                for k in fns:
                    row[k + "_us"] = statistics.median(times[k])
                    row[k + "_us_spread"] = [min(times[k]), max(times[k])]
                row["speedup_vs_eager"] = row["torch_eager_us"] / row["kernel_us"]
                row["speedup_vs_graph"] = row["torch_graph_us"] / row["kernel_us"]
                rows.append(row)
                print(json.dumps(row), flush=True)
                del graph
    out = {"card": name, "nvidia_smi": smi, "tf32": False, "rounds": args.rounds, "unit": "us per call, median over rounds",
           "rows": rows}
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
