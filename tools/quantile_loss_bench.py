"""Time ``quantile_huber_loss`` (quantile_huber_kernel + its one-block reduction, forward and backward) against sb3_contrib's
function in PyTorch fp32 with autograd, each eager and captured in a CUDA graph, with CUDA events; the four are alternated over
several rounds and the median per call is reported, with each one's peak memory; the kernel path is timed both from Python
and replayed from a CUDA graph, so per-call host overhead and device time are told apart.  In the same run both results are checked
against the fp64 restatement within the bounds of tests/test_quantile_loss_gpu.py.  Then one whole TQC critic update
(CriticTarget, critic forward, loss, backward, Adam) is timed with either loss, eager and as a graph, which gives the loss's
share of a gradient step.

    python tools/quantile_loss_bench.py --out profiles/quantile_loss_b200.json

Writes one JSON file: the card's name and power limit, then one row per (configuration, batch size)."""
import argparse
import copy
import json
import math
import os
import statistics
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from marinevehiclereinforcementlearning_b200 import CriticTarget, SquashedGaussianPolicy, quantile_huber_loss  # noqa: E402
from marinevehiclereinforcementlearning_b200.vec_tools import ReplayBufferSamples  # noqa: E402
# sb3_contrib's function as published, TQC's critic module and the fp64 restatement, shared with the tests
from test_quantile_loss_cpu import Critics, pair_count, restatement_sums  # noqa: E402
from test_quantile_loss_cpu import quantile_huber_loss as sb3_quantile_huber_loss  # noqa: E402

DEV = "cuda"
CONFIGS = [(2, 25, 2), (5, 25, 2)]   # TQC (n_critics, n_quantiles, top_quantiles_to_drop_per_net)
SIZES = [256, 4096, 65536]
OBS_DIM, ACT_DIM = 9, 6
U = 2.0 ** -24


def fp64_reference(cur, tgt, chunk=4096):
    """(loss, grad, sum_j |w h'| / N) of sum_over_quantiles=False in fp64, summed over chunks of rows."""
    parts = [restatement_sums(cur[lo:lo + chunk], tgt[lo:lo + chunk]) for lo in range(0, cur.shape[0], chunk)]
    n = pair_count(cur, tgt, False)
    return sum(p[0] for p in parts) / n, -torch.cat([p[1] for p in parts]) / n, torch.cat([p[2] for p in parts]) / n


def agreement(loss, grad, ref, t, rows):
    l64, g64, gabs = ref
    el = abs(float(loss) - l64) / ((t + math.log2(rows) + 8) * U * l64)
    eg = float(((grad.double() - g64).abs() / ((t + 8) * U * gabs).clamp(min=1e-300)).max())
    return el, eg


def time_calls(fn, reps):
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    for _ in range(reps):
        fn()
    e.record()
    e.synchronize()
    return s.elapsed_time(e) * 1e3 / reps   # us per call


def peak_bytes(fn):
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    fn()
    torch.cuda.synchronize()
    return torch.cuda.max_memory_allocated() - base


def capture(fn, warm=3):
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(warm):
            fn()
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    before = torch.cuda.memory_allocated()
    with torch.cuda.graph(graph):
        out = fn()
    torch.cuda.synchronize()
    return graph, out, torch.cuda.memory_allocated() - before


def measure(fns, rounds, min_ms):
    reps = {}
    for k, fn in fns.items():   # warm-up and a window of at least min_ms
        t = time_calls(fn, 3)
        reps[k] = max(10, int(min_ms * 1e3 / max(t, 1.0)))
    times = {k: [] for k in fns}
    for _ in range(rounds):
        for k, fn in fns.items():
            times[k].append(time_calls(fn, reps[k]))
    row = {}
    for k in fns:
        row[k + "_us"] = statistics.median(times[k])
        row[k + "_us_spread"] = [min(times[k]), max(times[k])]
    return row


def card():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=60).stdout.strip().splitlines()[0]
    except Exception as exc:   # the card's name from torch is still recorded
        q = "nvidia-smi unavailable: %s" % exc
    return name, q


def loss_rows(args):
    rows = []
    for n_critics, nq, drop in CONFIGS:
        t = n_critics * (nq - drop)
        for b in SIZES:
            g = torch.Generator(device=DEV).manual_seed(b + t)
            cur = (torch.randn((b, n_critics, nq), generator=g, device=DEV) * 1.5).requires_grad_(True)
            tgt = torch.randn((b, 1, t), generator=g, device=DEV) * 1.5

            # a fresh leaf per call (no kernel): its gradient node is made on the stream the call runs on, eager or captured
            def kern():
                x = cur.detach().requires_grad_(True)
                return torch.autograd.grad(quantile_huber_loss(x, tgt, sum_over_quantiles=False), x)[0]

            def eager():
                x = cur.detach().requires_grad_(True)
                return torch.autograd.grad(sb3_quantile_huber_loss(x, tgt, sum_over_quantiles=False), x)[0]

            ref = fp64_reference(cur.detach(), tgt)
            lk = quantile_huber_loss(cur, tgt, sum_over_quantiles=False)
            gk, lk = torch.autograd.grad(lk, cur)[0], lk.detach()
            le = sb3_quantile_huber_loss(cur, tgt, sum_over_quantiles=False)
            ge, le = torch.autograd.grad(le, cur)[0], le.detach()
            ek, egk = agreement(lk, gk, ref, t, cur.numel())
            et, egt = agreement(le, ge, ref, t, cur.numel())
            del ref, lk, gk, le, ge
            assert ek <= 1.0 and egk <= 1.0, (n_critics, nq, b, ek, egk)
            mem = {"kernel_peak_bytes": peak_bytes(kern), "torch_eager_peak_bytes": peak_bytes(eager)}
            kgraph, torch_graph = capture(kern)[0], capture(eager)[0]
            row = {"n_critics": n_critics, "n_quantiles": nq, "drop": drop, "n_target": t, "batch": b, "pairs": b * n_critics * nq * t,
                   "kernel_loss_err_over_bound": ek, "kernel_grad_err_over_bound": egk,
                   "torch_fp32_loss_err_over_bound": et, "torch_fp32_grad_err_over_bound": egt}
            row.update(mem)
            # eager: each call from Python (autograd, allocations, the C entry's checks); graph: the captured launches only
            row.update(measure({"kernel_eager": kern, "kernel_graph": kgraph.replay, "torch_eager": eager, "torch_graph": torch_graph.replay},
                               args.rounds, args.min_ms))
            row["speedup_eager"] = row["torch_eager_us"] / row["kernel_eager_us"]
            row["speedup_graph"] = row["torch_graph_us"] / row["kernel_graph_us"]
            row["kernel_graph_pair_rate_per_s"] = row["pairs"] / (row["kernel_graph_us"] * 1e-6)
            rows.append(row)
            print(json.dumps(row), flush=True)
            del kgraph, torch_graph
            torch.cuda.empty_cache()
    return rows


def update_rows(args):
    """One TQC critic update on a fixed batch: CriticTarget -> critic forward -> loss -> backward -> Adam step."""
    rows = []
    g = torch.Generator().manual_seed(0)
    asd = {}
    for i, fan_in in zip((0, 2, 4), (OBS_DIM, 128, 128)):
        asd["latent_pi.%d.weight" % i], asd["latent_pi.%d.bias" % i] = torch.randn(128, fan_in, generator=g) / math.sqrt(fan_in), torch.zeros(128)
    for k in ("mu", "log_std"):
        asd[k + ".weight"], asd[k + ".bias"] = torch.randn(ACT_DIM, 128, generator=g) / math.sqrt(128), torch.zeros(ACT_DIM)
    actor = SquashedGaussianPolicy(OBS_DIM, ACT_DIM, device=DEV, precision="fp32").load_state_dict(asd)
    alpha = torch.tensor([0.2], device=DEV)
    for n_critics, nq, drop in CONFIGS:
        for b in SIZES:
            torch.manual_seed(b)
            gd = torch.Generator(device=DEV).manual_seed(b)
            obs = torch.rand((b, OBS_DIM), generator=gd, device=DEV) * 2 - 1
            act = torch.rand((b, ACT_DIM), generator=gd, device=DEV) * 2 - 1
            batch = ReplayBufferSamples(obs, act, torch.rand((b, OBS_DIM), generator=gd, device=DEV) * 2 - 1,
                                        (torch.rand((b, 1), generator=gd, device=DEV) < 0.1).float(),
                                        torch.rand((b, 1), generator=gd, device=DEV) * 2 - 1)
            critic0 = Critics(OBS_DIM, ACT_DIM, n_critics, nq).to(DEV)
            tgt = CriticTarget(actor, kind="tqc", n_critics=n_critics, n_quantiles=nq, top_quantiles_to_drop_per_net=drop)
            tgt.load_state_dict(Critics(OBS_DIM, ACT_DIM, n_critics, nq).to(DEV).sb3_state_dict())
            fns = {}
            for name, lossfn in (("update_kernel_loss", quantile_huber_loss), ("update_torch_loss", sb3_quantile_huber_loss)):
                critic = copy.deepcopy(critic0)
                opt = torch.optim.Adam(critic.parameters(), lr=3e-4, capturable=True)

                def step(critic=critic, opt=opt, lossfn=lossfn):
                    y = tgt(batch, alpha)
                    loss = lossfn(critic(batch.observations, batch.actions), y.unsqueeze(1), sum_over_quantiles=False)
                    opt.zero_grad(set_to_none=False)
                    loss.backward()
                    opt.step()
                    return loss.detach()
                fns[name + "_eager"] = step
                fns[name + "_graph"] = capture(step)[0].replay
            row = {"n_critics": n_critics, "n_quantiles": nq, "drop": drop, "batch": b}
            row.update(measure(fns, args.rounds, args.min_ms))
            for mode in ("eager", "graph"):
                k, p = row["update_kernel_loss_%s_us" % mode], row["update_torch_loss_%s_us" % mode]
                row["update_saving_%s_us" % mode] = p - k
                row["update_speedup_%s" % mode] = p / k
            rows.append(row)
            print(json.dumps(row), flush=True)
            del fns
            torch.cuda.empty_cache()
    return rows


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
    out = {"card": name, "nvidia_smi": smi, "tf32": False, "rounds": args.rounds, "unit": "us per call, median over rounds",
           "loss": "sum_over_quantiles=False, forward + backward (torch.autograd.grad w.r.t. current)", "rows": loss_rows(args),
           "critic_update": update_rows(args)}
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
