"""Time ``Critic`` (critic_forward_kernel, critic_backward_kernel and its reduction) against the same critics in PyTorch fp32
(TF32 off) with autograd: forward + backward to every parameter, and the actor loss's path (forward, backward to the actions
only), each called eagerly and replayed from a CUDA graph, with CUDA events; the variants are alternated over several rounds
and the median per call is reported, with each one's peak memory.  In the same run both paths are checked against the fp64
restatement of tests/test_critic_grad_gpu.py within its bounds.  Then one whole critic update (CriticTarget, critic forward,
loss, backward, Adam, Polyak update, target sync) is timed with the PyTorch critic and with ``Critic``.

    python tools/critic_grad_bench.py --out profiles/critic_grad_b200.json

Writes one JSON file: the card's name, power limit and max SM clock, then one row per (configuration, batch size)."""
import argparse
import copy
import json
import os
import sys

import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from marinevehiclereinforcementlearning_b200 import Critic, CriticTarget, SquashedGaussianPolicy, quantile_huber_loss  # noqa: E402
from marinevehiclereinforcementlearning_b200.vec_tools import ReplayBufferSamples  # noqa: E402
from quantile_loss_bench import capture, card, measure, peak_bytes  # noqa: E402
from test_critic_grad_gpu import TOL_G, TOL_Q, make_critic, reference, worst  # noqa: E402

DEV = "cuda"
CONFIGS = [("sac", 2, 1), ("tqc", 2, 25), ("tqc", 5, 25)]
SIZES = [256, 4096, 65536]
OBS_DIM, ACT_DIM = 9, 6


def agreement(module, crit, kind, obs, act, grad_q, chunk=8192):
    """Worst error / bound of q, the parameter gradients and the action gradient, for the kernel and for fp32 PyTorch."""
    params = list(module.parameters())
    names = [n for n, _ in module.named_parameters()]
    out = {}
    for label, fn in (("kernel", lambda a: crit(obs, a)), ("torch_fp32", lambda a: module(obs, a))):
        a = act.clone().requires_grad_(True)
        q = fn(a)
        q = torch.stack(q, 1) if isinstance(q, tuple) else q
        grads = torch.autograd.grad(q, params + [a], grad_q)
        out[label] = (q.detach(), dict(zip(names, grads[:-1])), grads[-1])
    ref_q, ref_g, ref_a = [], {}, []
    for lo in range(0, obs.shape[0], chunk):
        q64, g64, a64 = reference(module, obs[lo:lo + chunk], act[lo:lo + chunk], grad_q[lo:lo + chunk])
        ref_q.append(q64)
        ref_a.append(a64)
        for k, (g, s) in g64.items():
            g0, s0 = ref_g.get(k, (0.0, 0.0))
            ref_g[k] = (g0 + g, s0 + s)
    q64 = torch.cat(ref_q)
    ga64, gas = torch.cat([x[0] for x in ref_a]), torch.cat([x[1] for x in ref_a])
    row = {}
    for label, (q, g, ga) in out.items():
        row[label + "_q_err_over_bound"] = worst(q, q64, max(1.0, float(q64.abs().max())), TOL_Q)
        row[label + "_grad_err_over_bound"] = max(worst(g[k], g64, s, TOL_G) for k, (g64, s) in ref_g.items())
        row[label + "_grad_act_err_over_bound"] = worst(ga, ga64, gas, TOL_G)
    return row


def grad_rows(args):
    rows = []
    for kind, n_c, nq in CONFIGS:
        for b in SIZES:
            module = make_critic(OBS_DIM, ACT_DIM, n_c, nq, b + n_c)
            crit = Critic(module, OBS_DIM, ACT_DIM, kind=kind, n_critics=n_c, n_quantiles=nq)
            params = list(module.parameters())
            g = torch.Generator(device=DEV).manual_seed(b)
            obs = torch.rand((b, OBS_DIM), generator=g, device=DEV) * 2 - 1
            act = torch.rand((b, ACT_DIM), generator=g, device=DEV) * 2 - 1
            grad_q = torch.randn((b, n_c, nq), generator=g, device=DEV) / b
            row = {"kind": kind, "n_critics": n_c, "n_quantiles": nq, "batch": b}
            row.update(agreement(module, crit, kind, obs, act, grad_q))
            assert max(v for k, v in row.items() if k.endswith("over_bound")) <= 1.0, row

            def q_of(fn, a):
                q = fn(obs, a)
                return torch.stack(q, 1) if isinstance(q, tuple) else q

            def kern():   # forward + backward to every parameter
                return torch.autograd.grad(q_of(crit, act), params, grad_q)

            def pt():
                return torch.autograd.grad(q_of(module, act), params, grad_q)

            def kern_actor():   # the actor loss's path: backward to the actions only
                a = act.detach().requires_grad_(True)
                return torch.autograd.grad(q_of(crit, a), a, grad_q)

            def pt_actor():
                a = act.detach().requires_grad_(True)
                return torch.autograd.grad(q_of(module, a), a, grad_q)

            row["kernel_peak_bytes"], row["torch_peak_bytes"] = peak_bytes(kern), peak_bytes(pt)
            fns = {"kernel_eager": kern, "kernel_graph": capture(kern)[0].replay, "torch_eager": pt, "torch_graph": capture(pt)[0].replay}
            row.update(measure(fns, args.rounds, args.min_ms))
            for p in params:
                p.requires_grad_(False)
            fns = {"actor_kernel_eager": kern_actor, "actor_kernel_graph": capture(kern_actor)[0].replay,
                   "actor_torch_eager": pt_actor, "actor_torch_graph": capture(pt_actor)[0].replay}
            row.update(measure(fns, args.rounds, args.min_ms))
            for pre in ("", "actor_"):
                for mode in ("eager", "graph"):
                    row["%sspeedup_%s" % (pre, mode)] = row["%storch_%s_us" % (pre, mode)] / row["%skernel_%s_us" % (pre, mode)]
            rows.append(row)
            print(json.dumps(row), flush=True)
            torch.cuda.empty_cache()
    return rows


def update_rows(args):
    """One critic update on a fixed batch: CriticTarget -> critic -> loss -> backward -> Adam -> Polyak -> target sync."""
    rows = []
    actor = SquashedGaussianPolicy(OBS_DIM, ACT_DIM, device=DEV, precision="fp32", seed=1)
    alpha = torch.tensor([0.2], device=DEV)
    for kind, n_c, nq in CONFIGS:
        for b in SIZES:
            gd = torch.Generator(device=DEV).manual_seed(b)
            obs = torch.rand((b, OBS_DIM), generator=gd, device=DEV) * 2 - 1
            act = torch.rand((b, ACT_DIM), generator=gd, device=DEV) * 2 - 1
            batch = ReplayBufferSamples(obs, act, torch.rand((b, OBS_DIM), generator=gd, device=DEV) * 2 - 1,
                                        (torch.rand((b, 1), generator=gd, device=DEV) < 0.1).float(),
                                        torch.rand((b, 1), generator=gd, device=DEV) * 2 - 1)
            critic0 = make_critic(OBS_DIM, ACT_DIM, n_c, nq, 7)
            fns = {}
            for name in ("torch_critic", "kernel_critic"):
                critic, critic_t = copy.deepcopy(critic0), copy.deepcopy(critic0)
                tgt = CriticTarget(actor, kind=kind, n_critics=n_c, n_quantiles=nq, top_quantiles_to_drop_per_net=2 if kind == "tqc" else 0)
                tgt.load_state_dict(critic_t.state_dict(), share=True)
                opt = torch.optim.Adam(critic.parameters(), lr=3e-4, capturable=True)
                fwd = Critic(critic, OBS_DIM, ACT_DIM, kind=kind, n_critics=n_c, n_quantiles=nq) if name == "kernel_critic" else critic
                params, tparams = list(critic.parameters()), list(critic_t.parameters())

                def step(fwd=fwd, opt=opt, tgt=tgt, params=params, tparams=tparams):
                    y = tgt(batch, alpha)
                    q = fwd(batch.observations, batch.actions)
                    if kind == "tqc":
                        loss = quantile_huber_loss(q, y.unsqueeze(1), sum_over_quantiles=False)
                    else:
                        qs = q if isinstance(q, tuple) else tuple(q[:, i] for i in range(n_c))
                        loss = 0.5 * sum(F.mse_loss(x, y) for x in qs)
                    opt.zero_grad(set_to_none=False)
                    loss.backward()
                    opt.step()
                    with torch.no_grad():
                        torch._foreach_lerp_(tparams, params, 0.005)
                    tgt.sync_weights()
                    return loss.detach()
                fns["update_%s_eager" % name] = step
                fns["update_%s_graph" % name] = capture(step)[0].replay
            row = {"kind": kind, "n_critics": n_c, "n_quantiles": nq, "batch": b}
            row.update(measure(fns, args.rounds, args.min_ms))
            for mode in ("eager", "graph"):
                row["update_speedup_%s" % mode] = row["update_torch_critic_%s_us" % mode] / row["update_kernel_critic_%s_us" % mode]
            rows.append(row)
            print(json.dumps(row), flush=True)
            torch.cuda.empty_cache()
    return rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "critic_grad_b200.json"))
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--min-ms", type=float, default=20.0)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("critic_grad_bench needs a CUDA device")
    torch.backends.cuda.matmul.allow_tf32 = torch.backends.cudnn.allow_tf32 = False
    name, smi = card()
    result = {"device": name, "nvidia_smi_name_power_limit_max_sm_clock": smi, "obs_dim": OBS_DIM, "act_dim": ACT_DIM,
              "tf32": False, "grad": grad_rows(args), "update": update_rows(args)}
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(result, f, indent=1)
    print("wrote", args.out)


if __name__ == "__main__":
    main()
