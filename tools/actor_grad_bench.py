"""Time ``Actor`` (the K12 kernels instantiated for the actor: forward with the squashed head, backward, reduction) against
SB3's actor in PyTorch fp32 (TF32 off; ``Normal(..., validate_args=False)``, without which it cannot be captured) with
autograd: ``action_log_prob`` forward + backward to every parameter from both outputs' gradients, each called eagerly and
replayed from a CUDA graph, with CUDA events; the variants are alternated over several rounds and the median per call is
reported, with each one's peak memory.  In the same run both paths are checked
against the fp64 restatement of tests/test_actor_grad_gpu.py within its bounds.  Then one whole SAC / TQC gradient step
(CriticTarget, Critic, critic loss and Adam, action_log_prob, actor loss and Adam, entropy-coefficient loss and Adam,
Polyak update, weight syncs) on a fixed batch is timed with the PyTorch actor and with ``Actor``.

    python tools/actor_grad_bench.py --out profiles/actor_grad_b200.json

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
from marinevehiclereinforcementlearning_b200 import Actor, Critic, CriticTarget, SquashedGaussianPolicy, quantile_huber_loss  # noqa: E402
from marinevehiclereinforcementlearning_b200.vec_tools import ReplayBufferSamples  # noqa: E402
from quantile_loss_bench import capture, card, measure, peak_bytes  # noqa: E402
from test_actor_grad_gpu import make_actor, reference, torch_action_log_prob, worst  # noqa: E402
from test_critic_grad_gpu import TOL_G, make_critic  # noqa: E402

DEV = "cuda"
CONFIGS = [("sac", 2, 1), ("tqc", 2, 25), ("tqc", 5, 25)]
SIZES = [256, 4096, 65536]
OBS_DIM, ACT_DIM = 9, 6


def agreement(m, actor, obs, g_a, g_lp, chunk=8192):
    """Worst error / bound of the parameter gradients, for the kernel and for fp32 PyTorch (both fed the kernel's eps)."""
    params = list(m.parameters())
    names = [n for n, _ in m.named_parameters()]
    eps = torch.empty((obs.shape[0], ACT_DIM), device=DEV)
    out = {"kernel": torch.autograd.grad(actor.action_log_prob(obs, eps=eps), params, [g_a, g_lp])}
    out["torch_fp32"] = torch.autograd.grad(torch_action_log_prob(m, obs, eps), params, [g_a, g_lp])
    ref = {}
    for lo in range(0, obs.shape[0], chunk):
        _, _, rc = reference(m, obs[lo:lo + chunk], eps[lo:lo + chunk], g_a[lo:lo + chunk], g_lp[lo:lo + chunk])
        for k, (g, s) in rc.items():
            g0, s0 = ref.get(k, (0.0, 0.0))
            ref[k] = (g0 + g, s0 + s)
    return {label + "_grad_err_over_bound": max(worst(g[names.index(k)], g64, s, TOL_G) for k, (g64, s) in ref.items())
            for label, g in out.items()}


def grad_rows(args):
    rows = []
    for b in SIZES:
        m = make_actor(OBS_DIM, ACT_DIM, b)
        actor = Actor(m, OBS_DIM, ACT_DIM, seed=1)
        params = list(m.parameters())
        g = torch.Generator(device=DEV).manual_seed(b)
        obs = torch.rand((b, OBS_DIM), generator=g, device=DEV) * 2 - 1
        g_a = torch.randn((b, ACT_DIM), generator=g, device=DEV) / b
        g_lp = torch.randn((b,), generator=g, device=DEV) / b
        row = {"batch": b}
        row.update(agreement(m, actor, obs, g_a, g_lp))
        assert max(v for k, v in row.items() if k.endswith("over_bound")) <= 1.0, row

        def kern():   # action_log_prob forward + backward to every parameter
            return torch.autograd.grad(actor.action_log_prob(obs), params, [g_a, g_lp])

        def pt():     # SB3's actor: rsample draws its eps with torch.randn
            return torch.autograd.grad(torch_action_log_prob(m, obs, torch.randn((b, ACT_DIM), device=DEV)), params, [g_a, g_lp])

        row["kernel_peak_bytes"], row["torch_peak_bytes"] = peak_bytes(kern), peak_bytes(pt)
        fns = {"kernel_eager": kern, "kernel_graph": capture(kern)[0].replay, "torch_eager": pt, "torch_graph": capture(pt)[0].replay}
        row.update(measure(fns, args.rounds, args.min_ms))
        for mode in ("eager", "graph"):
            row["speedup_%s" % mode] = row["torch_%s_us" % mode] / row["kernel_%s_us" % mode]
        rows.append(row)
        print(json.dumps(row), flush=True)
        torch.cuda.empty_cache()
    return rows


def step_rows(args):
    """One SAC / TQC gradient step on a fixed batch, every critic pass on Critic / CriticTarget, the actor's on PyTorch or
    on Actor."""
    rows = []
    target_entropy = -float(ACT_DIM)
    for kind, n_c, nq in CONFIGS:
        for b in SIZES:
            gd = torch.Generator(device=DEV).manual_seed(b)
            obs = torch.rand((b, OBS_DIM), generator=gd, device=DEV) * 2 - 1
            batch = ReplayBufferSamples(obs, torch.rand((b, ACT_DIM), generator=gd, device=DEV) * 2 - 1,
                                        torch.rand((b, OBS_DIM), generator=gd, device=DEV) * 2 - 1,
                                        (torch.rand((b, 1), generator=gd, device=DEV) < 0.1).float(),
                                        torch.rand((b, 1), generator=gd, device=DEV) * 2 - 1)
            actor0, critic0 = make_actor(OBS_DIM, ACT_DIM, 5), make_critic(OBS_DIM, ACT_DIM, n_c, nq, 7)
            fns = {}
            for name in ("torch_actor", "kernel_actor"):
                actor_m, critic, critic_t = copy.deepcopy(actor0), copy.deepcopy(critic0), copy.deepcopy(critic0)
                log_ent = torch.zeros(1, device=DEV, requires_grad=True)
                actor_t = SquashedGaussianPolicy(OBS_DIM, ACT_DIM, device=DEV, precision="fp32", seed=2)
                actor_t.load_state_dict(dict(actor_m.named_parameters()), share=True)
                tgt = CriticTarget(actor_t, kind=kind, n_critics=n_c, n_quantiles=nq, top_quantiles_to_drop_per_net=2 if kind == "tqc" else 0)
                tgt.load_state_dict(critic_t.state_dict(), share=True)
                crit = Critic(critic, OBS_DIM, ACT_DIM, kind=kind, n_critics=n_c, n_quantiles=nq)
                opts = [torch.optim.Adam(p, lr=3e-4, capturable=True) for p in (critic.parameters(), actor_m.parameters(), [log_ent])]
                if name == "kernel_actor":
                    act = Actor(actor_m, OBS_DIM, ACT_DIM, seed=4).action_log_prob
                else:
                    def act(o, actor_m=actor_m):
                        return torch_action_log_prob(actor_m, o, torch.randn((o.shape[0], ACT_DIM), device=DEV))
                params, tparams = list(critic.parameters()), list(critic_t.parameters())

                def q_of(o, a, crit=crit):
                    q = crit(o, a)
                    return torch.stack(q, 1) if isinstance(q, tuple) else q

                def step(act=act, q_of=q_of, opts=opts, tgt=tgt, actor_t=actor_t, log_ent=log_ent, params=params, tparams=tparams):
                    y = tgt(batch, log_ent.detach().exp())
                    q = q_of(batch.observations, batch.actions)
                    if kind == "tqc":
                        loss_c = quantile_huber_loss(q, y.unsqueeze(1), sum_over_quantiles=False)
                    else:
                        loss_c = 0.5 * sum(F.mse_loss(q[:, i], y) for i in range(n_c))
                    opts[0].zero_grad(set_to_none=False)
                    loss_c.backward()
                    opts[0].step()
                    a_pi, lp = act(batch.observations)
                    q_pi = q_of(batch.observations, a_pi)
                    q_pi = q_pi.min(1)[0] if kind == "sac" else q_pi.mean(2).mean(1, keepdim=True)
                    loss_a = (log_ent.detach().exp() * lp.unsqueeze(1) - q_pi).mean()
                    opts[1].zero_grad(set_to_none=False)
                    loss_a.backward()
                    opts[1].step()
                    loss_e = -(log_ent * (lp + target_entropy).detach()).mean()
                    opts[2].zero_grad(set_to_none=False)
                    loss_e.backward()
                    opts[2].step()
                    with torch.no_grad():
                        torch._foreach_lerp_(tparams, params, 0.005)
                    tgt.sync_weights()
                    actor_t.sync_weights()
                    return loss_a.detach()
                fns["step_%s_eager" % name] = step
                fns["step_%s_graph" % name] = capture(step)[0].replay
            row = {"kind": kind, "n_critics": n_c, "n_quantiles": nq, "batch": b}
            row.update(measure(fns, args.rounds, args.min_ms))
            for mode in ("eager", "graph"):
                row["step_speedup_%s" % mode] = row["step_torch_actor_%s_us" % mode] / row["step_kernel_actor_%s_us" % mode]
            rows.append(row)
            print(json.dumps(row), flush=True)
            torch.cuda.empty_cache()
    return rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "actor_grad_b200.json"))
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--min-ms", type=float, default=20.0)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("actor_grad_bench needs a CUDA device")
    torch.backends.cuda.matmul.allow_tf32 = torch.backends.cudnn.allow_tf32 = False
    name, smi = card()
    result = {"device": name, "nvidia_smi_name_power_limit_max_sm_clock": smi, "obs_dim": OBS_DIM, "act_dim": ACT_DIM,
              "tf32": False, "grad": grad_rows(args), "step": step_rows(args)}
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(result, f, indent=1)
    print("wrote", args.out)


if __name__ == "__main__":
    main()
