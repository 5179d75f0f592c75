"""CPU: ``quantile_huber_loss`` (marinevehiclereinforcementlearning_b200/policy.py) - the refusals decided before any launch,
the C entry's size checks, and the fp64 restatement of sb3_contrib's loss and gradient that tests/test_quantile_loss_gpu.py
compares the kernel with, pinned here against sb3_contrib's own text run in fp64 with autograd.  sb3_contrib's text and
TQC's critic (``Critics``) are kept here once for tests/test_quantile_loss_gpu.py and tools/quantile_loss_bench.py too."""
import ctypes as C
import os
import subprocess
import sys
import textwrap

import pytest
import torch
import torch as th

from conftest import ROOT
from marinevehiclereinforcementlearning_b200 import _lib
from marinevehiclereinforcementlearning_b200 import policy as P


# sb3_contrib 2.x common/utils.py, as published (its shape checks shortened to the comment); the reference of the
# restatement below.
def quantile_huber_loss(current_quantiles, target_quantiles, cum_prob=None, sum_over_quantiles=True):
    # shape checks: same ndim, same batch size, ndim in (2, 3)
    if cum_prob is None:
        n_quantiles = current_quantiles.shape[-1]
        cum_prob = (th.arange(n_quantiles, device=current_quantiles.device, dtype=th.float) + 0.5) / n_quantiles
        cum_prob = cum_prob.view(1, -1, 1) if current_quantiles.ndim == 2 else cum_prob.view(1, 1, -1, 1)
    pairwise_delta = target_quantiles.unsqueeze(-2) - current_quantiles.unsqueeze(-1)
    abs_pairwise_delta = th.abs(pairwise_delta)
    huber_loss = th.where(abs_pairwise_delta > 1, abs_pairwise_delta - 0.5, pairwise_delta**2 * 0.5)
    loss = th.abs(cum_prob - (pairwise_delta.detach() < 0).float()) * huber_loss
    if sum_over_quantiles:
        loss = loss.sum(dim=-2).mean()
    else:
        loss = loss.mean()
    return loss


def restatement_sums(current, target):
    """The pair sums of the loss in fp64 on the inputs' device: (sum of w h, sum_j w h' [B, C, Nq], sum_j |w h'| [B, C, Nq]).
    current [B, C, Nq] or [B, Nq], target [B, 1, T] or [B, T], any float dtype.  tau and w = |tau - [delta < 0]| are the
    fp32 values sb3_contrib (and the kernel) compute, tau by correctly rounded division; everything else is fp64."""
    cur = current.detach().double()
    cur = cur.unsqueeze(1) if cur.dim() == 2 else cur
    tgt = target.detach().double().reshape(cur.shape[0], -1)
    nq = cur.shape[-1]
    tau = ((torch.arange(nq, dtype=torch.float32) + 0.5) / nq).to(cur.device).view(1, 1, -1, 1)
    d = tgt[:, None, None, :] - cur[..., None]
    w = (tau - (d < 0).float()).abs().double()
    a = d.abs()
    outer = a > 1
    h = torch.where(outer, a - 0.5, d * d * 0.5)
    whp = w * torch.where(outer, torch.sign(d), d)
    return float((w * h).sum()), whp.sum(-1), whp.abs().sum(-1)


def pair_count(current, target, sum_over_quantiles):
    """N of the mean: B C T when the current quantiles are summed first, else B C Nq T."""
    b, nq, t = current.shape[0], current.shape[-1], target.shape[-1]
    c = current.shape[1] if current.dim() == 3 else 1
    return b * c * t * (1 if sum_over_quantiles else nq)


def restatement(current, target, sum_over_quantiles):
    """(loss, d loss / d current shaped like current, sum_j |w h'| / N) in fp64."""
    s, whp, gabs = restatement_sums(current, target)
    n = pair_count(current, target, sum_over_quantiles)
    return s / n, (-whp / n).reshape(current.shape), (gabs / n).reshape(current.shape)


class Critics(torch.nn.Module):
    """sb3_contrib TQC's critic: n_critics [128, 128, 128] GELU MLPs on [obs, action] -> n_quantiles each."""

    def __init__(self, obs_dim, act_dim, n_critics, n_quantiles):
        super().__init__()
        self.qfs = torch.nn.ModuleList(torch.nn.Sequential(
            torch.nn.Linear(obs_dim + act_dim, 128), torch.nn.GELU(), torch.nn.Linear(128, 128), torch.nn.GELU(),
            torch.nn.Linear(128, 128), torch.nn.GELU(), torch.nn.Linear(128, n_quantiles)) for _ in range(n_critics))

    def forward(self, obs, act):
        xa = torch.cat([obs, act], dim=1)
        return torch.stack([qf(xa) for qf in self.qfs], dim=1)

    def sb3_state_dict(self):
        return {"qf%d.%d.%s" % (i, j, p): getattr(qf[j], p).detach() for i, qf in enumerate(self.qfs) for j in (0, 2, 4, 6)
                for p in ("weight", "bias")}


CASES = [(4, 2, 25, 46), (3, 5, 25, 115), (2, 5, 32, 160), (5, 1, 1, 1), (7, 3, 7, 20), (6, None, 13, 9)]   # (B, C, Nq, T); C None: 2-D


def inputs(b, c, nq, t, seed, dtype=torch.float64):
    """fp32-representable values spread so that both Huber branches and both signs of delta occur."""
    g = torch.Generator().manual_seed(seed)
    cur = (torch.randn((b, nq) if c is None else (b, c, nq), generator=g) * 1.5).float()
    tgt = (torch.randn((b, t) if c is None else (b, 1, t), generator=g) * 1.5).float()
    return cur.to(dtype), tgt.to(dtype)


@pytest.mark.parametrize("sum_over", [False, True])
@pytest.mark.parametrize("case", CASES, ids=["B%d-C%s-Nq%d-T%d" % c for c in CASES])
def test_restatement_matches_sb3_text_in_fp64(case, sum_over):
    cur, tgt = inputs(*case, seed=sum(case[i] or 0 for i in range(4)))
    x = cur.clone().requires_grad_(True)
    ref = quantile_huber_loss(x, tgt, sum_over_quantiles=sum_over)
    ref.backward()
    loss, grad, gabs = restatement(cur, tgt, sum_over)
    ref = float(ref.detach())
    assert abs(loss - ref) <= 1e-13 * abs(ref)
    assert torch.allclose(grad, x.grad, rtol=1e-12, atol=1e-15 * float(gabs.max()))
    d = tgt.reshape(cur.shape[0], 1, -1) - cur.reshape(cur.shape[0], -1, 1)
    assert bool((d.abs() > 1).any()) and bool((d.abs() < 1).any()) and bool((d < 0).any()) and bool((d > 0).any())


def test_refusals_before_any_launch():
    cur, tgt = inputs(4, 2, 25, 46, seed=0, dtype=torch.float32)
    ok = [cur, tgt]
    for args, kw, match in (
            ([cur.double(), tgt], {}, "float32"), ([cur, tgt.half()], {}, "float32"), ([cur.tolist(), tgt], {}, "float32"),
            ([cur[0, 0], tgt[0, 0]], {}, "2-D"), ([cur[None], tgt[None]], {}, "2-D"), ([cur, tgt[:, 0]], {}, "2-D"),
            ([cur[:3], tgt], {}, "batch size"), ([cur[:0], tgt[:0]], {}, "batch size"),
            ([cur, tgt.expand(4, 2, 46)], {}, "per-critic"), (ok, {"cum_prob": torch.full((1, 1, 25, 1), 0.5)}, "cum_prob"),
            ([cur, tgt.clone().requires_grad_(True)], {}, "requires grad"), ([cur[:, :, :0], tgt], {}, "empty"),
            ([cur, tgt[:, :, :0]], {}, "empty")):
        with pytest.raises(ValueError, match=match):
            P.quantile_huber_loss(*args, **kw)
    # sb3_contrib's function is named as the way to what it accepts and this one refuses
    for args, kw in (([cur, tgt], {"cum_prob": 0}), ([cur, tgt.expand(4, 3, 46)], {}), ([cur, tgt.clone().requires_grad_(True)], {})):
        with pytest.raises(ValueError, match="sb3_contrib"):
            P.quantile_huber_loss(*args, **kw)


NO_CUDA = textwrap.dedent("""
    import sys
    sys.path.insert(0, %r)
    import torch
    from marinevehiclereinforcementlearning_b200 import quantile_huber_loss
    assert not torch.cuda.is_available()
    try:
        quantile_huber_loss(torch.zeros(4, 2, 25), torch.zeros(4, 1, 46))
    except RuntimeError as e:
        print("runtime error:", e)
""")


def test_without_cuda_raises_runtime_error():
    """Valid inputs without a CUDA device: RuntimeError (no CPU path), in a fresh interpreter that sees no device."""
    res = subprocess.run([sys.executable, "-c", NO_CUDA % ROOT], env=dict(os.environ, CUDA_VISIBLE_DEVICES=""),
                         capture_output=True, text=True, timeout=600)
    assert res.returncode == 0 and "runtime error:" in res.stdout and "CUDA device" in res.stdout, res.stdout[-2000:] + res.stderr[-2000:]


def test_c_entry_size_checks():
    """Sizes below 1 and products that overflow int64 are refused before any device work; the scratch is 8 bytes per
    block of 256 current quantiles."""
    lib = _lib.load()
    assert lib.mvrl_quantile_huber_scratch(0) == 0 and lib.mvrl_quantile_huber_scratch(1) == 8
    assert lib.mvrl_quantile_huber_scratch(256) == 8 and lib.mvrl_quantile_huber_scratch(257) == 16
    assert lib.mvrl_quantile_huber_scratch(65536 * 125) == 32000 * 8
    buf = (C.c_float * 16)()
    p = C.cast(buf, C.c_void_p)
    for dims, match in (((0, 2, 25, 46), b">= 1"), ((4, 0, 25, 46), b">= 1"), ((4, 2, 0, 46), b">= 1"), ((4, 2, 25, 0), b">= 1"),
                        ((-1, 2, 25, 46), b">= 1"), ((2 ** 62, 2, 25, 46), b"overflows"), ((2 ** 40, 5, 25, 2 ** 20), b"overflows"),
                        ((2 ** 33, 32, 32, 1), b"overflows")):
        assert lib.mvrl_quantile_huber_loss(*dims, p, p, 0, p, None, p, None) == -1, dims
        assert match in lib.mvrl_last_error(), (dims, lib.mvrl_last_error())
    assert lib.mvrl_quantile_huber_loss(4, 2, 25, 46, None, p, 0, p, None, p, None) == -1
    assert b"null" in lib.mvrl_last_error()
