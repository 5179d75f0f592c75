"""GPU: ``quantile_huber_loss`` (csrc/mvrl_loss.cu, quantile_huber_kernel) - loss and gradient against the fp64 restatement
of sb3_contrib's function (tests/test_quantile_loss_cpu.py) over TQC / QR-DQN shapes and batch sizes, single pairs bit for
bit against sb3_contrib's text in fp32 torch, autograd through a torch.nn.Linear, determinism, a captured TQC critic update
against its eager twin, the 65 536-row size and the refusals."""
import copy
import math

import pytest
import torch

from test_quantile_loss_cpu import Critics, pair_count, quantile_huber_loss as sb3_quantile_huber_loss, restatement, restatement_sums

pytestmark = pytest.mark.gpu

if torch.cuda.is_available():
    from marinevehiclereinforcementlearning_b200 import (BlueROV2Heavy6DoFVecEnv, CriticTarget, ReplayBuffer, SquashedGaussianPolicy,
                                                         _lib, quantile_huber_loss)

DEV = "cuda"
U = 2.0 ** -24
SIZES = (1, 127, 128, 129, 4099)
# (C, Nq, T); C None: QR-DQN's 2-D form.  The last two stage their target rows in several chunks (the kernel's chunk is
# 288 columns for C Nq = 50 and 16 for C Nq = 3), the second ending on a chunk of 13, not a multiple of 4.
CONFIGS = [(2, 25, 46), (5, 25, 115), (5, 32, 160), (1, 1, 1), (3, 7, 20), (None, 25, 50), (2, 25, 1000), (1, 3, 701)]


def make_inputs(b, c, nq, t, seed, scale=1.5):
    """current [B, C, Nq] (2-D: [B, Nq]) and target [B, 1, T] ([B, T]); the spread puts pairs in both Huber branches and on
    both sides of zero."""
    g = torch.Generator(device=DEV).manual_seed(seed)
    cur = torch.randn((b, nq) if c is None else (b, c, nq), generator=g, device=DEV) * scale
    tgt = torch.randn((b, t) if c is None else (b, 1, t), generator=g, device=DEV) * scale
    return cur, tgt


def kernel_loss_and_grad(cur, tgt, sum_over):
    x = cur.clone().requires_grad_(True)
    loss = quantile_huber_loss(x, tgt, sum_over_quantiles=sum_over)
    loss.backward()
    torch.cuda.synchronize()
    return loss.detach(), x.grad


def ratios(loss, grad, cur, tgt, sum_over, ref=None):
    """(|loss - fp64| / loss bound, max over the elements of |grad - fp64| / grad bound).  Every term of the loss is >= 0,
    so its bound is relative: (T + log2(rows) + 8) u; each gradient element sums T terms w h', so its bound is
    (T + 8) u sum_j |w h'| / N."""
    t = tgt.shape[-1]
    rows = cur.numel()
    l64, g64, gabs = ref if ref is not None else restatement(cur, tgt, sum_over)
    lb = (t + math.log2(rows) + 8) * U * l64
    el = abs(float(loss) - l64) / lb if lb > 0 else (0.0 if float(loss) == l64 else math.inf)
    gb = (t + 8) * U * gabs
    diff = (grad.double() - g64).abs()
    assert bool((diff[gb == 0] == 0).all())
    eg = float((diff / gb.clamp(min=1e-300)).max())
    return el, eg


@pytest.mark.parametrize("sum_over", [False, True])
@pytest.mark.parametrize("cfg", CONFIGS, ids=["C%s-Nq%d-T%d" % c for c in CONFIGS])
def test_loss_and_grad_match_fp64_restatement(cfg, sum_over):
    c, nq, t = cfg
    worst = [0.0, 0.0]
    for b in SIZES:
        cur, tgt = make_inputs(b, c, nq, t, seed=b * 7 + nq)
        loss, grad = kernel_loss_and_grad(cur, tgt, sum_over)
        assert loss.shape == () and loss.dtype == torch.float32 and grad.shape == cur.shape
        if b == 4099:
            d = tgt.reshape(b, 1, -1) - cur.reshape(b, -1, 1)
            assert bool((d.abs() > 1).any()) and bool((d.abs() <= 1).any()) and bool((d < 0).any()) and bool((d > 0).any())
        el, eg = ratios(loss, grad, cur, tgt, sum_over)
        worst = [max(worst[0], el), max(worst[1], eg)]
        assert el <= 1.0 and eg <= 1.0, (cfg, b, sum_over, el, eg)
    print("quantile huber %s sum_over_quantiles=%s: worst |loss - fp64| / bound %.3g, |grad - fp64| / bound %.3g"
          % (cfg, sum_over, worst[0], worst[1]))


def test_non_contiguous_inputs():
    cur, tgt = make_inputs(300, 5, 25, 115, seed=3)
    cur_nc = cur.transpose(1, 2).contiguous().transpose(1, 2)
    tgt_nc = tgt.expand(300, 1, 115).transpose(0, 1).contiguous().transpose(0, 1)
    assert not cur_nc.is_contiguous()
    l1, g1 = kernel_loss_and_grad(cur, tgt, False)
    l2, g2 = kernel_loss_and_grad(cur_nc, tgt_nc, False)
    assert torch.equal(l1, l2) and torch.equal(g1, g2)


def bits(x):
    """int32 view with -0 counted as +0 (the sign of a zero gradient follows the order autograd adds its branches' zero
    contributions)."""
    return (x.float() + 0.0).view(torch.int32)


ULP1 = float.fromhex("0x1.000002p+0")      # 1 + ulp
ONE_M = float.fromhex("0x1.fffffep-1")     # 1 - ulp
TINY = float.fromhex("0x1p-149")           # smallest subnormal
DELTAS = [0.0, -0.0, TINY, ONE_M, 1.0, ULP1, 0.75, 3.0, 2.0 ** 66]


@pytest.mark.parametrize("sum_over", [False, True])
def test_single_pairs_bitwise_equal_sb3_text_in_fp32(sum_over):
    """B = C = T = 1, Nq = 4 (tau 1/8, 3/8, 5/8, 7/8: exact in fp32 however torch divides): one current quantile i at
    delta, the others at delta = 0 (no loss, no gradient), so loss and gradient are one rounded term each - equal bit for
    bit to sb3_contrib's function in fp32 torch with autograd, for delta = +-0, +-smallest subnormal, +-(1 - ulp), +-1,
    +-(1 + ulp), +-0.75, +-3, +-2^66 and tau below and above 0.5."""
    n = 0
    for dm in DELTAS:
        for sgn in (1.0, -1.0):
            delta = sgn * dm
            for i in range(4):
                t = torch.tensor([[[-0.0 if math.copysign(1.0, delta) < 0 and delta == 0 else 0.0]]], device=DEV)
                cur = torch.zeros((1, 1, 4), device=DEV)
                cur[0, 0, i] = 0.0 if delta == 0 else -delta          # delta = t - q exactly
                x1, x2 = cur.clone().requires_grad_(True), cur.clone().requires_grad_(True)
                ref = sb3_quantile_huber_loss(x1, t, sum_over_quantiles=sum_over)
                ref.backward()
                got = quantile_huber_loss(x2, t, sum_over_quantiles=sum_over)
                got.backward()
                d = (t.reshape(1, 1, 1) - cur.reshape(1, 4, 1))[0, i, 0]
                assert float(d) == delta and math.copysign(1.0, float(d)) == math.copysign(1.0, delta)
                assert torch.equal(bits(got.detach()), bits(ref.detach())), (delta, i, float(got), float(ref))
                assert torch.equal(bits(x2.grad), bits(x1.grad)), (delta, i, x2.grad.tolist(), x1.grad.tolist())
                n += 1
    assert n == len(DELTAS) * 2 * 4


def test_autograd_through_a_linear_layer(monkeypatch):
    """current = Linear(x): the layer's weight and bias gradients against the fp64 restatement's gradient carried through
    the layer (the kernel's elementwise bound plus the fp32 product's); a scaled loss scales the gradient; a second
    backward on the retained graph gives the same gradient; under no_grad and without requires_grad no gradient is
    written (the C entry gets a null pointer) and the loss is the same."""
    b, c, nq, t, k = 129, 2, 25, 46, 16
    torch.manual_seed(0)
    lin = torch.nn.Linear(k, c * nq).to(DEV)
    x = torch.randn(b, k, device=DEV)
    _, tgt = make_inputs(b, c, nq, t, seed=11, scale=3.0)
    prev = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = False
    try:
        current = lin(x).view(b, c, nq)
        loss = quantile_huber_loss(current, tgt, sum_over_quantiles=False)
        loss.backward()
    finally:
        torch.backends.cuda.matmul.allow_tf32 = prev
    _, g64, gabs = restatement(current, tgt, False)
    g64, e = g64.reshape(b, -1), ((t + 8) * U * gabs).reshape(b, -1)
    x64 = x.double()
    w_ref, b_ref = g64.T @ x64, g64.sum(0)
    w_bound = e.T @ x64.abs() + (b + 2) * U * (g64.abs().T @ x64.abs())
    b_bound = e.sum(0) + (b + 2) * U * g64.abs().sum(0)
    rw = float(((lin.weight.grad.double() - w_ref).abs() / w_bound).max())
    rb = float(((lin.bias.grad.double() - b_ref).abs() / b_bound).max())
    assert rw <= 1.0 and rb <= 1.0, (rw, rb)
    print("autograd through Linear: |dW - fp64| / bound %.3g, |db - fp64| / bound %.3g" % (rw, rb))

    leaf = current.detach().clone().requires_grad_(True)
    loss = quantile_huber_loss(leaf, tgt, sum_over_quantiles=False)
    g1, = torch.autograd.grad(loss, leaf, retain_graph=True)
    g2, = torch.autograd.grad(loss, leaf, retain_graph=True)
    g25, = torch.autograd.grad(2.5 * loss, leaf)
    assert torch.equal(g1, g2) and torch.equal(g25, 2.5 * g1) and not torch.equal(g25, g1)

    seen = []

    class Spy:
        def __init__(self, lib):
            self.lib = lib

        def __getattr__(self, name):
            return getattr(self.lib, name)

        def mvrl_quantile_huber_loss(self, *args):
            seen.append(args[8])
            return self.lib.mvrl_quantile_huber_loss(*args)

    monkeypatch.setattr(_lib, "load", lambda lib=_lib.load(): Spy(lib))
    with_grad = quantile_huber_loss(leaf, tgt, sum_over_quantiles=False)
    with torch.no_grad():
        under_no_grad = quantile_huber_loss(leaf, tgt, sum_over_quantiles=False)
    plain = quantile_huber_loss(leaf.detach(), tgt, sum_over_quantiles=False)
    assert seen[0] is not None and seen[0].value is not None and seen[1] is None and seen[2] is None
    assert with_grad.grad_fn is not None and under_no_grad.grad_fn is None and plain.grad_fn is None
    assert not under_no_grad.requires_grad and not plain.requires_grad
    assert torch.equal(with_grad.detach(), under_no_grad) and torch.equal(plain, under_no_grad)


def test_repeated_calls_are_bitwise_equal():
    cur, tgt = make_inputs(4099, 5, 25, 115, seed=5)
    l0, g0 = kernel_loss_and_grad(cur, tgt, False)
    for _ in range(5):
        l1, g1 = kernel_loss_and_grad(cur, tgt, False)
        assert torch.equal(bits(l1), bits(l0)) and torch.equal(bits(g1), bits(g0))


def test_captured_tqc_critic_update_equals_eager_twin():
    """One TQC critic update - buf.sample -> CriticTarget -> critic forward -> quantile_huber_loss -> backward ->
    Adam(capturable=True).step() - captured in a CUDA graph and replayed R times gives the loss and parameters of an eager
    twin's R updates bit for bit."""
    n_critics, nq, drop, batch_size, R = 2, 25, 2, 256, 4
    env = BlueROV2Heavy6DoFVecEnv(512, action_mode="force", dtype=torch.float32, seed=1)
    obs_dim, act_dim = env.lenObs, env.lenAction
    g = torch.Generator(device=DEV).manual_seed(0)
    slots = 8
    state = {"observations": torch.rand((slots, 512, obs_dim), generator=g, device=DEV) * 2 - 1,
             "actions": torch.rand((slots, 512, act_dim), generator=g, device=DEV) * 2 - 1,
             "rewards": torch.rand((slots, 512), generator=g, device=DEV) * 2 - 1,
             "dones": (torch.rand((slots, 512), generator=g, device=DEV) < 0.1).to(torch.uint8),
             "timeouts": torch.zeros((slots, 512), dtype=torch.uint8, device=DEV),
             "last_obs": torch.zeros((obs_dim, env.ld), device=DEV),
             "cursor": torch.tensor([0, slots, 0, 0, 0], dtype=torch.int64), "seed": 3}
    state["next_observations"] = torch.rand((slots, 512, obs_dim), generator=g, device=DEV) * 2 - 1
    torch.manual_seed(1)
    actor = SquashedGaussianPolicy(obs_dim, act_dim, device=DEV, precision="fp32", seed=2)
    critic0 = Critics(obs_dim, act_dim, n_critics, nq).to(DEV)
    target_sd = Critics(obs_dim, act_dim, n_critics, nq).to(DEV).sb3_state_dict()
    alpha = torch.tensor([0.2], device=DEV)

    def twin():
        buf = ReplayBuffer(slots * 512, env, seed=3)
        buf.load_state_dict(state)
        tgt = CriticTarget(actor, kind="tqc", n_critics=n_critics, n_quantiles=nq, top_quantiles_to_drop_per_net=drop).load_state_dict(target_sd)
        critic = copy.deepcopy(critic0)
        opt = torch.optim.Adam(critic.parameters(), lr=3e-4, capturable=True)

        def step():
            batch = buf.sample(batch_size)
            y = tgt(batch, alpha)
            current = critic(batch.observations, batch.actions)
            loss = quantile_huber_loss(current, y.unsqueeze(1), sum_over_quantiles=False)
            opt.zero_grad(set_to_none=False)
            loss.backward()
            opt.step()
            return loss.detach()
        return critic, step

    warm = 3
    critic_e, step_e = twin()
    for _ in range(warm):
        step_e()
    eager = []
    for _ in range(R):
        loss = step_e()
        eager.append((loss.clone(), [p.detach().clone() for p in critic_e.parameters()]))
    torch.cuda.synchronize()

    critic_g, step_g = twin()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        for _ in range(warm):
            step_g()
    torch.cuda.current_stream().wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        loss_g = step_g()
    for r in range(R):
        graph.replay()
        torch.cuda.synchronize()
        assert torch.equal(bits(loss_g), bits(eager[r][0])), (r, float(loss_g), float(eager[r][0]))
        for p, q in zip(critic_g.parameters(), eager[r][1]):
            assert torch.equal(bits(p.detach()), bits(q)), r
    assert not torch.equal(eager[0][0], eager[1][0])


@pytest.mark.parametrize("sum_over", [False, True])
def test_full_size_against_chunked_fp64(sum_over):
    """B = 65 536, 5 x 25 quantiles, T = 115 (942 M pairs) in one call, against the fp64 restatement summed over chunks of
    4096 rows."""
    b, c, nq, t, chunk = 65536, 5, 25, 115, 4096
    cur, tgt = make_inputs(b, c, nq, t, seed=65536)
    loss, grad = kernel_loss_and_grad(cur, tgt, sum_over)
    s, whp, gabs = 0.0, [], []
    for lo in range(0, b, chunk):
        cs, cw, ca = restatement_sums(cur[lo:lo + chunk], tgt[lo:lo + chunk])
        s, whp, gabs = s + cs, whp + [cw], gabs + [ca]
    n = pair_count(cur, tgt, sum_over)
    el, eg = ratios(loss, grad, cur, tgt, sum_over, ref=(s / n, -torch.cat(whp) / n, torch.cat(gabs) / n))
    assert el <= 1.0 and eg <= 1.0, (el, eg)
    print("quantile huber B = 65536, 5 x 25, T = 115, sum_over_quantiles=%s: |loss - fp64| / bound %.3g, |grad - fp64| / bound %.3g"
          % (sum_over, el, eg))


def test_refusals():
    cur, tgt = make_inputs(64, 2, 25, 46, seed=0)
    with pytest.raises(ValueError, match="same CUDA device"):
        quantile_huber_loss(cur, tgt.cpu())
    with pytest.raises(ValueError, match="same CUDA device"):
        quantile_huber_loss(cur.cpu(), tgt.cpu())
    with pytest.raises(ValueError, match="float32"):
        quantile_huber_loss(cur.double(), tgt.double())
    with pytest.raises(ValueError, match="requires grad"):
        quantile_huber_loss(cur, tgt.requires_grad_(True))
    tgt = tgt.detach()
    if torch.cuda.device_count() >= 2:
        with pytest.raises(ValueError, match="same CUDA device"):
            quantile_huber_loss(cur, tgt.to("cuda:1"))
    lib = _lib.load()
    loss = torch.empty((), device=DEV)
    scratch = torch.empty(lib.mvrl_quantile_huber_scratch(64 * 50), dtype=torch.uint8, device=DEV)
    st = _lib.current_stream(cur.device)

    def call(c, t, out=loss):
        return lib.mvrl_quantile_huber_loss(64, 2, 25, 46, _lib.ptr(c), _lib.ptr(t), 0, _lib.ptr(out), None, _lib.ptr(scratch), st)
    assert call(cur, tgt.cpu()) == -1 and b"not device memory" in lib.mvrl_last_error()
    assert call(cur, tgt, out=loss.cpu()) == -1 and b"not a device pointer" in lib.mvrl_last_error()
    assert call(cur, tgt) == 0
    torch.cuda.synchronize()
    assert torch.equal(loss, quantile_huber_loss(cur, tgt, sum_over_quantiles=False))
