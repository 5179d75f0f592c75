"""GPU: ``Critic`` (csrc/mvrl_policy.cu, critic_forward_kernel / critic_backward_kernel / critic_grad_reduce_kernel) against
an fp64 restatement of SB3's critics and their backward pass - q, every parameter gradient and the action gradient over
shapes, batch sizes, critic configurations and the three combinations of what requires grad; bit-for-bit repeats and graph
replays; a captured TQC critic update against its eager twin and against 20 updates in fp64; SAC's tuple form; the
refusals in Python and C."""
import copy
import ctypes as C

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

if torch.cuda.is_available():
    from marinevehiclereinforcementlearning_b200 import BlueROV2Heavy6DoFVecEnv, Critic, CriticTarget, ReplayBuffer, SquashedGaussianPolicy, _lib
    from marinevehiclereinforcementlearning_b200.policy import quantile_huber_loss
    from test_critic_target_gpu import critic_state_dict

DEV = "cuda"
SHAPES = [(9, 6), (11, 3), (5, 3), (1, 1), (10, 6)]
SIZES = (1, 127, 128, 129, 4099)
# (kind, n_critics, n_quantiles): n_critics 1 / 2 / 5, n_quantiles 1 / 25 / 32
CONFIGS = [("sac", 1, 1), ("sac", 2, 1), ("sac", 5, 1), ("tqc", 2, 25), ("tqc", 1, 1), ("tqc", 5, 32), ("tqc", 5, 25)]
# K10's forward bound: |q - fp64| <= TOL_Q max(1, |q|max).  Gradients: |g - fp64| <= TOL_G S element-wise, S the fp64 sum
# of absolute products that forms g (for dW_l: |dZ_l|^T |H_{l-1}| with |dZ| carried down the network in absolute values:
# |dZ_{l-1}| = (|dZ_l| |W_l|) (|GELU'(z)| + |GELU''(z)| |z|abs), z = z_{l-1}).  The forward's rounding of z is relative to
# |z|abs = |H| |W|^T + |b|, not to |z|, so it enters as |z|abs times the derivative: in GELU' above, and in H itself
# (|H| + |GELU'(z)| |z|abs in place of |H|).  Both matter where a single row makes the sum and z cancels to near 0 or to
# GELU''s zero.  fp32 PyTorch (TF32 off) passes the same bounds (asserted below).
TOL_Q, TOL_G = 5e-5, 1e-4


def bits(t):
    return t.contiguous().view(torch.int32)


class SB3Critic(torch.nn.Module):
    """SB3's ContinuousCritic / sb3_contrib's TQC Critic body: qf{i} = Sequential(Linear, GELU, Linear, GELU, Linear, GELU, Linear)."""

    def __init__(self, obs_dim, act_dim, n_critics, n_out):
        super().__init__()
        self.n_critics = n_critics
        for i in range(n_critics):
            self.add_module("qf%d" % i, torch.nn.Sequential(
                torch.nn.Linear(obs_dim + act_dim, 128), torch.nn.GELU(), torch.nn.Linear(128, 128), torch.nn.GELU(),
                torch.nn.Linear(128, 128), torch.nn.GELU(), torch.nn.Linear(128, n_out)))

    def forward(self, obs, act):
        xa = torch.cat([obs, act], dim=1)
        return torch.stack([getattr(self, "qf%d" % i)(xa) for i in range(self.n_critics)], dim=1)


def make_critic(obs_dim, act_dim, n_critics, n_out, seed):
    m = SB3Critic(obs_dim, act_dim, n_critics, n_out)
    m.load_state_dict(critic_state_dict(obs_dim, act_dim, n_critics, n_out, seed))
    return m.to(DEV)


def batch(b, obs_dim, act_dim, seed):
    g = torch.Generator(device=DEV).manual_seed(seed)
    return torch.randn((b, obs_dim), generator=g, device=DEV), torch.rand((b, act_dim), generator=g, device=DEV) * 2 - 1


def gelu_grad64(z):
    return 0.5 * (1.0 + torch.erf(z / 2 ** 0.5)) + z * torch.exp(-0.5 * z * z) / (2 * torch.pi) ** 0.5


def gelu_grad2_64(z):
    return (2.0 - z * z) * torch.exp(-0.5 * z * z) / (2 * torch.pi) ** 0.5


def reference(module, obs, act, grad_q):
    """fp64: q [B, C, Nq], {param name: (grad, scale)}, (grad_act, scale)."""
    x = torch.cat([obs, act], 1).double()
    qs, out, ga, gs = [], {}, 0.0, 0.0
    for i in range(module.n_critics):
        qf = getattr(module, "qf%d" % i)
        W = [qf[j].weight.detach().double() for j in (0, 2, 4, 6)]
        b = [qf[j].bias.detach().double() for j in (0, 2, 4, 6)]
        h, hs, has, zs, za = x, [x], [x.abs()], [], []
        for l in range(3):
            z = h @ W[l].T + b[l]
            zs.append(z)
            za.append(h.abs() @ W[l].abs().T + b[l].abs())
            h = F.gelu(z)
            hs.append(h)
            has.append(h.abs() + gelu_grad64(z).abs() * za[l])
        qs.append(h @ W[3].T + b[3])
        if grad_q is None:
            continue
        dz = grad_q[:, i].double()
        dza = dz.abs()
        for l in (3, 2, 1, 0):
            name = "qf%d.%d." % (i, 2 * l)
            out[name + "weight"] = (dz.T @ hs[l], dza.T @ has[l])
            out[name + "bias"] = (dz.sum(0), dza.sum(0))
            dh, dha = dz @ W[l], dza @ W[l].abs()
            if l > 0:
                d = gelu_grad64(zs[l - 1])
                dz, dza = dh * d, dha * (d.abs() + gelu_grad2_64(zs[l - 1]).abs() * za[l - 1])
        ga, gs = ga + dh[:, obs.shape[1]:], gs + dha[:, obs.shape[1]:]
    return torch.stack(qs, 1), out, (ga, gs)


def worst(got, ref, scale, tol):
    return float(((got.double() - ref).abs() / (tol * scale + 1e-30)).max())


def run_kernel(module, kind, obs, act, grad_q, want_w, want_a):
    n_c = module.n_critics
    crit = Critic(module, obs.shape[1], act.shape[1], kind=kind, n_critics=n_c, n_quantiles=module.qf0[6].out_features)
    for p in module.parameters():
        p.requires_grad_(want_w)
        p.grad = None
    a = act.clone().requires_grad_(want_a)
    q = crit(obs, a)
    qt = torch.stack(q, 1) if kind == "sac" else q
    if grad_q is not None:
        qt.backward(grad_q)
    return qt.detach(), {n: p.grad for n, p in module.named_parameters()}, a.grad


def run_torch32(module, obs, act, grad_q):
    m = copy.deepcopy(module)
    a = act.clone().requires_grad_(True)
    q = m(obs, a)
    q.backward(grad_q)
    return q.detach(), {n: p.grad for n, p in m.named_parameters()}, a.grad


@pytest.fixture(autouse=True)
def no_tf32():
    old = torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = torch.backends.cudnn.allow_tf32 = False
    yield
    torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32 = old


def check_forward(module, kind, obs, act):
    with torch.no_grad():
        q, _, _ = run_kernel(module, kind, obs, act, None, False, False)
        q32 = module(obs, act)
    q64, _, _ = reference(module, obs, act, None)
    scale = max(1.0, float(q64.abs().max()))
    rk, rt = worst(q, q64, scale, TOL_Q), worst(q32, q64, scale, TOL_Q)
    print("forward worst ratio: kernel %.3f torch fp32 %.3f" % (rk, rt))
    assert rk <= 1.0 and rt <= 1.0, (rk, rt)


@pytest.mark.parametrize("obs_dim,act_dim", SHAPES)
def test_forward_shapes(obs_dim, act_dim):
    check_forward(make_critic(obs_dim, act_dim, 2, 25, obs_dim), "tqc", *batch(129, obs_dim, act_dim, 1))


@pytest.mark.parametrize("b", SIZES)
@pytest.mark.parametrize("cfg", CONFIGS, ids=["%s-%d-%d" % c for c in CONFIGS])
def test_forward_configs_and_sizes(cfg, b):
    kind, n_c, nq = cfg
    check_forward(make_critic(9, 6, n_c, nq, n_c * 7 + nq), kind, *batch(b, 9, 6, b))


def check_gradients(module, kind, obs, act, grad_q, want_w, want_a):
    q, grads, gact = run_kernel(module, kind, obs, act, grad_q, want_w, want_a)
    _, g32, a32 = run_torch32(module, obs, act, grad_q)
    _, ref, (ga64, gas) = reference(module, obs, act, grad_q)
    worst_k = worst_t = 0.0
    if want_w:
        for name, (g64, s) in ref.items():
            worst_k = max(worst_k, worst(grads[name], g64, s, TOL_G))
            worst_t = max(worst_t, worst(g32[name], g64, s, TOL_G))
    else:
        assert all(g is None for g in grads.values())
    if want_a:
        worst_k = max(worst_k, worst(gact, ga64, gas, TOL_G))
        worst_t = max(worst_t, worst(a32, ga64, gas, TOL_G))
    else:
        assert gact is None
    print("gradient worst ratio: kernel %.3f torch fp32 %.3f" % (worst_k, worst_t))
    assert worst_k <= 1.0 and worst_t <= 1.0, (worst_k, worst_t)


def real_grad_q(q, seed):
    """d loss / d q of TQC's loss on a random target (fp32 PyTorch autograd of the loss)."""
    g = torch.Generator(device=DEV).manual_seed(seed)
    target = q.detach().reshape(q.shape[0], -1) + torch.randn((q.shape[0], q.shape[1] * q.shape[2]), generator=g, device=DEV)
    cur = q.detach().clone().requires_grad_(True)
    quantile_huber_loss(cur, target.unsqueeze(1), sum_over_quantiles=False).backward()
    return cur.grad


MODES = [(False, True), (True, False), (True, True)]   # (weights, actions) require grad


@pytest.mark.parametrize("mode", MODES, ids=["actions", "params", "both"])
@pytest.mark.parametrize("cfg", CONFIGS, ids=["%s-%d-%d" % c for c in CONFIGS])
@pytest.mark.parametrize("b", (129, 4099))
def test_gradients_random_grad_q(cfg, mode, b):
    kind, n_c, nq = cfg
    module = make_critic(9, 6, n_c, nq, 3 + n_c)
    obs, act = batch(b, 9, 6, 2)
    g = torch.Generator(device=DEV).manual_seed(4)
    check_gradients(module, kind, obs, act, torch.randn((b, n_c, nq), generator=g, device=DEV), *mode)


@pytest.mark.parametrize("obs_dim,act_dim", SHAPES)
@pytest.mark.parametrize("b", (1, 128, 1000))
def test_gradients_of_the_tqc_loss(obs_dim, act_dim, b):
    module = make_critic(obs_dim, act_dim, 2, 25, 5)
    obs, act = batch(b, obs_dim, act_dim, 6)
    with torch.no_grad():
        q = module(obs, act)
    check_gradients(module, "tqc", obs, act, real_grad_q(q, 7), True, True)


def test_full_size_against_chunked_fp64():
    b, n_c, nq = 65536, 5, 25
    module = make_critic(9, 6, n_c, nq, 11)
    obs, act = batch(b, 9, 6, 12)
    g = torch.Generator(device=DEV).manual_seed(13)
    grad_q = torch.randn((b, n_c, nq), generator=g, device=DEV) / b
    q, grads, gact = run_kernel(module, "tqc", obs, act, grad_q, True, True)
    q64, ref, gas = None, {}, []
    qmax, rq = 0.0, []
    for s in range(0, b, 8192):
        qc, rc, (ga, gs) = reference(module, obs[s:s + 8192], act[s:s + 8192], grad_q[s:s + 8192])
        rq.append(qc)
        gas.append((ga, gs))
        for k, (gk, sk) in rc.items():
            g0, s0 = ref.get(k, (0.0, 0.0))
            ref[k] = (g0 + gk, s0 + sk)
    q64 = torch.cat(rq)
    assert worst(q, q64, max(1.0, float(q64.abs().max())), TOL_Q) <= 1.0
    wk = max(worst(grads[k], g64, s, TOL_G) for k, (g64, s) in ref.items())
    wa = worst(gact, torch.cat([x[0] for x in gas]), torch.cat([x[1] for x in gas]), TOL_G)
    print("full size worst ratio: weights %.3f actions %.3f" % (wk, wa))
    assert wk <= 1.0 and wa <= 1.0


def test_repeats_and_graph_replays_are_bitwise_equal():
    b, n_c, nq = 4099, 2, 25
    module = make_critic(9, 6, n_c, nq, 21)
    crit = Critic(module, 9, 6, kind="tqc", n_critics=n_c, n_quantiles=nq)
    obs, act0 = batch(b, 9, 6, 22)
    act = act0.clone().requires_grad_(True)
    grad_q = torch.randn((b, n_c, nq), device=DEV)

    def step():
        for p in module.parameters():
            p.grad = None
        act.grad = None
        crit(obs, act).backward(grad_q)
        return [p.grad for p in module.parameters()] + [act.grad]

    first = [t.clone() for t in step()]
    second = [t.clone() for t in step()]
    for x, y in zip(first, second):
        assert torch.equal(bits(x), bits(y))
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        step()
    torch.cuda.current_stream().wait_stream(s)
    for p in module.parameters():
        p.grad = None
    act.grad = None
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        crit(obs, act).backward(grad_q)
    for _ in range(2):
        graph.replay()
        torch.cuda.synchronize()
        for x, y in zip([p.grad for p in module.parameters()] + [act.grad], first):
            assert torch.equal(bits(x), bits(y))


def test_captured_tqc_critic_update():
    """sample -> CriticTarget -> Critic -> quantile_huber_loss -> backward -> Adam(capturable) -> Polyak -> sync_weights,
    captured and replayed R times, equals R eager updates bit for bit; 20 updates stay within a bound of the same 20
    updates in fp64 PyTorch (fed the same samples and targets), a bound that fp32 PyTorch also meets."""
    n_c, nq, drop, bs, R, tau = 2, 25, 2, 256, 4, 0.005
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
    actor = SquashedGaussianPolicy(obs_dim, act_dim, device=DEV, precision="fp32", seed=2)
    critic0 = make_critic(obs_dim, act_dim, n_c, nq, 31)
    alpha = torch.tensor([0.2], device=DEV)

    def twin(kernel=True, dtype=torch.float32, log=None):
        buf = ReplayBuffer(slots * 512, env, seed=3)
        buf.load_state_dict(state)
        critic = copy.deepcopy(critic0).to(dtype)
        critic_t = copy.deepcopy(critic0).to(dtype)
        tsd = critic_t.state_dict()
        tgt = CriticTarget(actor, kind="tqc", n_critics=n_c, n_quantiles=nq, top_quantiles_to_drop_per_net=drop)
        tgt.load_state_dict(tsd if dtype == torch.float32 else {k: v.float() for k, v in tsd.items()}, share=dtype == torch.float32)
        opt = torch.optim.Adam(critic.parameters(), lr=3e-4, capturable=True)
        crit = Critic(critic, obs_dim, act_dim, kind="tqc", n_critics=n_c, n_quantiles=nq) if kernel else critic
        params, tparams = list(critic.parameters()), list(critic_t.parameters())

        def step(replay=None):
            if replay is None:
                batch = buf.sample(bs)
                y = tgt(batch, alpha)
                if log is not None:
                    log.append((batch.observations.clone(), batch.actions.clone(), y.clone()))
                o, a = batch.observations, batch.actions
            else:   # the fp64 twin: the same samples and targets
                o, a, y = [t.to(dtype) for t in replay]
            current = crit(o, a)
            loss = quantile_huber_loss(current.float(), y.float().unsqueeze(1), sum_over_quantiles=False) if dtype == torch.float32 else \
                sb3_loss64(current, y.unsqueeze(1))
            opt.zero_grad(set_to_none=False)
            loss.backward()
            opt.step()
            with torch.no_grad():
                torch._foreach_lerp_(tparams, params, tau)
            if dtype == torch.float32:
                tgt.sync_weights()
            return loss.detach()
        return critic, step

    critic_e, step_e = twin()
    eager = []
    for _ in range(R + 3):
        loss = step_e()
        eager.append((loss.clone(), [p.detach().clone() for p in critic_e.parameters()]))
    critic_g, step_g = twin()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        for _ in range(3):
            step_g()
    torch.cuda.current_stream().wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        loss_g = step_g()
    for r in range(R):
        graph.replay()
        torch.cuda.synchronize()
        assert torch.equal(bits(loss_g), bits(eager[3 + r][0])), r
        for p, q in zip(critic_g.parameters(), eager[3 + r][1]):
            assert torch.equal(bits(p.detach()), bits(q)), r

    # 20 updates: kernel and fp32 PyTorch against fp64 PyTorch on the same samples and targets
    log = []
    critic_k, step_k = twin(log=log)
    for _ in range(20):
        step_k()
    critic_32, step_32 = twin(kernel=False)
    critic_64, step_64 = twin(kernel=False, dtype=torch.float64)
    for rec in log:
        step_32(rec)
        step_64(rec)
    # Adam moves each parameter by about lr per step whatever the gradient's size, so the bound is a share of the movement
    worst_k = worst_t = 0.0
    for pk, p32, p64, p0 in zip(critic_k.parameters(), critic_32.parameters(), critic_64.parameters(), critic0.parameters()):
        scale = (p64.detach() - p0.detach().double()).abs().max() + 1e-12
        worst_k = max(worst_k, float((pk.detach().double() - p64.detach()).abs().max() / scale))
        worst_t = max(worst_t, float((p32.detach().double() - p64.detach()).abs().max() / scale))
    print("20 updates: worst |p - p64| / max |p64 - p0|: kernel %.3g torch fp32 %.3g" % (worst_k, worst_t))
    assert worst_k <= 0.05 and worst_t <= 0.05, (worst_k, worst_t)


def sb3_loss64(current, target):
    """sb3_contrib's quantile_huber_loss (sum_over_quantiles=False) in fp64."""
    nq = current.shape[-1]
    cum_prob = (torch.arange(nq, device=current.device, dtype=current.dtype) + 0.5) / nq
    cum_prob = cum_prob.view(1, 1, -1, 1)
    delta = target.unsqueeze(-2) - current.unsqueeze(-1)
    abs_delta = delta.abs()
    huber = torch.where(abs_delta > 1, abs_delta - 0.5, delta ** 2 * 0.5)
    return (torch.abs(cum_prob - (delta.detach() < 0).to(current.dtype)) * huber).mean()


def test_sac_tuple_form_critic_loss_and_actor_loss():
    """SB3 SAC's critic loss 0.5 sum(F.mse_loss(q, y) for q in critic(obs, a)) and its actor loss on th.cat(critic(obs, a_pi), 1)
    give fp32 PyTorch's gradients within twice TOL_G (both are within TOL_G of fp64), scaled with the loss's d loss / d q."""
    b, n_c = 300, 2
    module = make_critic(9, 6, n_c, 1, 41)
    crit = Critic(module, 9, 6, kind="sac", n_critics=n_c)
    obs, act = batch(b, 9, 6, 42)
    y = torch.randn((b, 1), device=DEV)
    qs = crit(obs, act)
    assert isinstance(qs, tuple) and len(qs) == n_c and all(q.shape == (b, 1) for q in qs)
    (0.5 * sum(F.mse_loss(q, y) for q in qs)).backward()
    ref = copy.deepcopy(module)
    q_ref = ref(obs, act)
    (0.5 * sum(F.mse_loss(q_ref[:, i], y) for i in range(n_c))).backward()
    _, scales, _ = reference(module, obs, act, (q_ref.detach() - y.unsqueeze(1)) / b)
    for (n, p), pr in zip(module.named_parameters(), ref.parameters()):
        assert worst(p.grad, pr.grad.double(), scales[n][1], 2 * TOL_G) <= 1.0, n
    # actor loss: (ent_coef * log_prob - min_qf_pi).mean(); the critic parameters frozen
    for p in module.parameters():
        p.requires_grad_(False)
    a_pi = act.clone().requires_grad_(True)
    (-torch.cat(crit(obs, a_pi), 1).min(1, keepdim=True)[0].mean()).backward()
    a_ref = act.clone().requires_grad_(True)
    q_pi = ref(obs, a_ref)[:, :, 0]
    (-q_pi.min(1, keepdim=True)[0].mean()).backward()
    g_q = torch.zeros((b, n_c, 1), device=DEV)
    g_q[torch.arange(b), q_pi.argmin(1), 0] = -1.0 / b
    _, _, (_, ga_scale) = reference(module, obs, act, g_q)
    assert worst(a_pi.grad, a_ref.grad.double(), ga_scale, 2 * TOL_G) <= 1.0


def test_in_place_change_between_forward_and_backward_raises():
    module = make_critic(9, 6, 2, 25, 51)
    crit = Critic(module, 9, 6, kind="tqc", n_critics=2, n_quantiles=25)
    obs, act = batch(64, 9, 6, 52)
    q = crit(obs, act)
    with torch.no_grad():
        module.qf1[2].weight.mul_(1.5)
    with pytest.raises(RuntimeError, match="modified by an inplace operation"):
        q.sum().backward()


def test_no_grad_saves_nothing_and_module_or_mapping():
    module = make_critic(9, 6, 2, 25, 61)
    obs, act = batch(200, 9, 6, 62)
    by_module = Critic(module, 9, 6, kind="tqc", n_critics=2, n_quantiles=25)
    by_map = Critic({"critic." + k: v for k, v in module.named_parameters()}, 9, 6, kind="tqc", n_critics=2, n_quantiles=25)
    with torch.no_grad():
        q = by_module(obs, act)
    assert q.grad_fn is None
    assert torch.equal(bits(q), bits(by_map(obs, act).detach()))


def test_refusals():
    module = make_critic(9, 6, 2, 25, 71)
    crit = Critic(module, 9, 6, kind="tqc", n_critics=2, n_quantiles=25)
    obs, act = batch(16, 9, 6, 72)
    crit(obs, act)   # packs the weights: the C checks below are past "no weights"
    for bad_obs, bad_act, what in ((obs.clone().requires_grad_(True), act, "obs requires grad"), (obs.double(), act, "float32"),
                                   (obs, act.double(), "float32"), (obs.cpu(), act, "is on"), (obs, act.cpu(), "is on"),
                                   (obs[:, :5], act, r"\[B, 9\]"), (obs, act[:8], "same batch size"),
                                   (obs[:0], act[:0], "same batch size")):
        with pytest.raises(ValueError, match=what):
            crit(bad_obs, bad_act)
    with pytest.raises(ValueError, match="CUDA device"):
        Critic(copy.deepcopy(module).cpu(), 9, 6, kind="tqc", n_critics=2, n_quantiles=25)
    with pytest.raises(ValueError, match="n_critics"):
        Critic(module, 9, 6, kind="tqc", n_critics=6, n_quantiles=25)
    with pytest.raises(ValueError, match="obs_dim \\+ act_dim"):
        Critic(module, 12, 6, kind="tqc", n_critics=2, n_quantiles=25)
    # C: bad sizes, missing weights, non-device pointers
    lib = _lib.load()
    b = 16
    q = torch.empty((b, 2, 25), device=DEV)
    saved = torch.empty(int(lib.mvrl_critic_saved_bytes(crit._h, b)), dtype=torch.uint8, device=DEV)
    scratch = torch.empty(int(lib.mvrl_critic_grad_scratch(crit._h, b)), dtype=torch.uint8, device=DEV)
    ga = torch.empty((b, 6), device=DEV)
    s = _lib.current_stream(torch.device(DEV))
    P = _lib.ptr
    assert lib.mvrl_critic_forward(crit._h, 0, P(obs), P(act), P(q), None, s) == -1
    assert lib.mvrl_critic_forward(crit._h, b, P(obs.cpu()), P(act), P(q), None, s) == -1
    assert "obs is not device memory" in lib.mvrl_last_error().decode()
    assert lib.mvrl_critic_forward(crit._h, b, P(obs), P(act), None, None, s) == -1
    assert lib.mvrl_critic_backward(crit._h, b, P(obs), P(act), P(saved), P(q), None, None, P(scratch), s) == -1
    assert lib.mvrl_critic_backward(crit._h, -1, P(obs), P(act), P(saved), P(q), None, P(ga), P(scratch), s) == -1
    assert lib.mvrl_critic_backward(crit._h, b, P(obs), P(act), P(saved), P(q), None, P(ga), P(scratch.cpu()), s) == -1
    host = torch.zeros(16)
    grads = (C.c_void_p * 16)(*([host.data_ptr()] * 16))
    assert lib.mvrl_critic_backward(crit._h, b, P(obs), P(act), P(saved), P(q), grads, None, P(scratch), s) == -1
    fresh = _lib.Handle("mvrl_critic", 0, 9, 6, 1, 2, 25)
    assert lib.mvrl_critic_forward(fresh._h, b, P(obs), P(act), P(q), None, s) == -1
    assert "no weights" in lib.mvrl_last_error().decode()
