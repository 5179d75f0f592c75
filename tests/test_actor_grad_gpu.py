"""GPU: ``Actor`` (csrc/mvrl_policy.cu, critic_forward_kernel / critic_backward_kernel / critic_grad_reduce_kernel
instantiated for the actor) against an fp64 restatement of SB3's ``Actor.action_log_prob`` fed the kernel's own eps -
actions, log-prob and every parameter gradient over shapes, batch sizes and the three combinations of output gradients; eps
against the NumPy Philox stream 11; both clamp bounds of log_std and saturated actions; bitwise repeats and graph replays;
the actor loss through ``Critic``; a whole captured SAC / TQC gradient step against its eager twin and 20 steps against
fp64; the refusals in Python and C."""
import copy
import ctypes as C

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from test_actor_grad_cpu import SB3Actor, stream11_pair

pytestmark = pytest.mark.gpu

if torch.cuda.is_available():
    from marinevehiclereinforcementlearning_b200 import (Actor, BlueROV2Heavy6DoFVecEnv, Critic, CriticTarget, ReplayBuffer,
                                                         SquashedGaussianPolicy, _lib)
    from marinevehiclereinforcementlearning_b200.policy import quantile_huber_loss
    from test_critic_grad_gpu import TOL_G, bits, make_critic, sb3_loss64
    from test_critic_grad_gpu import reference as critic_reference
    from test_critic_target_gpu import actor_state_dict
    from test_random_streams_gpu import draw_bound

DEV = "cuda"
SHAPES = [(9, 6), (11, 3), (5, 3), (1, 1), (10, 6)]
SIZES = (1, 127, 128, 129, 4099)
# Forward: the fp32 actor's bounds of the critic target's tests (the same head code): |a - fp64| <= TOL_A and |logp - fp64|
# <= 4 TOL_A act_dim max(1, |logp|).  Gradients: |g - fp64| <= TOL_G S element-wise with K12's absolute-value scales S,
# extended through the head (reference() below): the head's dZ scale is the fp64 sum of absolute terms of g_mu / g_ls plus
# the forward's rounding carried through their derivative with respect to a - relative (TOL) to |x|abs = |mu|abs + exp(ls)
# |eps| |ls|abs through 1 - a^2, and a's own fp32 rounding, 2^-22 absolute (tanhf within 2 ulp, ulp <= 2^-24 below 1, and
# 1 - a^2 doubles it), divided by TOL_G.  That last term is what makes a saturated component (|x| >= 8: a within a few ulps
# of +-1, 1 - a^2 of the order of its rounding) finite but loose: there the fp32 forward cannot resolve 1 - a^2, in the
# kernel and in PyTorch alike.  fp32 PyTorch (TF32 off) passes the same bounds (asserted below).
TOL_A = 5e-5
MODES = {"actions": (True, False), "log_prob": (False, True), "both": (True, True)}


def make_actor(obs_dim, act_dim, seed):
    m = SB3Actor(obs_dim, act_dim)
    m.load_state_dict(actor_state_dict(obs_dim, act_dim, seed))
    return m.to(DEV)


def observations(b, obs_dim, seed):
    g = torch.Generator(device=DEV).manual_seed(seed)
    return torch.rand((b, obs_dim), generator=g, device=DEV) * 2 - 1


def torch_action_log_prob(m, obs, eps):
    """SB3's Actor.action_log_prob in the module's dtype with the given eps, written as SB3 writes it: rsample, tanh,
    Normal.log_prob summed minus the tanh correction (without argument validation, a host synchronisation a CUDA graph
    cannot hold)."""
    h = m.latent_pi(obs.to(m.mu.weight.dtype))
    mu = m.mu(h)
    std = m.log_std(h).clamp(-20.0, 2.0).exp()
    x = mu + std * eps.to(mu.dtype)
    a = torch.tanh(x)
    lp = torch.distributions.Normal(mu, std, validate_args=False).log_prob(x).sum(1) - torch.log(1.0 - a * a + 1e-6).sum(1)
    return a, lp


def gelu_grad64(z):
    return 0.5 * (1.0 + torch.erf(z / 2 ** 0.5)) + z * torch.exp(-0.5 * z * z) / (2 * torch.pi) ** 0.5


def gelu_grad2_64(z):
    return (2.0 - z * z) * torch.exp(-0.5 * z * z) / (2 * torch.pi) ** 0.5


def reference(m, obs, eps, g_a, g_lp, g_a_abs=None):
    """fp64: actions, log_prob, {param name: (grad, scale)} for the loss sum(g_a a) + sum(g_lp log_prob) (g_a / g_lp None:
    that output does not enter).  The gradients are torch's fp64 autograd of the literal restatement; the scales follow the
    module docstring.  ``g_a_abs``: a bound on |g_a| entry by entry if g_a itself carries an error (the actor loss chain)."""
    m64 = copy.deepcopy(m).double()
    a, lp = torch_action_log_prob(m64, obs.double(), eps.double())
    params = list(m64.parameters())
    names = [n for n, _ in m64.named_parameters()]
    outs = [(t, g.double()) for t, g in ((a, g_a), (lp, g_lp)) if g is not None]
    grads = torch.autograd.grad([t for t, _ in outs], params, [g for _, g in outs])
    P = {n: p.detach() for n, p in m64.named_parameters()}
    b = obs.shape[0]
    ga = torch.zeros_like(a) if g_a is None else g_a.double()
    ga_abs = ga.abs() if g_a_abs is None else g_a_abs.double()
    gl = torch.zeros(b, dtype=torch.float64, device=DEV) if g_lp is None else g_lp.double()
    with torch.no_grad():
        h, hs, has, zs, za = obs.double(), [], [], [], []
        hs.append(h)
        has.append(h.abs())
        for l, j in enumerate((0, 2, 4)):
            W, bb = P["latent_pi.%d.weight" % j], P["latent_pi.%d.bias" % j]
            z = h @ W.T + bb
            zs.append(z)
            za.append(h.abs() @ W.abs().T + bb.abs())
            h = F.gelu(z)
            hs.append(h)
            has.append(h.abs() + gelu_grad64(z).abs() * za[l])
        mu_abs = h.abs() @ P["mu.weight"].abs().T + P["mu.bias"].abs()
        ls_pre = h @ P["log_std.weight"].T + P["log_std.bias"]
        ls_abs = h.abs() @ P["log_std.weight"].abs().T + P["log_std.bias"].abs()
        s = ls_pre.clamp(-20.0, 2.0).exp()
        e = eps.double().abs()
        ad = a.detach()
        om = 1.0 - ad * ad
        f = om / (om + 1e-6)
        gx = ga * om + gl[:, None] * 2 * ad * f
        sens_a = 2 * ga_abs * ad.abs() + 2 * gl.abs()[:, None] * (f + 2 * ad * ad * 1e-6 / (om + 1e-6) ** 2)
        s_gx = ga_abs * om + 2 * gl.abs()[:, None] * ad.abs() * f + sens_a * (om * (mu_abs + s * e * ls_abs) + 2.0 ** -22 / TOL_G)
        inside = ((ls_pre >= -20.0) & (ls_pre <= 2.0)).double()
        s_ls = (s_gx * s * e + gx.abs() * s * e * ls_abs + gl.abs()[:, None]) * inside
        scales = {"mu.weight": s_gx.T @ has[3], "mu.bias": s_gx.sum(0), "log_std.weight": s_ls.T @ has[3], "log_std.bias": s_ls.sum(0)}
        dha = s_gx @ P["mu.weight"].abs() + s_ls @ P["log_std.weight"].abs()
        for l in (2, 1, 0):
            dza = dha * (gelu_grad64(zs[l]).abs() + gelu_grad2_64(zs[l]).abs() * za[l])
            j = 2 * l
            scales["latent_pi.%d.weight" % j], scales["latent_pi.%d.bias" % j] = dza.T @ has[l], dza.sum(0)
            dha = dza @ P["latent_pi.%d.weight" % j].abs()
    return a.detach(), lp.detach(), {n: (g, scales[n]) for n, g in zip(names, grads)}


def worst(got, ref, scale, tol):
    return float(((got.double() - ref).abs() / (tol * scale + 1e-30)).max())


@pytest.fixture(autouse=True)
def no_tf32():
    old = torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = torch.backends.cudnn.allow_tf32 = False
    yield
    torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32 = old


def check_forward(m, actor, obs, call):
    b, act_dim = obs.shape[0], actor.act_dim
    eps = torch.full((b, act_dim), 7.0, device=DEV)
    actor.calls.copy_(torch.tensor([call, 0]))
    with torch.no_grad():
        a, lp = actor.action_log_prob(obs, eps=eps)
    assert a.grad_fn is None and lp.grad_fn is None and a.shape == (b, act_dim) and lp.shape == (b,)
    assert int(actor.calls[0]) == call + 1 and int(actor.calls[1]) == 0
    e_np = eps.cpu().numpy().astype(np.float64)
    for pr in range((act_dim + 1) // 2):
        k1, k2, z0, z1 = stream11_pair(actor.seed, np.arange(b), call, pr)
        for c, z in enumerate((z0, z1)):
            if 2 * pr + c < act_dim:
                d = np.abs(e_np[:, 2 * pr + c] - z)
                assert np.all(d <= draw_bound(k1, k2, z)), (pr, c)
    a64, lp64, _ = reference(m, obs, eps, None, torch.ones(b, device=DEV))
    e_a = float((a.double() - a64).abs().max())
    e_lp = float(((lp.double() - lp64).abs() / lp64.abs().clamp(min=1.0)).max())
    assert e_a <= TOL_A and e_lp <= 4 * TOL_A * act_dim, (e_a, e_lp)
    return e_a, e_lp


@pytest.mark.parametrize("obs_dim,act_dim", SHAPES)
def test_forward_and_eps_over_shapes_and_sizes(obs_dim, act_dim):
    """actions and log_prob against fp64 fed the kernel's eps, eps against NumPy stream 11, at calls on both sides of 2^32."""
    m = make_actor(obs_dim, act_dim, obs_dim * 10 + act_dim)
    actor = Actor(m, obs_dim, act_dim, seed=0xD1B54A32D192ED03)
    worst_a = worst_lp = 0.0
    for i, b in enumerate(SIZES):
        e_a, e_lp = check_forward(m, actor, observations(b, obs_dim, b), (0, 1, 2 ** 32 - 1, 2 ** 32 + 3, 5)[i])
        worst_a, worst_lp = max(worst_a, e_a), max(worst_lp, e_lp)
    print("forward (%d, %d): max |a - fp64| %.3g, rel |logp - fp64| %.3g" % (obs_dim, act_dim, worst_a, worst_lp))


def run_kernel(m, obs, g_a, g_lp, eps=None):
    actor = Actor(m, obs.shape[1], m.mu.out_features)
    if eps is None:
        eps = torch.empty((obs.shape[0], actor.act_dim), device=DEV)
    a, lp = actor.action_log_prob(obs, eps=eps)
    outs = [(t, g) for t, g in ((a, g_a), (lp, g_lp)) if g is not None]
    grads = torch.autograd.grad([t for t, _ in outs], list(m.parameters()), [g for _, g in outs])
    return eps, dict(zip([n for n, _ in m.named_parameters()], grads))


def run_torch32(m, obs, eps, g_a, g_lp):
    a, lp = torch_action_log_prob(m, obs, eps)
    outs = [(t, g) for t, g in ((a, g_a), (lp, g_lp)) if g is not None]
    grads = torch.autograd.grad([t for t, _ in outs], list(m.parameters()), [g for _, g in outs])
    return dict(zip([n for n, _ in m.named_parameters()], grads))


def check_gradients(m, obs, g_a, g_lp, torch_too=True):
    eps, grads = run_kernel(m, obs, g_a, g_lp)
    g32 = run_torch32(m, obs, eps, g_a, g_lp)
    _, _, ref = reference(m, obs, eps, g_a, g_lp)
    wk = max(worst(grads[n], g64, s, TOL_G) for n, (g64, s) in ref.items())
    wt = max(worst(g32[n], g64, s, TOL_G) for n, (g64, s) in ref.items())
    print("gradient worst ratio: kernel %.3f torch fp32 %.3f" % (wk, wt))
    assert wk <= 1.0 and (wt <= 1.0 or not torch_too), (wk, wt)
    return grads, ref, g32


def output_grads(b, act_dim, mode, seed):
    g = torch.Generator(device=DEV).manual_seed(seed)
    want_a, want_lp = MODES[mode]
    g_a = torch.randn((b, act_dim), generator=g, device=DEV) if want_a else None
    g_lp = torch.randn((b,), generator=g, device=DEV) if want_lp else None
    return g_a, g_lp


@pytest.mark.parametrize("mode", list(MODES))
@pytest.mark.parametrize("b", (1, 129, 4099))
def test_gradients_random_output_grads(mode, b):
    m = make_actor(9, 6, 3)
    check_gradients(m, observations(b, 9, 2), *output_grads(b, 6, mode, 4))


@pytest.mark.parametrize("obs_dim,act_dim", SHAPES)
def test_gradients_over_shapes(obs_dim, act_dim):
    m = make_actor(obs_dim, act_dim, 5)
    check_gradients(m, observations(300, obs_dim, 6), *output_grads(300, act_dim, "both", 7))


def test_clamp_bounds_and_saturated_actions():
    """log_std columns whose pre-activation is beyond either clamp bound (3, -25: zero gradient, exactly) and exactly at
    either bound (2, -20: torch's clamp passes the gradient); mu columns at +-9 with a small std (|x| >= 8, a within a few
    ulps of +-1): finite gradients within the bound of the module docstring."""
    act_dim = 6
    m = make_actor(9, act_dim, 8)
    with torch.no_grad():
        m.log_std.weight.zero_()
        m.log_std.bias.copy_(torch.tensor([3.0, -25.0, 2.0, -20.0, -3.0, -3.0]))
        m.mu.weight[4:].zero_()
        m.mu.bias[4:] = torch.tensor([9.0, -9.0])
    b = 300
    obs = observations(b, 9, 9)
    # the kernel only: fp32 PyTorch cannot be held to a bound in the column at -20.  There std = exp(-20) puts std eps far
    # below the ulp of mu, so in SB3's fp32 graph x - mu is 0 or a multiple of ulp(mu), and the Normal term's two paths to
    # mu (through x and directly), each ~|g_lp| ulp(mu) / std^2 ~ 1e10, cancel catastrophically: its mu gradient there and
    # everything below it is noise.  The kernel's reduced formula (g_mu = g_x) has neither term.
    grads, ref, _ = check_gradients(m, obs, *output_grads(b, act_dim, "both", 10), torch_too=False)
    for k in (0, 1):
        assert torch.equal(grads["log_std.bias"][k], torch.zeros((), device=DEV))
        assert not bool(grads["log_std.weight"][k].any())
    for k in (2, 3):
        assert float(grads["log_std.bias"][k].abs()) > 0 and float(ref["log_std.bias"][0][k].abs()) > 0
    assert all(bool(torch.isfinite(g).all()) for g in grads.values())
    eps = torch.empty((b, act_dim), device=DEV)
    with torch.no_grad():
        a, _ = Actor(m, 9, act_dim).action_log_prob(obs, eps=eps)
    x = m.mu.bias[4:].detach() + np.exp(-3.0) * eps[:, 4:]
    assert bool((x.abs() >= 8).all()) and float((1 - a[:, 4:].abs()).max()) <= 4 * 2.0 ** -24


def test_full_size_against_chunked_fp64():
    b = 65536
    m = make_actor(9, 6, 11)
    obs = observations(b, 9, 12)
    g_a, g_lp = output_grads(b, 6, "both", 13)
    g_a, g_lp = g_a / b, g_lp / b
    eps, grads = run_kernel(m, obs, g_a, g_lp)
    ref = {}
    for s in range(0, b, 8192):
        _, _, rc = reference(m, obs[s:s + 8192], eps[s:s + 8192], g_a[s:s + 8192], g_lp[s:s + 8192])
        for k, (gk, sk) in rc.items():
            g0, s0 = ref.get(k, (0.0, 0.0))
            ref[k] = (g0 + gk, s0 + sk)
    wk = max(worst(grads[k], g64, s, TOL_G) for k, (g64, s) in ref.items())
    print("full size worst ratio: %.3f" % wk)
    assert wk <= 1.0


def test_repeats_and_graph_replays():
    """The same call number gives the same bits; T = 2 calls captured and replayed R = 3 times give the bits of 6 eager
    calls (new eps on every replay)."""
    b = 4099
    m = make_actor(9, 6, 21)
    actor = Actor(m, 9, 6, seed=5)
    obs = observations(b, 9, 22)
    g_a, g_lp = output_grads(b, 6, "both", 23)
    params = list(m.parameters())

    def call():
        a, lp = actor.action_log_prob(obs)
        return [a.detach(), lp.detach()] + list(torch.autograd.grad([a, lp], params, [g_a, g_lp]))

    actor.calls.zero_()
    first = [t.clone() for t in call()]
    actor.calls.zero_()
    for x, y in zip(call(), first):
        assert torch.equal(bits(x), bits(y))
    T, R = 2, 3
    actor.calls.zero_()
    eager = [[t.clone() for t in call()] for _ in range(T * R)]
    assert int(actor.calls[0]) == T * R
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        call()
    torch.cuda.current_stream().wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        outs = [call() for _ in range(T)]
    actor.calls.zero_()
    for r in range(R):
        graph.replay()
        torch.cuda.synchronize()
        for t in range(T):
            for x, y in zip(outs[t], eager[r * T + t]):
                assert torch.equal(bits(x), bits(y)), (r, t)
    assert int(actor.calls[0]) == T * R
    assert not torch.equal(eager[0][0], eager[1][0])


@pytest.mark.parametrize("kind", ["sac", "tqc"])
def test_actor_loss_through_critic(kind):
    """SAC's (alpha log_prob - min_c q_c).mean() and TQC's (alpha log_prob - q.mean(2).mean(1)).mean() with q = Critic(obs,
    actions_pi): the actor gradients against the fp64 chain (fp64 actor and critics, the kernel's eps) within twice TOL_G
    of the scales, with d loss / d a's own bound (K12's action-gradient scale) carried into the actor's."""
    b, alpha = 500, 0.2
    n_c, nq = (2, 1) if kind == "sac" else (2, 25)
    m = make_actor(9, 6, 31)
    critic_m = make_critic(9, 6, n_c, nq, 32)
    for p in critic_m.parameters():
        p.requires_grad_(False)
    crit = Critic(critic_m, 9, 6, kind=kind, n_critics=n_c, n_quantiles=nq)
    actor = Actor(m, 9, 6)
    obs = observations(b, 9, 33)
    eps = torch.empty((b, 6), device=DEV)
    a, lp = actor.action_log_prob(obs, eps=eps)

    def q_pi(q):
        return torch.cat(q, 1).min(1, keepdim=True)[0] if kind == "sac" else q.mean(2).mean(1, keepdim=True)

    loss = (alpha * lp.unsqueeze(1) - q_pi(crit(obs, a))).mean()
    grads = dict(zip([n for n, _ in m.named_parameters()], torch.autograd.grad(loss, list(m.parameters()))))
    # fp64 chain: d loss / d q of the fp64 critics at the fp64 actions, then the actor's reference with that g_a
    a64 = reference(m, obs, eps, None, torch.ones(b, device=DEV))[0]
    cm64 = copy.deepcopy(critic_m).double()
    a_req = a64.clone().requires_grad_(True)
    q64 = cm64(obs.double(), a_req)
    q64t = q64[:, :, 0] if kind == "sac" else q64
    qp = q64t.min(1, keepdim=True)[0] if kind == "sac" else q64t.mean(2).mean(1, keepdim=True)
    ga64 = torch.autograd.grad(-qp.mean(), a_req)[0]
    g_q = torch.zeros((b, n_c, nq), dtype=torch.float64, device=DEV)
    if kind == "sac":
        g_q[torch.arange(b), q64t.argmin(1), 0] = -1.0 / b
    else:
        g_q[:] = -1.0 / (b * n_c * nq)
    _, _, (_, gas) = critic_reference(cm64, obs.double(), a64, g_q)
    # the kernel's d loss / d a is within TOL_G gas of ga64 (K12's bound), an error that enters the actor's gradients
    # linearly: |ga64| + gas in place of |g_a| in the scales
    _, _, ref = reference(m, obs, eps, ga64, torch.full((b,), alpha / b, device=DEV), g_a_abs=ga64.abs() + gas)
    wk = max(worst(grads[n], g64, s, 2 * TOL_G) for n, (g64, s) in ref.items())
    print("actor loss (%s) worst ratio: %.3f" % (kind, wk))
    assert wk <= 1.0


@pytest.mark.parametrize("kind", ["sac", "tqc"])
def test_captured_gradient_step(kind):
    """sample -> CriticTarget -> Critic -> critic loss -> critic Adam -> Actor.action_log_prob -> actor loss -> actor Adam ->
    entropy-coefficient loss and Adam -> Polyak -> sync_weights, every network pass on the library's kernels, captured and
    replayed R times, equals R eager steps bit for bit; 20 steps stay within a share of an fp64 PyTorch twin's parameter
    movement (fed the same samples, targets and actor eps), a share fp32 PyTorch also meets."""
    n_c, nq, drop = (2, 1, 0) if kind == "sac" else (2, 25, 2)
    bs, R, tau, slots = 256, 4, 0.005, 8
    env = BlueROV2Heavy6DoFVecEnv(512, action_mode="force", dtype=torch.float32, seed=1)
    obs_dim, act_dim = env.lenObs, env.lenAction
    g = torch.Generator(device=DEV).manual_seed(0)
    state = {"observations": torch.rand((slots, 512, obs_dim), generator=g, device=DEV) * 2 - 1,
             "actions": torch.rand((slots, 512, act_dim), generator=g, device=DEV) * 2 - 1,
             "rewards": torch.rand((slots, 512), generator=g, device=DEV) * 2 - 1,
             "dones": (torch.rand((slots, 512), generator=g, device=DEV) < 0.1).to(torch.uint8),
             "timeouts": torch.zeros((slots, 512), dtype=torch.uint8, device=DEV),
             "last_obs": torch.zeros((obs_dim, env.ld), device=DEV),
             "cursor": torch.tensor([0, slots, 0, 0, 0], dtype=torch.int64), "seed": 3}
    state["next_observations"] = torch.rand((slots, 512, obs_dim), generator=g, device=DEV) * 2 - 1
    actor0 = make_actor(obs_dim, act_dim, 30)
    critic0 = make_critic(obs_dim, act_dim, n_c, nq, 31)
    target_entropy = -float(act_dim)

    def twin(kernel=True, dtype=torch.float32, log=None):
        buf = ReplayBuffer(slots * 512, env, seed=3)
        buf.load_state_dict(state)
        actor_m = copy.deepcopy(actor0).to(dtype)
        critic, critic_t = copy.deepcopy(critic0).to(dtype), copy.deepcopy(critic0).to(dtype)
        log_ent = torch.zeros(1, dtype=dtype, device=DEV, requires_grad=True)
        opt_c = torch.optim.Adam(critic.parameters(), lr=3e-4, capturable=True)
        opt_a = torch.optim.Adam(actor_m.parameters(), lr=3e-4, capturable=True)
        opt_e = torch.optim.Adam([log_ent], lr=3e-4, capturable=True)
        if dtype == torch.float32:
            actor_t = SquashedGaussianPolicy(obs_dim, act_dim, device=DEV, precision="fp32", seed=2)
            actor_t.load_state_dict(dict(actor_m.named_parameters()), share=True)
            tgt = CriticTarget(actor_t, kind=kind, n_critics=n_c, n_quantiles=nq, top_quantiles_to_drop_per_net=drop)
            tgt.load_state_dict(critic_t.state_dict(), share=True)
        crit = Critic(critic, obs_dim, act_dim, kind=kind, n_critics=n_c, n_quantiles=nq) if kernel else critic
        act = Actor(actor_m, obs_dim, act_dim, seed=4) if kernel else None
        params, tparams = list(critic.parameters()), list(critic_t.parameters())

        def q_of(o, a):
            q = crit(o, a)
            return torch.stack(q, 1) if isinstance(q, tuple) else q

        def step(replay=None):
            if replay is None:
                batch = buf.sample(bs)
                y = tgt(batch, log_ent.detach().exp())
                o, a_b = batch.observations, batch.actions
            else:
                o, a_b, y, eps = [t.to(dtype) for t in replay]
            q = q_of(o, a_b)
            if kind == "tqc":
                loss_c = sb3_loss64(q, y.unsqueeze(1)) if dtype == torch.float64 else quantile_huber_loss(q, y.unsqueeze(1), sum_over_quantiles=False)
            else:
                loss_c = 0.5 * sum(F.mse_loss(q[:, i], y) for i in range(n_c))
            opt_c.zero_grad(set_to_none=False)
            loss_c.backward()
            opt_c.step()
            if replay is None:
                eps = torch.empty((o.shape[0], act_dim), device=DEV)
                a_pi, lp = act.action_log_prob(o, eps=eps)
                if log is not None:
                    log.append((o.clone(), a_b.clone(), y.clone(), eps.clone()))
            else:
                a_pi, lp = torch_action_log_prob(actor_m, o, eps)
            alpha = log_ent.detach().exp()
            q_pi = q_of(o, a_pi)
            q_pi = q_pi.min(1)[0] if kind == "sac" else q_pi.mean(2).mean(1, keepdim=True)
            loss_a = (alpha * lp.unsqueeze(1) - q_pi).mean()
            opt_a.zero_grad(set_to_none=False)
            loss_a.backward()
            opt_a.step()
            loss_e = -(log_ent * (lp + target_entropy).detach()).mean()
            opt_e.zero_grad(set_to_none=False)
            loss_e.backward()
            opt_e.step()
            with torch.no_grad():
                torch._foreach_lerp_(tparams, params, tau)
            if replay is None:
                tgt.sync_weights()
                actor_t.sync_weights()
            return torch.stack([loss_c.detach().float(), loss_a.detach().float()])

        return actor_m, critic, log_ent, step

    def state_of(actor_m, critic, log_ent):
        return [p.detach().clone() for p in list(actor_m.parameters()) + list(critic.parameters())] + [log_ent.detach().clone()]

    am, cm, le, step_e = twin()
    eager = []
    for _ in range(R + 3):
        loss = step_e()
        eager.append((loss.clone(), state_of(am, cm, le)))
    am, cm, le, step_g = twin()
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
        for p, q in zip(state_of(am, cm, le), eager[3 + r][1]):
            assert torch.equal(bits(p), bits(q)), r

    log = []
    k_state = twin(log=log)
    for _ in range(20):
        k_state[3]()
    t32 = twin(kernel=False)
    t64 = twin(kernel=False, dtype=torch.float64)
    for rec in log:
        t32[3](rec)
        t64[3](rec)
    # Adam moves each parameter by about lr per step whatever the gradient's size, so the bound is a share of the movement
    p0 = state_of(actor0, critic0, torch.zeros(1, device=DEV))
    worst_k = worst_t = 0.0
    for pk, p32, p64, q0 in zip(state_of(*k_state[:3]), state_of(*t32[:3]), state_of(*t64[:3]), p0):
        scale = (p64 - q0.double()).abs().max() + 1e-12
        worst_k = max(worst_k, float((pk.double() - p64).abs().max() / scale))
        worst_t = max(worst_t, float((p32.double() - p64).abs().max() / scale))
    print("20 %s steps: worst |p - p64| / max |p64 - p0|: kernel %.3g torch fp32 %.3g" % (kind, worst_k, worst_t))
    assert worst_k <= 0.05 and worst_t <= 0.05, (worst_k, worst_t)


def test_in_place_change_between_forward_and_backward_raises():
    m = make_actor(9, 6, 51)
    a, lp = Actor(m, 9, 6).action_log_prob(observations(64, 9, 52))
    with torch.no_grad():
        m.latent_pi[2].weight.mul_(1.5)
    with pytest.raises(RuntimeError, match="modified by an inplace operation"):
        (a.sum() + lp.sum()).backward()


def test_no_grad_saves_nothing_and_module_policy_or_mapping():
    m = make_actor(9, 6, 61)
    obs = observations(200, 9, 62)
    by_module = Actor(m, 9, 6, seed=1)
    by_map = Actor({"actor." + k: v for k, v in m.named_parameters()}, 9, 6, seed=1)
    with torch.no_grad():
        a, lp = by_module.action_log_prob(obs)
    assert a.grad_fn is None and lp.grad_fn is None
    a2, lp2 = by_map.action_log_prob(obs)
    assert a2.grad_fn is not None
    assert torch.equal(bits(a), bits(a2.detach())) and torch.equal(bits(lp), bits(lp2.detach()))
    for p in m.parameters():
        p.requires_grad_(False)
    a3, _ = by_module.action_log_prob(obs)
    assert a3.grad_fn is None


def test_refusals():
    m = make_actor(9, 6, 71)
    actor = Actor(m, 9, 6)
    obs = observations(16, 9, 72)
    for bad, what in ((obs.clone().requires_grad_(True), "obs requires grad"), (obs.double(), "float32"), (obs.cpu(), "is on"),
                      (obs[:, :5], r"\[B, 9\]"), (obs[:0], r"\[B, 9\]"), (obs[0], r"\[B, 9\]")):
        with pytest.raises(ValueError, match=what):
            actor.action_log_prob(bad)
    for eps in (torch.empty((16, 5), device=DEV), torch.empty((16, 6), device=DEV, dtype=torch.float64), torch.empty((16, 6)),
                torch.empty((6, 16), device=DEV).T):
        with pytest.raises(ValueError, match="eps"):
            actor.action_log_prob(obs, eps=eps)
    with pytest.raises(ValueError, match="share=True needs float32"):
        Actor(copy.deepcopy(m).double(), 9, 6)
    sd = {k: v.detach().clone() for k, v in m.named_parameters()}
    sd["mu.weight"] = sd["mu.weight"].T.contiguous().T
    with pytest.raises(ValueError, match="non-contiguous"):
        Actor(sd, 9, 6)
    # C: bf16 and fixed-head handles, bad sizes, null and host pointers, both output gradients null
    lib = _lib.load()
    b = 16
    P = _lib.ptr
    st = _lib.current_stream(torch.device(DEV))
    h = actor._policy._h
    acts, lp, calls = torch.empty((b, 6), device=DEV), torch.empty(b, device=DEV), torch.zeros(2, dtype=torch.int64, device=DEV)
    saved = torch.empty(int(lib.mvrl_actor_saved_bytes(h, b)), dtype=torch.uint8, device=DEV)
    scratch = torch.empty(int(lib.mvrl_actor_grad_scratch(h, b)), dtype=torch.uint8, device=DEV)
    grads = [torch.empty_like(p) for p in m.parameters()]
    arr = (C.c_void_p * 10)(*[t.data_ptr() for t in grads])
    ga, gl = torch.zeros((b, 6), device=DEV), torch.zeros(b, device=DEV)
    assert lib.mvrl_actor_forward(h, b, P(obs), P(acts), P(lp), None, P(saved), 0, P(calls), st) == 0
    assert lib.mvrl_actor_backward(h, b, P(obs), P(saved), P(ga), None, arr, P(scratch), st) == 0
    torch.cuda.synchronize()
    bf16 = SquashedGaussianPolicy(9, 6, device=DEV)
    assert lib.mvrl_actor_saved_bytes(bf16._h, b) == 0 and lib.mvrl_actor_grad_scratch(bf16._h, b) == 0
    assert lib.mvrl_actor_forward(bf16._h, b, P(obs), P(acts), P(lp), None, None, 0, P(calls), st) == -1
    assert "squashed head and the fp32 precision" in lib.mvrl_last_error().decode()
    fixed = _lib.Handle("mvrl_policy", 0, 9, 6, _lib.POLICY_HEAD_FIXED_STD, _lib.POLICY_PRECISION_FP32, create="create_ex")
    assert lib.mvrl_actor_backward(fixed._h, b, P(obs), P(saved), P(ga), None, arr, P(scratch), st) == -1
    assert "squashed head and the fp32 precision" in lib.mvrl_last_error().decode()
    fresh = _lib.Handle("mvrl_policy", 0, 9, 6, _lib.POLICY_HEAD_SQUASHED, _lib.POLICY_PRECISION_FP32, create="create_ex")
    assert lib.mvrl_actor_forward(fresh._h, b, P(obs), P(acts), P(lp), None, None, 0, P(calls), st) == -1
    assert "no weights" in lib.mvrl_last_error().decode()
    for B in (0, -1, 2 ** 31):
        assert lib.mvrl_actor_forward(h, B, P(obs), P(acts), P(lp), None, None, 0, P(calls), st) == -1
        assert "B must be" in lib.mvrl_last_error().decode()
    for i, name in enumerate(("obs", "actions", "log_prob", "calls")):
        args = [P(obs), P(acts), P(lp), P(calls)]
        args[i] = None
        assert lib.mvrl_actor_forward(h, b, args[0], args[1], args[2], None, None, 0, args[3], st) == -1
        assert "null argument %s" % name in lib.mvrl_last_error().decode()
    assert lib.mvrl_actor_forward(h, b, P(obs.cpu()), P(acts), P(lp), None, None, 0, P(calls), st) == -1
    assert "obs is not device memory" in lib.mvrl_last_error().decode()
    assert lib.mvrl_actor_forward(h, b, P(obs), P(acts), P(lp), P(torch.empty((b, 6))), None, 0, P(calls), st) == -1
    assert "eps is not device memory" in lib.mvrl_last_error().decode()
    assert lib.mvrl_actor_backward(h, b, P(obs), P(saved), None, None, arr, P(scratch), st) == -1
    assert "both null" in lib.mvrl_last_error().decode()
    assert lib.mvrl_actor_backward(h, b, P(obs), None, P(ga), None, arr, P(scratch), st) == -1
    assert "null argument saved" in lib.mvrl_last_error().decode()
    assert lib.mvrl_actor_backward(h, b, P(obs), P(saved), P(ga), None, None, P(scratch), st) == -1
    assert "null argument grads" in lib.mvrl_last_error().decode()
    assert lib.mvrl_actor_backward(h, b, P(obs), P(saved), P(ga.cpu()), None, arr, P(scratch), st) == -1
    assert "grad_actions is not device memory" in lib.mvrl_last_error().decode()
    host = torch.zeros(16)
    bad = (C.c_void_p * 10)(*([t.data_ptr() for t in grads[:9]] + [host.data_ptr()]))
    assert lib.mvrl_actor_backward(h, b, P(obs), P(saved), None, P(gl), bad, P(scratch), st) == -1
    assert "log_std.bias is not device memory" in lib.mvrl_last_error().decode()
    nul = (C.c_void_p * 10)(*([t.data_ptr() for t in grads[:3]] + [None] + [t.data_ptr() for t in grads[4:]]))
    assert lib.mvrl_actor_backward(h, b, P(obs), P(saved), None, P(gl), nul, P(scratch), st) == -1
    assert "null gradient latent_pi.2.bias" in lib.mvrl_last_error().decode()
