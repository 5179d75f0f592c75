"""GPU: the fused actor's Gaussian draws against the NumPy Philox reference (oracle_np.philox_normal_pair): ``eps``
(stream 7) and the squashed head's action noise ``xi`` (stream 8) of every kernel variant, entry by entry, with the log-prob
and the action built from them, at 64-bit keys (a seed above 2^63 with both words non-zero, env ids straddling 2^32, steps
up to 2^32 - 1) and at keys that hit the tails of Box-Muller.  Also the environments' reset draws at 64-bit keys against
their oracles.

Error bound of one draw, from the documented error of each step of ``normal_pair`` (csrc/mvrl_policy.cu):
  * ln u1 by __logf: dL = 2^-21.41 absolute for u1 in [0.5, 2], 3 ulp of the result below 0.5;
  * r = sqrtf(-2 ln u1): dr <= min(2 dL / r, sqrt(2 dL)) (r'^2 - r^2 = 2 (L' - L), r' >= 0) plus the rounding of sqrtf;
  * the angle: 2pi_f u2 rounded (2pi_f - 2pi = 1.7e-7, half an ulp of x <= 2.4e-7), the multiply by 1 / (2 pi) in float32
    rounded toward zero before MUFU.SIN / COS (<= 2^-24 revolution, 3.7e-7, and 2.5e-7 from the constant): at most 2.2
    ulp of 2pi_f, allowed 3 (1.43e-6), plus 2^-21.41 for __sincosf itself, times r;
  * the final product r cos(theta) rounded to float32.
"""
import math

import numpy as np
import pytest
import torch

from oracle import oracle_np as o
from test_random_streams_cpu import SEED, TAIL_SEED, TAIL_STEP, TAIL_TARGETS

pytestmark = pytest.mark.gpu

if torch.cuda.is_available():
    from marinevehiclereinforcementlearning_b200 import (AuvCylVecEnv, AuvVecEnv, BlueROV2Heavy3DoFVecEnv, BlueROV2Heavy6DoFVecEnv,
                                                         MlpGaussianPolicy, SquashedGaussianPolicy)
    from test_auv_gpu import make_flows
    from test_policy_squashed_gpu import head_reference
    from conftest import load_golden

DEV = "cuda"
N = 2 ** 20
ENV0 = 2 ** 32 - 2 ** 19          # the window straddles the 2^32 word boundary of the env id
LD = N + 32                       # columns >= N are padding
STEPS = (0, 1, 2 ** 32 - 1)
OBS_DIM = 9
FILL = 7.0
KERNELS = ("tcgen05", "mma_sync", "fp32")
DL_NEAR_ONE = 2.0 ** -21.41       # __logf on [0.5, 2]; also __sincosf on [-pi, pi]
DTHETA = 3 * float(np.spacing(np.float32(2 * np.pi)))
NOISE_STD = 0.125                 # a power of two: 0.125 xi is exact
BANDS = ("r < 0.05", "bulk", "r > 4", "theta > pi")
STATS = {b: [0, 0.0, 0.0] for b in BANDS}   # draws, worst |d|, worst |d| / bound (all kernels, both streams)


def draw_bound(k1, k2, z):
    """Bound on |kernel - reference| of a component z of the pairs with words k1, k2 (module docstring)."""
    u1 = o.normal_pair_u1(k1)
    L = np.abs(np.log(u1.astype(np.float64)))             # -ln u1 without the -0 of u1 = 1
    dL = np.where(u1 >= 0.5, DL_NEAR_ONE, 3.0 * np.spacing(L.astype(np.float32)).astype(np.float64))
    r = np.sqrt(2.0 * L)
    with np.errstate(divide="ignore"):
        dr = np.minimum(2.0 * dL / r, np.sqrt(2.0 * dL)) + 2.0 ** -24 * r
    return dr + (r + dr) * (DTHETA + DL_NEAR_ONE) + 0.5 * np.spacing(np.abs(z).astype(np.float32)).astype(np.float64)


def band_of(k1, k2):
    r = np.sqrt(-2.0 * np.log(o.normal_pair_u1(k1).astype(np.float64)))
    return np.where(r < 0.05, 0, np.where(r > 4.0, 2, np.where(k2 > 2 ** 23, 3, 1))).astype(np.int8)


_REF = {}


def reference(stream, step):
    """[8, N] reference draws of the window (row 2 blk + c = component c of pair blk), their bounds and bands, on the GPU."""
    if (stream, step) not in _REF:
        env = np.arange(ENV0, ENV0 + N, dtype=np.uint64)
        z, bound, band = np.empty((8, N)), np.empty((8, N)), np.empty((8, N), dtype=np.int8)
        for blk in range(4):
            k1, k2, z0, z1 = o.philox_normal_pair(SEED, env, step, blk, stream)
            for c, zc in enumerate((z0, z1)):
                z[2 * blk + c], bound[2 * blk + c], band[2 * blk + c] = zc, draw_bound(k1, k2, zc), band_of(k1, k2)
        _REF[(stream, step)] = {k: torch.as_tensor(v, device=DEV) for k, v in (("z", z), ("bound", bound), ("band", band))}
    return _REF[(stream, step)]


def check_draws(got, ref, rows, what):
    """got [rows, N] float32 (kernel) vs the reference: every entry within its bound; the per-band statistics."""
    d = (got.double() - ref["z"][:rows]).abs()
    ratio = d / ref["bound"][:rows]
    assert bool(torch.isfinite(got).all()), what
    worst = int(ratio.flatten().argmax())
    assert float(ratio.max()) <= 1.0, (what, "row %d col %d" % divmod(worst, N), float(d.flatten()[worst]), float(ratio.max()))
    for i, b in enumerate(BANDS):
        m = ref["band"][:rows] == i
        if bool(m.any()):
            s = STATS[b]
            s[0] = max(s[0], int(m.sum()))
            s[1], s[2] = max(s[1], float(d[m].max())), max(s[2], float(ratio[m].max()))


def make_policy(kernel, head, act_dim, monkeypatch, noise=None, seed=SEED):
    monkeypatch.setenv("MVRL_POLICY_MMA_SYNC", "1" if kernel == "mma_sync" else "0")
    precision = "fp32" if kernel == "fp32" else "bf16"
    if head == "fixed":
        pol = MlpGaussianPolicy(OBS_DIM, act_dim, device=DEV, seed=seed, precision=precision)
        pol.log_std = torch.linspace(-1.3, 0.4, act_dim)
        pol.sync_weights()
    else:
        pol = SquashedGaussianPolicy(OBS_DIM, act_dim, device=DEV, seed=seed, action_noise_std=noise, precision=precision)
    return pol


def zero_head(pol):
    """mu = 0 and log_std = -20 exactly: a = tanh(exp(-20) eps) ~ 2e-9 eps, so act - a exposes the action noise."""
    for k in ("mu.weight", "mu.bias", "log_std.weight"):
        pol.params[k].zero_()
    pol.params["log_std.bias"].fill_(-20.0)
    pol.sync_weights()


def run(pol, obs, n, env_id0, step, head):
    ld = obs.shape[1]
    b = {k: torch.full((8, ld), FILL, device=DEV) for k in ("act", "mean", "eps", "log_std")}
    b["logp"] = torch.full((ld,), FILL, device=DEV)
    pol.act_into(obs, b["act"], n, logp=b["logp"], mean=b["mean"], eps=b["eps"], log_std=b["log_std"] if head == "squashed" else None,
                 env_id0=env_id0, step=step)
    torch.cuda.synchronize()
    return b


def random_obs(ld, seed=0):
    g = torch.Generator(device=DEV).manual_seed(seed)
    return torch.rand((OBS_DIM, ld), generator=g, device=DEV) * 2 - 1


def check_head(b, ref, pol, head, a, n, what):
    """act and logp of the kernel against the formulas evaluated in fp64 with the reference eps."""
    z, bound = ref["z"][:a, :n], ref["bound"][:a, :n]
    act, mean, logp = b["act"][:a, :n].double(), b["mean"][:a, :n].double(), b["logp"][:n].double()
    assert bool(torch.isfinite(b["logp"][:n]).all()) and bool(torch.isfinite(b["act"][:a, :n]).all()), what
    ebound = (z.abs() * bound + 0.5 * bound * bound).sum(0)      # |sum z^2 / 2 - sum eps^2 / 2|
    if head == "fixed":
        ls = pol.log_std.double().to(DEV)[:, None]
        std = ls.exp()
        a_ref = (mean + std * z).clamp(-1.0, 1.0)
        tol_a = std * (bound + 2.0 ** -22 * z.abs()) + 2.0 ** -23
        lp_ref = -0.5 * (z * z).sum(0) - ls.sum()
        # fp32: a squares and a + 1 additions, each rounded within 2^-24 of the sum of the magnitudes
        tol_lp = ebound + (2 * a + 2) * 2.0 ** -24 * (0.5 * (z * z).sum(0) + ls.abs().sum())
    else:
        ls = b["log_std"][:a, :n].double()
        a_ref, lp_ref = head_reference(mean.T, ls.T, z.T, act.T)
        a_ref = a_ref.T
        tol_a = ls.exp() * bound + 2e-6                           # test_policy_squashed_gpu: 2e-6 with the kernel's eps
        tol_lp = ebound + 1e-5 * a
    assert bool(((act - a_ref).abs() <= tol_a).all()), (what, float(((act - a_ref).abs() / tol_a).max()))
    assert bool(((logp - lp_ref).abs() <= tol_lp).all()), (what, float(((logp - lp_ref).abs() / tol_lp).max()))


def check_padding(b, a, n, head, what):
    for k in ("act", "mean", "eps") + (("log_std",) if head == "squashed" else ()):
        assert bool((b[k][a:] == FILL).all()) and bool((b[k][:, n:] == FILL).all()), (what, k)
    assert bool((b["logp"][n:] == FILL).all()), what


@pytest.mark.parametrize("kernel", KERNELS)
def test_eps_matches_reference_at_64bit_keys(kernel, monkeypatch):
    """Every eps entry of 2^20 environments around env id 2^32, at steps 0, 1 and 2^32 - 1, for both heads: within the
    bound of each draw; act and logp from the reference eps; padding rows and columns untouched."""
    obs = random_obs(LD)
    for head in ("fixed", "squashed"):
        for a in ((1, 2, 3, 6, 7, 8) if kernel == "tcgen05" else (1, 7, 8)):
            pol = make_policy(kernel, head, a, monkeypatch)
            for step in STEPS:
                what = (kernel, head, a, step)
                b = run(pol, obs, N, ENV0, step, head)
                ref = reference(7, step)
                check_draws(b["eps"][:a, :N], ref, a, what)
                check_head(b, ref, pol, head, a, N, what)
                check_padding(b, a, N, head, what)
    print_stats("eps, %s" % kernel)


def print_stats(title):
    print("\n%s (cumulative over the tests so far), per band: draws per run, worst |d|, worst |d| / bound" % title)
    for k, (cnt, d, q) in STATS.items():
        print("  %-10s %9d  %.3g  %.3f" % (k, cnt, d, q))


@pytest.mark.parametrize("kernel", KERNELS)
def test_action_noise_matches_stream_8(kernel, monkeypatch):
    """The squashed head's action noise xi = (act - a) / 0.125 through a head with mu = 0 and log_std = -20 (it never
    clips: |0.125 xi| <= 0.74) against stream 8 of the reference; eps does not move."""
    obs = random_obs(LD, seed=1)
    for a in (7, 8):
        pol = make_policy(kernel, "squashed", a, monkeypatch, noise=NOISE_STD)
        zero_head(pol)
        for step in (0, 2 ** 32 - 1):
            what = (kernel, a, step)
            b = run(pol, obs, N, ENV0, step, "squashed")
            eps, act = b["eps"][:a, :N], b["act"][:a, :N]
            assert bool((act.abs() <= 0.74).all()), what
            a_pre = torch.tanh(math.exp(-20.0) * eps.double())
            xi = (act.double() - a_pre) / NOISE_STD
            check_draws(eps, reference(7, step), a, what + ("eps",))
            ref = dict(reference(8, step))
            # act = fma(0.125, xi, a) rounds once: half an ulp of act, over 0.125
            ref["bound"] = ref["bound"][:a] + 0.5 * torch.as_tensor(np.spacing(act.abs().cpu().numpy()), device=DEV).double() / NOISE_STD + 1e-12
            check_draws(xi, ref, a, what + ("xi",))
            check_padding(b, a, N, "squashed", what)
    print_stats("eps and xi, %s" % kernel)


@pytest.mark.parametrize("kernel", KERNELS)
def test_tail_draws(kernel, monkeypatch):
    """The committed tail targets (u1 = 1 and the u1 values just below 1, the largest radii, the quadrant edges) through
    each head with act_dim 8, one environment at a time: u1 = 1 gives eps = +-0 exactly; eps, xi, act and logp are finite;
    every draw is within its bound."""
    pols = {"fixed": make_policy(kernel, "fixed", 8, monkeypatch, seed=TAIL_SEED),
            "squashed": make_policy(kernel, "squashed", 8, monkeypatch, seed=TAIL_SEED),
            "noise": make_policy(kernel, "squashed", 8, monkeypatch, noise=NOISE_STD, seed=TAIL_SEED)}
    zero_head(pols["noise"])
    obs = random_obs(32, seed=2)
    worst = 0.0
    for word, k, env, stream, blk in TAIL_TARGETS:
        k1, k2, z0, z1 = o.philox_normal_pair(TAIL_SEED, [env], TAIL_STEP, blk, stream)
        want = np.array([z0[0], z1[0]])
        bound = np.array([draw_bound(k1, k2, z0)[0], draw_bound(k1, k2, z1)[0]])
        for name, pol in pols.items():
            head = "fixed" if name == "fixed" else "squashed"
            what = (kernel, name, word, hex(k), stream, blk)
            b = run(pol, obs, 1, env, TAIL_STEP, head)
            for key in ("act", "eps", "mean"):
                assert bool(torch.isfinite(b[key][:, 0]).all()), what + (key,)
            assert math.isfinite(float(b["logp"][0])), what
            eps = b["eps"][2 * blk:2 * blk + 2, 0].double().cpu().numpy()
            if name == "noise":
                act = b["act"][2 * blk:2 * blk + 2, 0].cpu().numpy()
                got = (act.astype(np.float64) - np.tanh(math.exp(-20.0) * eps)) / NOISE_STD
                tol = bound + 0.5 * np.spacing(np.abs(act)).astype(np.float64) / NOISE_STD + 1e-12
            else:
                got, tol = eps, bound
            if stream == 8 and name != "noise" or stream == 7 and name == "noise":
                continue
            if stream == 7 and word == "k1" and k == 0xFFFFFF:
                assert got[0] == 0.0 and got[1] == 0.0, what
            assert np.all(np.abs(got - want) <= tol), (what, got, want, tol)
            worst = max(worst, float((np.abs(got - want) / tol).max()))
    print("\n%s: tail targets, worst |d| / bound %.3f" % (kernel, worst))


def test_padding_keeps_fill_values(monkeypatch):
    """eps, mean, act (and log_std) with 8 rows while act_dim is odd, n off the 128-row tile: rows >= act_dim and columns
    >= n keep their fill value in every kernel and head."""
    obs = random_obs(1024, seed=3)
    for kernel in KERNELS:
        for head in ("fixed", "squashed"):
            for a in (1, 3, 7):
                pol = make_policy(kernel, head, a, monkeypatch)
                for n in (1, 129, 1000):
                    check_padding(run(pol, obs, n, ENV0 - 500, 9, head), a, n, head, (kernel, head, a, n))


RESET_N = 256
RESET_ENV0 = 2 ** 32 - RESET_N // 2


def _reset_pair(kind):
    kw = dict(maxSteps=3, auto_reset=True, seed=SEED, env_id0=RESET_ENV0)
    okw = dict(max_steps=3, auto_reset=True, seed=SEED, env_id0=RESET_ENV0)
    if kind == "rov6":
        return (BlueROV2Heavy6DoFVecEnv(RESET_N, action_mode="rpm", dtype=torch.float64, device=DEV, **kw),
                o.Rov6EnvOracle(RESET_N, mode=o.MODE_RPM, **okw), 8, 3500.0)
    if kind == "rov3":
        return (BlueROV2Heavy3DoFVecEnv(RESET_N, action_mode="rpm", dtype=torch.float64, device=DEV, **kw),
                o.Rov3EnvOracle(RESET_N, mode=o.MODE_RPM, **okw), 4, 3500.0)
    flow, rflow = make_flows(load_golden("legacy"), smooth=True)
    noise = dict(noiseMagCoeffs=0.1, noiseMagActuation=0.1)
    if kind == "auv":
        return AuvVecEnv(RESET_N, flow, dtype=torch.float64, **noise, **kw), o.AuvEnvOracle(RESET_N, rflow, **noise, **okw), 3, 1.0
    return AuvCylVecEnv(RESET_N, flow, dtype=torch.float64, **noise, **kw), o.AuvCylEnvOracle(RESET_N, rflow, **noise, **okw), 3, 0.5


@pytest.mark.parametrize("kind", ["rov6", "rov3", "auv", "auv_cyl"])
def test_reset_draws_at_64bit_keys(kind):
    """reset() and two auto-resets (maxSteps 3) with a seed above 2^63 and env ids straddling 2^32 against the oracle at
    the tolerances of the envs' own auto-reset tests; the drawn quantities (way-points and set-points, or the AUV's
    multipliers, heading target and flow time offset) directly."""
    env, ref, act_dim, scale = _reset_pair(kind)
    rng = np.random.default_rng(41)
    n = RESET_N

    def drawn_agree():
        if kind in ("rov6", "rov3"):
            assert np.abs(env.path.cpu().numpy().reshape(n, -1) - ref.path).max() < 1e-12
            assert np.abs(env.setPoint.cpu().numpy() - ref.set_point).max() < 1e-12
        else:
            assert np.abs(env._mults[:, :n].T.cpu().numpy() - ref.mults).max() < 1e-15
            assert np.abs(env.headingTarget.cpu().numpy() - ref.heading_target).max() < 1e-12
            assert np.abs(env.flowDataTimeOffset.cpu().numpy() - ref.t_offset).max() < 1e-12

    assert np.abs(env.reset().cpu().numpy() - ref.reset()).max() < 1e-12
    drawn_agree()
    resets = 0
    for k in range(7):
        act = rng.uniform(-scale, scale, (n, act_dim))
        obs, rew, done, info = env.step(torch.as_tensor(act, device=DEV))
        ro, rr, rd, _ = ref.step(act)
        assert np.array_equal(done.cpu().numpy(), rd), k
        assert np.abs(obs.cpu().numpy() - ro).max() < 1e-9, k
        resets += int(rd.sum())
        drawn_agree()
    assert resets >= 2 * n
