"""The rare branches of the fused step kernels, against fp64 references.

The parity tests in test_parity_modes_gpu.py start from reset() states and drive them with random actions: strong on the
common path, silent on the code only unusual environments take.  This file constructs those environments:

1. `sincos_f32` (rov6_model.cuh), the fp32 sin / cos of every 6DoF and 3DoF evaluation, against fp64 sin / cos: exhaustively on
   [0, 2 pi), around every reduction boundary k pi / 4 up to 2^16, at random in (-2 pi, 0) and [2 pi, 2^16], at the specials.
2. RK4 stages 2-4 take sin / cos from the addition theorem while the squared stage offsets sum to at most
   MVRL_TRIG_DELTA_MAX2, and the full evaluation above it: environments on both sides and at the threshold, classified by an
   fp64 replay of the stages, step once against the C oracle.  At n_sub = 8 the truncation of the addition theorem stays
   below the fp32 rounding up to offsets of ~1 rad; with n_sub = 4 the offsets are large enough for the threshold to show.
3. That decision is taken per environment: an environment's results do not depend on the one sharing its thread (F2, two
   fp32 environments per thread), nor on what sits in the padding column of an odd batch.
4. Epilogue phase B (the exact wrap of angles outside (-2 pi, 4 pi) or 2 pi away from their set-point), the set-point PID's
   exact angle error, and the fp32 out-of-range flag (|angle| > 2^16) in the non-finite counter.
5. The PID's yaw-wrap fall-back: the wrapped yaw error jumps by 2 pi inside a step (6DoF and 3DoF).
6. The 3DoF fp32 step flags a yaw outside the range of `sincos_f32` like the 6DoF step.

One-step comparisons use the exclusions of test_parity_modes_gpu.py (1 / cos(theta) pole, PID sign margin, thruster
dead-band edge); its docstring explains them.
"""
import time

import numpy as np
import pytest
import torch

from oracle import c_oracle as c
from oracle import oracle_np as o
from test_parity_modes_gpu import MODES, SCALE6, TOL, scaled_err, sync3, sync6

pytestmark = pytest.mark.gpu

if torch.cuda.is_available():
    from marinevehiclereinforcementlearning_b200 import BlueROV2Heavy3DoFVecEnv, BlueROV2Heavy6DoFVecEnv, resources

DEV = "cuda"
TWO_PI = 2.0 * np.pi
F32_MAX_ARG = 65536.0           # MVRL_SINCOS_F32_MAX_ARG
DELTA_MAX2 = 0.0625             # MVRL_TRIG_DELTA_MAX2
NO_STEP_LIMIT = 10 ** 9


def as_dtype(x, dtype):
    """x rounded to the env's precision, held in fp64: what both sides of a comparison start from."""
    return np.asarray(x, dtype=np.float32 if dtype == torch.float32 else np.float64).astype(np.float64)


def ulp(x, dtype):
    """Spacing of the floating-point numbers of the env's precision at |x|."""
    return np.spacing(np.abs(as_dtype(x, dtype)).astype(np.float32 if dtype == torch.float32 else np.float64)).astype(np.float64)


def component_errors(got, ref, ang):
    """scaled_err of every column on its own: [n, dim]."""
    return np.stack([scaled_err(got[:, j:j + 1], ref[:, j:j + 1], slice(0, 1) if j in ang else slice(0, 0))
                     for j in range(ref.shape[1])], axis=1)


def random_states6(rng, n, rate):
    """theta in [-1.2, 1.2], roll and yaw in [0, 2 pi), body rates U(-rate, rate)."""
    s = np.zeros((n, 12))
    s[:, 0:3] = rng.uniform(-2, 2, (n, 3))
    s[:, 3] = rng.uniform(0, TWO_PI, n)
    s[:, 4] = rng.uniform(-1.2, 1.2, n)
    s[:, 5] = rng.uniform(0, TWO_PI, n)
    s[:, 6:9] = rng.uniform(-1, 1, (n, 3))
    s[:, 9:12] = rng.uniform(-rate, rate, (n, 3))
    return s


def random_actions6(rng, mode, n):
    return rng.uniform(-1, 1, (n, len(SCALE6[mode]))) * SCALE6[mode]


def step6(mode, dtype, state, action, set_point=None, n_sub=8):
    """One env step of a fresh CUDA env and of the C oracle from the same state, actions and (set_point given: fixed)
    set-points, with a fresh controller.  -> dict of host arrays."""
    n = len(state)
    fixed = set_point is not None
    ref = c.Rov6EnvC(n, mode=MODES[mode], max_steps=NO_STEP_LIMIT, n_sub=n_sub)
    ref.reset(initial_setpoint=np.zeros(6) if fixed else None)
    ref.state[:] = state
    if fixed:
        ref.set_point[:] = set_point
    env = BlueROV2Heavy6DoFVecEnv(n, action_mode=mode, dtype=dtype, device=DEV, auto_reset=False, maxSteps=NO_STEP_LIMIT, n_sub=n_sub)
    env.reset(initialSetpoint=np.zeros(6) if fixed else None)
    sync6(env, ref, mode)
    ref.mincos[:] = 1.0
    ref.dbmargin[:] = np.inf
    ref.ctrl_np["margin"] = np.inf
    sp0 = ref.set_point.copy()
    env.episode_stats()
    obs = env.step(torch.as_tensor(action, dtype=dtype, device=DEV))[0].cpu().numpy().astype(np.float64)
    ro = ref.step(action)[0].copy()
    return dict(state=env.systemState.cpu().numpy().astype(np.float64), ref=ref.state.copy(), obs=obs, ref_obs=ro,
                sp=ref.set_point.copy(), sp0=sp0, nonfinite=env.episode_stats()["nonfinite"],
                mincos=ref.mincos.copy(), margin=ref.ctrl_np["margin"].copy(), dbmargin=ref.dbmargin.copy())


def step3(mode, dtype, state, action, set_point=None):
    """step6 for the 3DoF env against oracle_np.Rov3EnvOracle."""
    n = len(state)
    fixed = set_point is not None
    ref = o.Rov3EnvOracle(n, mode=MODES[mode], max_steps=NO_STEP_LIMIT)
    ref.reset(initial_setpoint=np.zeros(3) if fixed else None)
    ref.state[:] = state
    if fixed:
        ref.set_point[:] = set_point
    env = BlueROV2Heavy3DoFVecEnv(n, action_mode=mode, dtype=dtype, device=DEV, auto_reset=False, maxSteps=NO_STEP_LIMIT)
    env.reset(initialSetpoint=np.zeros(3) if fixed else None)
    sync3(env, ref, mode)
    ref.ctrl["margin"] = np.full(n, np.inf)
    o.DIAG["dbmargin"] = np.full(n, np.inf)
    try:
        env.episode_stats()
        env.step(torch.as_tensor(action, dtype=dtype, device=DEV))
        ref.step(action)
        dbmargin = o.DIAG["dbmargin"].copy()
    finally:
        o.DIAG["dbmargin"] = None
    return dict(state=env.systemState.cpu().numpy().astype(np.float64), ref=ref.state.copy(), sp=ref.set_point.copy(),
                nonfinite=env.episode_stats()["nonfinite"], margin=ref.ctrl["margin"].copy(), dbmargin=dbmargin)


def well_conditioned(r, mode, pole=1e-2, dead_band=1e-4):
    """Away from the three discontinuities of the reference's model (test_parity_modes_gpu.py): |cos theta| >= pole,
    PID margin >= 1e-7, relative distance of the thruster rpm from the dead-band edge >= dead_band (scalar or per env)."""
    well = np.ones(len(r["ref"]), dtype=bool)
    if "mincos" in r:
        well &= r["mincos"] >= pole
    if mode == "setpoint":
        well &= r["margin"] >= 1e-7
    if mode != "rpm":
        well &= r["dbmargin"] >= dead_band
    return well


# ----------------------------------------------------------------- 1. sincos_f32 against fp64 -----------------------------
# coordinateTransform(dof=6) runs trig6<float> of the step kernels (same translation unit, same -fmad=false) and builds J
# from kinematics6.  With the other two angles 0 (sin 0 = 0, cos 0 = 1 exactly) these entries ARE sin_f32 / cos_f32 of the
# third angle: (row, column, sign) of sin, (row, column) of cos, for phi, theta, psi.
TRIG_ENTRIES = (((2, 1, 1.0), (1, 1)), ((2, 0, -1.0), (0, 0)), ((1, 0, 1.0), (0, 0)))


def sincos_errors(x, acc):
    """Largest absolute error and largest error in fp32 ulps of the true value (where |value| >= 1/16 and
    -2 pi < x < 4 pi) of sin / cos over the three channels, for the fp32 CUDA tensor x; folded into acc."""
    z = torch.zeros_like(x)
    xd = x.double()
    in_ulp_range = (xd > -TWO_PI) & (xd < 2 * TWO_PI)
    refs = (torch.sin(xd), torch.cos(xd))
    for ch, ((sr, sc, sg), (cr, cc)) in enumerate(TRIG_ENTRIES):
        args = [z, z, z]
        args[ch] = x
        J = resources.coordinateTransform(*args, dof=6)
        for got, ref in ((J[:, sr, sc] * sg, refs[0]), (J[:, cr, cc], refs[1])):
            err = (got.double() - ref).abs()
            acc["abs"] = max(acc["abs"], err.max().item())
            _, e = torch.frexp(ref)
            sel = in_ulp_range & (ref.abs() >= 1.0 / 16)
            if bool(sel.any()):
                acc["ulp"] = max(acc["ulp"], (err[sel] / torch.ldexp(torch.ones_like(err[sel]), e[sel] - 24)).max().item())
        del J
    acc["n"] += x.numel()


def test_sincos_f32_against_fp64():
    """Maximum absolute error <= 1.2e-7 for |x| <= 2^16, at most 2 ulps of the true value wherever |value| >= 1/16 on
    (-2 pi, 4 pi).  Relative error near the zeros of large arguments is not bounded and not asserted.  sincos_f32 returns
    +0 for sin(-0) (the polynomial adds +0 to r = -0), and every J entry sums in an exact +0: only the value of a zero is
    checked."""
    t0 = time.time()
    f32 = lambda v: torch.as_tensor(np.asarray(v, dtype=np.float32), device=DEV)
    sets = {}

    # every fp32 in [0, 2 pi): bit patterns 0 .. bits(largest float < 2 pi)
    acc = sets["all fp32 in [0, 2pi)"] = dict(abs=0.0, ulp=0.0, n=0)
    end = int(np.array(TWO_PI, dtype=np.float32).view(np.int32))      # fp32(2 pi) > 2 pi: excluded
    assert float(np.float32(TWO_PI)) > TWO_PI
    chunk = 1 << 26
    for lo in range(0, end, chunk):
        sincos_errors(torch.arange(lo, min(end, lo + chunk), dtype=torch.int32, device=DEV).view(torch.float32), acc)
    assert acc["n"] == end

    # 2^24 random points in each of (-2 pi, 0), [2 pi, 4 pi) and [2 pi, 2^16]
    gen = torch.Generator(device=DEV).manual_seed(11)
    for lo, hi in ((-TWO_PI, 0.0), (TWO_PI, 2 * TWO_PI), (TWO_PI, F32_MAX_ARG)):
        x = (lo + (hi - lo) * torch.rand(1 << 24, generator=gen, dtype=torch.float64, device=DEV)).float()
        x = x[(x.double() > lo) & (x.double() < hi)] if lo < 0 else x[(x.double() >= lo) & (x.double() <= hi)]
        sincos_errors(x, sets.setdefault("random in [%.4g, %.4g]" % (lo, hi), dict(abs=0.0, ulp=0.0, n=0)))

    # every fp32 within 64 ulps of k pi / 4 (reduction boundaries at odd k, zeros of sin / cos at even k), |x| <= 2^16
    k = np.arange(1, int(F32_MAX_ARG * 4 / np.pi) + 1)
    centre = (k * (np.pi / 4)).astype(np.float32).view(np.int32)
    bits = (centre[:, None] + np.arange(-64, 65, dtype=np.int32)[None, :]).reshape(-1)
    x = torch.as_tensor(bits.view(np.float32), device=DEV)
    x = x[x <= F32_MAX_ARG]
    x = torch.cat([x, -x])
    acc = sets["+-64 ulp around k pi/4"] = dict(abs=0.0, ulp=0.0, n=0)
    for part in torch.split(x, chunk):
        sincos_errors(part.contiguous(), acc)

    # specials
    tiny = [0.0, -0.0, np.finfo(np.float32).tiny, -np.finfo(np.float32).tiny, np.float32(1.4e-45), -np.float32(1.4e-45)]
    sp = f32(tiny + [F32_MAX_ARG, -F32_MAX_ARG])
    sincos_errors(sp, sets.setdefault("specials", dict(abs=0.0, ulp=0.0, n=0)))
    z = torch.zeros_like(sp)
    for ch, ((sr, sc, sg), (cr, cc)) in enumerate(TRIG_ENTRIES):
        args = [z, z, z]
        args[ch] = sp
        J = resources.coordinateTransform(*args, dof=6).cpu().numpy()
        s, co = J[:6, sr, sc] * sg, J[:6, cr, cc]
        assert np.array_equal(s, np.float32(tiny)) and np.array_equal(co, np.ones(6, np.float32)), (ch, s, co)   # sin x = x, cos x = 1
    torch.cuda.synchronize()

    for name, a in sets.items():
        print("sincos_f32 %-28s %11d points: max abs error %.3e, max %.3f ulp (|value| >= 1/16, -2pi < x < 4pi)"
              % (name, a["n"], a["abs"], a["ulp"]))
    print("sincos_f32: %.1f s" % (time.time() - t0))
    for name, a in sets.items():
        assert a["abs"] <= 1.2e-7, (name, a)
        assert a["ulp"] <= 2.0, (name, a)


# ----------------------------------------------------------------- 2. anchored stage trig on both sides of the threshold ---
def stage_offsets(mode, state, action, set_point=None, dt=0.2, n_sub=8):
    """fp64 replay (oracle_np) of one env step: zs = |c_k k_angle|^2 of the angle offset of RK4 stages 2-4 from the
    sub-step's stage-1 angles, which the fp32 step kernel compares with MVRL_TRIG_DELTA_MAX2.  -> [n, 3 n_sub]."""
    p = o.Rov6Params()
    if mode == "rpm":
        f = lambda t, y: o.derivs6_rpm(p, y, action)
    elif mode == "force":
        f = lambda t, y: o.derivs6_force(p, y, action)
    else:
        if set_point is None:   # 6DoF.py:545-552
            L2, qa = 2. * p.Length, np.pi / 4
            set_point = action * np.array([L2, L2, L2, qa, qa, qa]) + state[:, :6]
        ctrl = o.pid6_new_state(len(state))
        f = lambda t, y: o.derivs6_pid(p, t, y, ctrl, set_point)
    h = dt / n_sub
    y, zs = state.copy(), []
    for j in range(n_sub):
        t = j * h
        k1 = f(t, y)
        k2 = f(t + 0.5 * h, y + 0.5 * h * k1)
        k3 = f(t + 0.5 * h, y + 0.5 * h * k2)
        k4 = f(t + h, y + h * k3)
        for cp, k in ((0.5 * h, k1), (0.5 * h, k2), (h, k3)):
            zs.append(((cp * k[:, 3:6]) ** 2).sum(axis=1))
        y = y + (h / 6.0) * (k1 + 2.0 * k2 + 2.0 * k3 + k4)
    return np.stack(zs, axis=1)


def trig_classes(zs):
    """anchored: every stage below 0.95 x the threshold; fall-back: some stage above 1.05 x; edge: some stage within 5 %."""
    lo, hi = 0.95 * DELTA_MAX2, 1.05 * DELTA_MAX2
    return {"anchored": (zs < lo).all(axis=1), "fall-back": (zs > hi).any(axis=1),
            "edge": ((zs >= lo) & (zs <= hi)).any(axis=1)}


def test_trig_threshold_with_four_substeps():
    """The threshold itself, fp32 rpm mode: with n_sub = 4 and body rates U(-6, 6) the stage offsets reach 0.5-1.5 rad
    (the integration stays finite), where the truncation of sincos_delta is no longer below the fp32 rounding.  Away from
    the pole (|cos theta| >= 0.05, where the 1 / cos(theta) of J2 leaves the rounding alone) every class agrees with the C
    oracle within 1.5e-6; measured on B200: at most 7.8e-7, against 2.7e-6 for the addition theorem applied up to a
    squared offset of 1 and 4e-4 for the addition theorem at every offset.  Near the pole: 1e-4."""
    n = 16384
    rng = np.random.default_rng(23)
    state = as_dtype(random_states6(rng, n, 6.0), torch.float32)
    action = as_dtype(random_actions6(rng, "rpm", n), torch.float32)
    zmax = stage_offsets("rpm", state, action, n_sub=4).max(axis=1)
    r = step6("rpm", torch.float32, state, action, n_sub=4)
    assert np.isfinite(r["ref"]).all() and r["nonfinite"] == 0
    err = scaled_err(r["state"], r["ref"], slice(3, 6))
    classes = {"anchored": zmax < 0.95 * DELTA_MAX2, "fall-back, zs <= 1": (zmax > 1.05 * DELTA_MAX2) & (zmax <= 1.0),
               "fall-back, zs > 1": zmax > 1.0}
    near_pole, far = well_conditioned(r, "rpm", pole=2e-2), well_conditioned(r, "rpm", pole=5e-2)
    for name, m in classes.items():
        print("6DoF rpm fp32 n_sub=4 %-18s: %5d envs, %5d with |cos theta| >= 0.05: max error %.3e; %3d nearer the pole: max %.3e" %
              (name, m.sum(), (m & far).sum(), err[m & far].max(), (m & near_pole & ~far).sum(), err[m & near_pole & ~far].max(initial=0.0)))
    for name, m in classes.items():
        assert (m & far).sum() >= 70, (name, (m & far).sum())
        assert err[m & far].max() <= 1.5e-6, (name, err[m & far].max())
        assert err[m & near_pole].max() <= TOL[torch.float32], (name, err[m & near_pole].max())


@pytest.mark.parametrize("mode", ["rpm", "force", "setpoint"])
def test_anchored_trig_both_sides_of_threshold(mode):
    """fp32, dt = 0.2, n_sub = 8: 16384 environments each with body rates U(-5, 5) and U(-12, 12); every class of
    trig_classes has hundreds of environments and all of them agree with the C oracle within 1e-4 after one step.  This
    checks both trig paths; the threshold between them is checked by test_trig_threshold_with_four_substeps, because at
    these offsets a Taylor evaluation up to ~1 rad stays below the fp32 rounding."""
    n, tol = 16384, TOL[torch.float32]
    rng = np.random.default_rng(21)
    state = as_dtype(np.concatenate([random_states6(rng, n, 5.0), random_states6(rng, n, 12.0)]), torch.float32)
    rate = np.repeat([5, 12], n)
    action = as_dtype(random_actions6(rng, mode, 2 * n), torch.float32)
    classes = trig_classes(stage_offsets(mode, state, action))
    r = step6(mode, torch.float32, state, action)
    err = scaled_err(r["state"], r["ref"], slice(3, 6))
    # these states pass theta = +-pi/2 far more often than reset-born ones: the 1 / cos(theta) of J2 amplifies the fp32
    # rounding to 1.2e-4 at |cos theta| = 0.012 (measured on B200), hence a wider pole exclusion than 1e-2
    well = well_conditioned(r, mode, pole=2e-2)
    assert np.isfinite(r["ref"]).all() and r["nonfinite"] == 0
    for name, m in classes.items():
        for R in (5, 12):
            mr = m & (rate == R)
            print("6DoF %s fp32 R=%2d %-9s: %5d envs (%.3f), %5d well-conditioned, max error %.3e" %
                  (mode, R, name, mr.sum(), mr.mean() * 2, (mr & well).sum(), err[mr & well].max() if (mr & well).any() else 0))
    for name, m in classes.items():
        assert (m & well).sum() >= 300, (name, (m & well).sum())
        assert err[m & well].max() <= tol, (name, err[m & well].max())


# ----------------------------------------------------------------- 3. the decision does not depend on the neighbour -------
def env_set_a(rng, mode, m):
    """The environments A of the neighbour test: random states with body rates 5 and 12 (both trig paths and the edge),
    angles outside (-2 pi, 4 pi) with set-points 10-30 rad away (phase B), yaw errors within 0.05 of +-pi with yaw rates
    +-1 (the PID's yaw-wrap fall-back).  -> state [m, 12], action, set-point [m, 6]."""
    q = m // 8
    state = np.concatenate([random_states6(rng, 3 * q, 5.0), random_states6(rng, 3 * q, 12.0), random_states6(rng, 2 * q, 0.3)])
    sp = state[:, :6] + rng.uniform(-1, 1, (m, 6))
    far = slice(6 * q, 7 * q)
    state[np.arange(6 * q, 7 * q), 3 + rng.integers(0, 3, q)] = rng.choice([-7.0, 13.0, 100.0, 3e4, -TWO_PI - 0.3, 2 * TWO_PI + 0.3], q)
    sp[far, 3:6] = state[far, 3:6] + rng.choice([-1, 1], (q, 3)) * rng.uniform(10, 30, (q, 3))
    wrap = slice(7 * q, 8 * q)
    state[wrap, 11] = rng.choice([-1.0, 1.0], q)
    sp[wrap, 5] = state[wrap, 5] + rng.choice([-1, 1], q) * (np.pi - rng.uniform(0, 0.05, q))
    return state, random_actions6(rng, mode, m), sp


def columns6(state, action, sp, ctrl=None):
    """Feature-major fp32 inputs of a 6DoF batch (fresh controller unless ctrl is given)."""
    n = len(state)
    if ctrl is None:
        ctrl = np.zeros((13, n))
        ctrl[0] = np.nan                 # eOld is None
    path = np.concatenate([sp[:, :3], sp[:, :3]], axis=1)
    return {k: np.ascontiguousarray(v, dtype=np.float32) for k, v in
            dict(state=state.T, action=action.T, setpoint=sp.T, path=path.T, ctrl=ctrl).items()}


def launch6(monkeypatch, mode, cols, packed=True, pad=None):
    """One fp32 6DoF step of the batch cols with set-points held fixed, on the two-environment-per-thread (packed) or the
    one-environment-per-thread kernel; pad fills the padding columns (index >= n) of state, action and ctrl first.
    -> (state, obs, ctrl) [rows, n] and the non-finite count."""
    n = cols["state"].shape[1]
    monkeypatch.setenv("MVRL_NO_X2", "0" if packed else "1")    # read when the env creates its handle (in reset)
    env = BlueROV2Heavy6DoFVecEnv(n, action_mode=mode, dtype=torch.float32, device=DEV, auto_reset=False, maxSteps=NO_STEP_LIMIT)
    env.reset(initialSetpoint=np.zeros(6))
    for k in ("state", "setpoint", "path", "ctrl"):
        getattr(env, "_" + k)[:, :n] = torch.as_tensor(cols[k], device=DEV)
    if pad is not None:
        assert env.ld > n
        for buf in (env._state, env._action, env._ctrl):
            buf[:, n:] = pad
    env.episode_stats()
    env.step(torch.as_tensor(cols["action"], device=DEV))
    out = tuple(t[:, :n].cpu().numpy() for t in (env._state, env._obs, env._ctrl))
    return out, env.episode_stats()["nonfinite"]


def canonical(t):
    """+-0 as +0 (angle_error_v's exact path returns -0.0 for equal angles), NaN (fresh-controller marker) as a number."""
    return np.nan_to_num(t + np.float32(0.0), nan=12345.0)


@pytest.mark.parametrize("mode", ["rpm", "force", "setpoint"])
def test_trig_decision_independent_of_neighbour(monkeypatch, mode):
    """The environments A step to the same bits whatever shares their thread: a small-offset partner and a fall-back
    partner (each in both lane orders), a copy of themselves, a NaN state, an angle of 1e4, or no partner at all
    (MVRL_NO_X2=1).  An odd batch gives the same bits and the same non-finite count with NaN in its padding column."""
    m = 512
    rng = np.random.default_rng(31)
    a_state, a_act, a_sp = (as_dtype(v, torch.float32) for v in env_set_a(rng, mode, m))
    classes = trig_classes(stage_offsets(mode, a_state, a_act, a_sp if mode == "setpoint" else None))
    sizes = {k: int(v.sum()) for k, v in classes.items()}
    assert sizes["anchored"] >= 50 and sizes["fall-back"] >= 50 and sizes["edge"] >= 5, sizes

    small = random_states6(rng, m, 0.0)
    small[:, 3:5] = rng.uniform(-0.3, 0.3, (m, 2))  # near upright: the restoring moments stay small
    small[:, 6:9] = 0.0
    small_act = np.zeros_like(a_act)                 # no thrust, no rates: only the restoring moments turn the vehicle
    fast = random_states6(rng, m, 0.0)
    fast[:, 9:12] = rng.choice([-1, 1], (m, 3)) * rng.uniform(12, 15, (m, 3))
    fast_act = random_actions6(rng, mode, m)
    assert (stage_offsets(mode, small, small_act, small[:, :6] if mode == "setpoint" else None).max(axis=1) < 0.95 * DELTA_MAX2).all()
    assert (stage_offsets(mode, fast, fast_act, fast[:, :6] if mode == "setpoint" else None).max(axis=1) > 1.05 * DELTA_MAX2).all()
    big_angle = random_states6(rng, m, 1.0)
    big_angle[:, 5] = 1e4
    partners = {"small-offset": (small, small_act, small[:, :6]), "fall-back": (fast, fast_act, fast[:, :6]),
                "itself": (a_state, a_act, a_sp), "NaN": (np.full_like(a_state, np.nan), a_act, a_sp),
                "angle 1e4": (big_angle, random_actions6(rng, mode, m), big_angle[:, :6])}
    a_cols = columns6(a_state, a_act, a_sp)

    ref, ref_bad = launch6(monkeypatch, mode, a_cols, packed=False)
    assert ref_bad == 0
    for name, (ps, pa, psp) in partners.items():
        p_cols = columns6(as_dtype(ps, torch.float32), as_dtype(pa, torch.float32), as_dtype(psp, torch.float32))
        for a_lane in ((0, 1) if name in ("small-offset", "fall-back") else (0,)):
            cols = {}
            for k in a_cols:
                cols[k] = np.empty((a_cols[k].shape[0], 2 * m), np.float32)
                cols[k][:, a_lane::2] = a_cols[k]
                cols[k][:, 1 - a_lane::2] = p_cols[k]
            got, _ = launch6(monkeypatch, mode, cols)
            for what, g, r in zip(("state", "obs", "ctrl"), got, ref):
                assert np.array_equal(canonical(g[:, a_lane::2]), canonical(r)), (name, a_lane, what)
    odd = {k: np.ascontiguousarray(v[:, :m - 1]) for k, v in a_cols.items()}
    got0, bad0 = launch6(monkeypatch, mode, odd, pad=0.0)
    got1, bad1 = launch6(monkeypatch, mode, odd, pad=np.nan)
    for what, g0, g1, r in zip(("state", "obs", "ctrl"), got0, got1, ref):
        assert np.array_equal(canonical(g0), canonical(r[:, :m - 1])) and np.array_equal(canonical(g1), canonical(r[:, :m - 1])), what
    assert bad0 == bad1 == 0
    print("6DoF %s fp32: %d environments A (%s) bitwise equal beside %s, alone, and in an odd batch with NaN padding" %
          (mode, m, ", ".join("%s %d" % kv for kv in sizes.items()), " / ".join(partners)))


# ----------------------------------------------------------------- 4. phase B and the out-of-range flag ------------------
OUT_OF_RANGE = (-7.0, -TWO_PI - 0.3, 2 * TWO_PI + 0.3, 13.0, 100.0, 3e4, 6.5e4, 7e4, 1e5)
POSE_ULPS, VEL_ULPS = 4.0, 16.0
# a thruster demand of up to ~50 N computed from angles rounded at ulp/2 moves by ~25 ulp N; at the 0.29 N dead-band edge
# that is ~40 ulp of relative rpm, where the thrust jumps by 0.29 N: excluded with a factor 2 to spare
DEAD_BAND_ULPS = 100.0


def check_against_oracle(r, mode, dtype, ang, angle_in, label):
    """Per-component scaled error <= TOL plus an allowance of ulps of the environment's largest initial angle: the sum y +
    increment of the pose rounds at that ulp at every sub-step, before any kernel arithmetic, and the rounded angles feed
    the trigonometry of every later evaluation.  Observations: 10 TOL plus the same allowance on the heading-error rows,
    except within 1e-3 of the +-pi wrap of the heading error.  -> (errors [n, dim], well-conditioned mask).

    The wrapped angles are the output of the wrap itself, so they are compared as numbers: every one lies in [0, 2 pi],
    and a whole turn of difference counts in full; only within 1e-3 of the 0 / 2 pi seam may the two sides sit on
    opposite ends."""
    tol = TOL[dtype]
    npos = ang.stop       # the angles are the last components of the pose
    u = ulp(angle_in, dtype)[:, None]
    got_a, ref_a = r["state"][:, ang], r["ref"][:, ang]
    two_pi = float(as_dtype(TWO_PI, dtype))        # the kernels wrap with 2 pi rounded to the env's precision
    outside = ~((got_a >= 0.0) & (got_a <= two_pi))
    assert not outside.any(), (label, "wrapped angle outside [0, 2 pi]", got_a[outside.any(axis=1)][:5])
    e = component_errors(r["state"], r["ref"], range(ang.start, ang.stop))
    seam = np.minimum(ref_a, TWO_PI - ref_a) < 1e-3 + 8 * u
    e[:, ang] = np.where(seam, e[:, ang], np.abs(got_a - ref_a) / (1.0 + np.abs(ref_a)))
    allow = np.where(np.arange(e.shape[1]) < npos, POSE_ULPS, VEL_ULPS) * u / (1.0 + np.abs(r["ref"]))
    well = well_conditioned(r, mode, dead_band=1e-4 + DEAD_BAND_ULPS * u[:, 0])
    bad = (e > tol + allow) & well[:, None]
    assert not bad.any(), (label, np.argwhere(bad)[:5], e[bad][:5], angle_in[bad.any(axis=1)][:5])
    if "obs" in r:
        od = np.abs(r["obs"] - r["ref_obs"])
        near_wrap = np.abs(np.abs(o.angle_error(r["sp"][:, 3:6], r["ref"][:, 3:6])) - np.pi) < 1e-3 + 8 * u
        od[:, 6:9][near_wrap] = 0.0
        od_allow = np.where(np.arange(9) >= 6, (VEL_ULPS * 4 / np.pi) * u, 0.0)
        bad = (od > 10 * tol + od_allow) & well[:, None]
        assert not bad.any(), (label, "obs", np.argwhere(bad)[:5], od[bad][:5])
    return e, well


@pytest.mark.parametrize("dtype", [torch.float32, torch.float64], ids=["fp32", "fp64"])
@pytest.mark.parametrize("mode", ["rpm", "setpoint"])
def test_phase_b_and_out_of_range_flag(mode, dtype):
    """6DoF, fixed set-points 10-30 rad from the pose (the PID's exact angle error in set-point mode; phase B of the
    epilogue in every mode) and initial angles in OUT_OF_RANGE on one channel, plus environments with a NaN state.
    nonfinite counts exactly the NaN environments and, in fp32, the ones whose angle ends beyond 2^16."""
    per, n_nan = 96, 16
    rng = np.random.default_rng(41)
    vals = np.repeat(np.array(OUT_OF_RANGE), 3 * per)
    ch = np.tile(np.repeat([0, 1, 2], per), len(OUT_OF_RANGE))
    n = len(vals)
    state = random_states6(rng, n, 0.2)
    state[np.arange(n), 3 + ch] = vals
    sp = state[:, :6] + rng.uniform(-0.5, 0.5, (n, 6))
    sp[:, 3:6] = state[:, 3:6] + rng.choice([-1, 1], (n, 3)) * rng.uniform(10, 30, (n, 3))
    action = random_actions6(rng, mode, n)
    state = np.concatenate([state, np.full((n_nan, 12), np.nan)])
    sp = np.concatenate([sp, rng.uniform(0, TWO_PI, (n_nan, 6))])
    action = np.concatenate([action, random_actions6(rng, mode, n_nan)])
    vals = np.concatenate([vals, np.full(n_nan, np.nan)])
    state, sp, action = (as_dtype(v, dtype) for v in (state, sp, action))
    angle_in = np.abs(state[:, 3:6]).max(axis=1)
    r = step6(mode, dtype, state, action, sp)

    flagged = np.isnan(angle_in) | ((angle_in > F32_MAX_ARG) if dtype == torch.float32 else False)
    print("6DoF %s %s: nonfinite %d, expected %d (%d NaN states)" % (mode, dtype, r["nonfinite"], flagged.sum(), n_nan))
    assert r["nonfinite"] == flagged.sum()
    checked = ~flagged
    sub = {k: v[checked] for k, v in r.items() if isinstance(v, np.ndarray)}
    e, well = check_against_oracle(sub, mode, dtype, slice(3, 6), angle_in[checked], (mode, dtype))
    for v in OUT_OF_RANGE:
        m = (vals[checked] == v) & well
        if dtype == torch.float64 or abs(v) <= F32_MAX_ARG:
            print("  initial angle %9.4g: %3d of %d envs compared, max pose error %.3e, max velocity error %.3e" %
                  (v, m.sum(), 3 * per, e[m, :6].max(initial=0.0), e[m, 6:].max(initial=0.0)))
            # fp32 set-point mode beyond ~100 rad: most environments sit within the widened dead-band exclusion
            assert m.sum() >= (per if mode == "rpm" or DEAD_BAND_ULPS * ulp(v, dtype) < 1e-2 else 8), (v, m.sum())


@pytest.mark.parametrize("dtype", [torch.float32, torch.float64], ids=["fp32", "fp64"])
def test_phase_b_setpoint_below_zero_while_angle_wraps(dtype):
    """Set-point actions (not fixed) that put the set-point below 0 while the angle wraps below 0, or above 2 pi while the
    angle wraps past 2 pi: after the wrap the set-point is more than 2 pi from the angle."""
    n = 2048
    rng = np.random.default_rng(43)
    state = random_states6(rng, n, 0.1)
    state[:, 4] = rng.uniform(-0.5, 0.5, n)
    ch = rng.choice([0, 2], n)                       # roll or yaw
    up = rng.random(n) < 0.5
    rows = np.arange(n)
    state[rows, 3 + ch] = np.where(up, TWO_PI - rng.uniform(0.01, 0.1, n), rng.uniform(0.01, 0.1, n))
    state[rows, 9 + ch] = np.where(up, 1.0, -1.0) * rng.uniform(0.8, 1.5, n)
    action = rng.uniform(-1, 1, (n, 6))
    action[rows, 3 + ch] = np.where(up, 1.0, -1.0)
    state, action = as_dtype(state, dtype), as_dtype(action, dtype)
    r = step6("setpoint", dtype, state, action)
    wrapped = np.abs(r["sp"][rows, 3 + ch] - r["ref"][rows, 3 + ch]) >= TWO_PI
    print("6DoF setpoint %s: %d of %d environments end more than 2 pi from their set-point" % (dtype, wrapped.sum(), n))
    assert wrapped.sum() >= 300
    assert r["nonfinite"] == 0
    e, well = check_against_oracle(r, "setpoint", dtype, slice(3, 6), np.abs(state[:, 3:6]).max(axis=1), dtype)
    print("  max error %.3e over %d well-conditioned envs (%d of them past the wrap)" % (e[well].max(), well.sum(), (well & wrapped).sum()))
    assert (well & wrapped).sum() >= 300


# ----------------------------------------------------------------- 5. the PID's yaw-wrap fall-back ----------------------
def yaw_wrap_case(rng, n, dof):
    """Fixed set-points with the yaw error within 0.05 of +-pi (log-uniform distance, so that the fast 3DoF yaw
    controller, which stops a 1 rad/s turn within a few milliseconds, crosses too) and yaw rates +-1 rad/s."""
    gap = np.exp(rng.uniform(np.log(1e-4), np.log(0.05), n))
    side = rng.choice([-1.0, 1.0], n)
    if dof == 6:
        state = np.zeros((n, 12))
        state[:, 3:5] = rng.uniform(-0.3, 0.3, (n, 2))
        state[:, 5] = rng.uniform(0, TWO_PI, n)
        state[:, 6:11] = rng.uniform(-0.1, 0.1, (n, 5))
        state[:, 11] = rng.choice([-1.0, 1.0], n)
        sp = np.concatenate([rng.uniform(-0.5, 0.5, (n, 3)), rng.uniform(-0.3, 0.3, (n, 2)), np.zeros((n, 1))], axis=1)
        yaw = 5
    else:
        state = np.zeros((n, 6))
        state[:, 2] = rng.uniform(0, TWO_PI, n)
        state[:, 3:5] = rng.uniform(-0.1, 0.1, (n, 2))
        state[:, 5] = rng.choice([-1.0, 1.0], n)
        sp = np.concatenate([rng.uniform(-0.5, 0.5, (n, 2)), np.zeros((n, 1))], axis=1)
        yaw = 2
    sp[:, yaw] = state[:, yaw] + side * (np.pi - gap)
    return state, sp, yaw


@pytest.mark.parametrize("dtype", [torch.float32, torch.float64], ids=["fp32", "fp64"])
@pytest.mark.parametrize("dof", [6, 3])
def test_pid_yaw_wrap_fallback(dof, dtype):
    """Fixed set-points, yaw error near +-pi, yaw rate +-1: the error crosses +-pi inside the step in hundreds of
    environments, where the PID's e - eOld jumps by 2 pi.  One-step error <= TOL (PID margin exclusion)."""
    n, tol = 4096, TOL[dtype]
    rng = np.random.default_rng(51 + dof)
    state, sp, yaw = yaw_wrap_case(rng, n, dof)
    state, sp = as_dtype(state, dtype), as_dtype(sp, dtype)
    action = np.zeros((n, 6 if dof == 6 else 3))
    r = (step6 if dof == 6 else step3)("setpoint", dtype, state, action, sp)
    ang = slice(3, 6) if dof == 6 else slice(2, 3)
    err = scaled_err(r["state"], r["ref"], ang)
    e0 = o.angle_error(sp[:, yaw], state[:, yaw])
    e1 = o.angle_error(sp[:, yaw], r["ref"][:, yaw])
    crossed = (np.sign(e0) != np.sign(e1)) & (np.abs(e0) > np.pi / 2) & (np.abs(e1) > np.pi / 2)
    well = well_conditioned(r, "setpoint")
    print("%dDoF setpoint %s: %d of %d environments crossed +-pi (%d well-conditioned); max error %.3e crossed, %.3e not; "
          "%d excluded" % (dof, dtype, crossed.sum(), n, (crossed & well).sum(), err[crossed & well].max(),
                           err[~crossed & well].max(), (~well).sum()))
    assert (crossed & well).sum() >= 300
    assert err[well].max() <= tol, err[well].max()
    assert well.mean() >= (0.9 if dof == 6 else 0.5), well.mean()   # the 3DoF controller meets small margins often
    assert r["nonfinite"] == 0


# ----------------------------------------------------------------- 6. 3DoF fp32 yaw range -------------------------------
@pytest.mark.parametrize("dtype", [torch.float32, torch.float64], ids=["fp32", "fp64"])
def test_rov3_yaw_out_of_sincos_range_is_flagged(dtype):
    """3DoF, rpm actions, yaw 6e4 / 7e4 / 1e7: in fp32 the two beyond 2^16 are counted in nonfinite (as by the 6DoF
    step); 6e4 is not, and matches the oracle within the allowance of test_phase_b_and_out_of_range_flag.  fp64 counts
    none and matches everywhere."""
    per = 64
    rng = np.random.default_rng(61)
    yaws = np.repeat([6e4, 7e4, 1e7], per)
    n = len(yaws)
    state = np.zeros((n, 6))
    state[:, :2] = rng.uniform(-2, 2, (n, 2))
    state[:, 2] = yaws
    state[:, 3:6] = rng.uniform(-0.5, 0.5, (n, 3))
    action = rng.uniform(-3500, 3500, (n, 4))
    state, action = as_dtype(state, dtype), as_dtype(action, dtype)
    r = step3("rpm", dtype, state, action)
    flagged = (yaws > F32_MAX_ARG) if dtype == torch.float32 else np.zeros(n, dtype=bool)
    print("3DoF rpm %s: nonfinite %d, expected %d" % (dtype, r["nonfinite"], flagged.sum()))
    assert r["nonfinite"] == flagged.sum()
    sub = {k: v[~flagged] for k, v in r.items() if isinstance(v, np.ndarray)}
    e, _ = check_against_oracle(sub, "rpm", dtype, slice(2, 3), yaws[~flagged], dtype)
    print("  max pose error %.3e, max velocity error %.3e" % (e[:, :3].max(), e[:, 3:].max()))
