"""GPU parity tests of the 3DoF path (kernel K3) through the C ABI: vs the
golden vectors produced by the unmodified reference and vs the numpy oracle.
Tolerances as for the 6DoF path: derivatives 1e-10 relative (fp64),
trajectories 1e-8 (fp64) / 1e-4 (fp32)."""
import numpy as np
import pytest
import torch

from conftest import load_golden
from oracle import oracle_np as o

pytestmark = pytest.mark.gpu

if torch.cuda.is_available():
    from marinevehiclereinforcementlearning_b200.rov3 import BlueROV2Heavy3DoFVecEnv, Rov3Derivs
    from marinevehiclereinforcementlearning_b200 import dynamicsModel_BlueROV2_Heavy_3DoF as m3, vec_tools

DEV = "cuda"


def rel_err(a, ref):
    ref = np.asarray(ref)
    scale = np.abs(ref) + np.abs(ref).max(axis=-1, keepdims=True)
    return (np.abs(np.asarray(a) - ref) / np.maximum(scale, 1e-300)).max()


def fm(x, dtype=torch.float64):
    return torch.as_tensor(np.ascontiguousarray(np.asarray(x).T), dtype=dtype, device=DEV)


def sample_states(rng, n):
    return rng.uniform(-1, 1, (n, 6)) * np.array([5., 5., np.pi, 2., 2., 3.])


def test_derivs_rpm_fp64_vs_oracle():
    rng = np.random.default_rng(21)
    s = sample_states(rng, 100_000)
    rpm = rng.uniform(-4000, 4000, (100_000, 4))
    rpm[:100] = 0.0
    s[100:200, 3] = 0.0
    ref = o.derivs3_rpm(o.Rov3Params(), s, rpm)
    got = Rov3Derivs(dtype=torch.float64, action_mode="rpm")(fm(s), fm(rpm)).T.cpu().numpy()
    assert rel_err(got, ref) < 1e-10


def test_thruster_model_vs_golden():
    g = load_golden("rov3")
    f = Rov3Derivs(dtype=torch.float64, action_mode="rpm")
    F, X = f.thrusterModel(torch.as_tensor(g["thr3_uv"][:, 0]), torch.as_tensor(g["thr3_rpm"]))
    assert rel_err(torch.stack([F, X], dim=1).cpu().numpy(), g["thr3_FX"]) < 1e-12


def test_derivs_pid_sequences_fp64_vs_golden():
    g = load_golden("rov3")
    f = Rov3Derivs(dtype=torch.float64, action_mode="setpoint")
    n_env, n_call = g["pid3_t"].shape
    ctrl = Rov3Derivs.new_ctrl(n_env)
    sp = fm(g["pid3_sp"])
    for c in range(n_call):
        d, aux = f(fm(g["pid3_states"][:, c]), t=torch.as_tensor(g["pid3_t"][:, c], device=DEV), setpoint=sp, ctrl=ctrl, want_aux=True)
        assert rel_err(d.T.cpu().numpy(), g["pid3_derivs"][:, c]) < 1e-9, c
        assert np.abs(aux[0:3].T.cpu().numpy() - g["pid3_gcf"][:, c]).max() < 1e-9, c
        assert np.abs(aux[3:7].T.cpu().numpy() - g["pid3_cv"][:, c]).max() < 1e-6, c
    with pytest.raises(ValueError, match="ctrl must be a contiguous"):   # a [7, N] view of an [N, 7] tensor
        f(fm(g["pid3_states"][:, 0]), t=torch.as_tensor(g["pid3_t"][:, 0], device=DEV), setpoint=sp, ctrl=ctrl.T.contiguous().T)


def test_kat3_single_vehicle_dropin():
    """SURVEY.md KAT-3 through the reference-shaped class."""
    g = load_golden("rov3")
    r = m3.BlueROV2Heavy3DoF(np.array([1., -1., 280. / 180. * np.pi]))
    d = r.derivs(0.1, g["kat3_state"])
    assert rel_err(d, g["kat3_derivs"]) < 1e-12
    assert np.abs(r.controlVector - g["kat3_cv"]).max() < 1e-8
    assert np.abs(r.Ainv - g["Ainv3"]).max() < 1e-15
    F, X = r.thrusterModel(0.3, -0.1, 1500.)
    Fr, Xr = o.thruster_model3(o.Rov3Params(), 0.3, 1500.)
    assert abs(F - Fr) < 1e-12 and abs(X - Xr) < 1e-12


def test_trajectory_rpm_fp64_and_fp32_vs_oracle():
    n, steps = 256, 300
    rng = np.random.default_rng(22)
    acts = rng.uniform(-3500, 3500, (steps, n, 4))
    ref = o.Rov3EnvOracle(n, mode=o.MODE_RPM, max_steps=10 ** 9)
    ref.reset(initial_setpoint=np.zeros(3))
    e64 = BlueROV2Heavy3DoFVecEnv(n, action_mode="rpm", dtype=torch.float64, device=DEV, maxSteps=10 ** 9, auto_reset=False)
    e32 = BlueROV2Heavy3DoFVecEnv(n, action_mode="rpm", dtype=torch.float32, device=DEV, maxSteps=10 ** 9, auto_reset=False)
    e64.reset(initialSetpoint=np.zeros(3)); e32.reset(initialSetpoint=np.zeros(3))
    w64 = w32 = 0.0
    for k in range(steps):
        ro, _, _, _ = ref.step(acts[k])
        o64, _, _, _ = e64.step(torch.as_tensor(acts[k], device=DEV))
        e32.step(torch.as_tensor(acts[k], device=DEV, dtype=torch.float32))
        for env, which in ((e64, 0), (e32, 1)):
            d = env.systemState.cpu().numpy().astype(np.float64) - ref.state
            d[:, 2] = (d[:, 2] + np.pi) % (2 * np.pi) - np.pi
            err = (np.abs(d) / (1.0 + np.abs(ref.state))).max()
            if which == 0:
                w64 = max(w64, err)
            else:
                w32 = max(w32, err)
        assert np.abs(o64.cpu().numpy() - ro).max() < 1e-8
    print("3DoF rpm trajectories: fp64 %.2e fp32 %.2e" % (w64, w32))
    assert w64 < 1e-8 and w32 < 1e-4


def test_env_semantics_vs_reference_env_golden():
    g = load_golden("rov3")
    env = BlueROV2Heavy3DoFVecEnv(1, action_mode="setpoint", dtype=torch.float64, device=DEV, maxSteps=50, auto_reset=False, record_aux=True)
    obs = [env.reset(initialSetpoint=g["env3_fixed_sp"]).cpu().numpy()[0]]
    states = []
    for k in range(50):
        ob, r, d, _ = env.step(torch.zeros((1, 3), dtype=torch.float64, device=DEV))
        obs.append(ob.cpu().numpy()[0]); states.append(env.systemState.cpu().numpy()[0])
        assert bool(d[0]) == bool(g["env3_fixed_done"][k]) and float(r[0]) == 0.0
    assert np.abs(np.array(obs) - g["env3_fixed_obs"]).max() < 1e-8
    assert np.abs(np.array(states) - g["env3_fixed_history"][1:, 1:7]).max() < 1e-8

    env = BlueROV2Heavy3DoFVecEnv(1, action_mode="setpoint", dtype=torch.float64, device=DEV, maxSteps=40, auto_reset=False)
    env.reset(initialSetpoint=np.append(g["env3_act_path"][0], g["env3_act_heading"]))
    env._path[:, 0] = torch.as_tensor(g["env3_act_path"].reshape(-1), device=DEV)
    env.fixedSp = False
    for k in range(40):
        ob, r, d, _ = env.step(torch.as_tensor(g["env3_act_actions"][k:k + 1], device=DEV))
        assert np.abs(ob.cpu().numpy()[0] - g["env3_act_obs"][k + 1]).max() < 1e-7, k
        assert np.abs(env.systemState.cpu().numpy()[0] - g["env3_act_history"][k + 1, 1:7]).max() < 1e-7, k
        assert bool(d[0]) == bool(g["env3_act_done"][k])


def test_single_env_dropin_matches_reference_env_golden():
    g = load_golden("rov3")
    env = m3.BlueROV2Heavy3DoFEnv(maxSteps=50)
    assert env.action_space.shape == (3,) and env.observation_space.shape == (5,)
    obs = [env.reset(initialSetpoint=list(g["env3_fixed_sp"]))]
    for k in range(50):
        ob, r, d, info = env.step(np.zeros(3))
        obs.append(ob)
        assert r == 0.0 and info == {} and d == bool(g["env3_fixed_done"][k])
    assert np.abs(np.array(obs) - g["env3_fixed_obs"]).max() < 1e-8
    h = env.timeHistory  # pandas DataFrame on done, 17 columns (3DoF.py:502-508)
    assert list(h.columns)[:2] == ["t", "x0"] and h.shape == (51, 17)
    ref = g["env3_fixed_history"]
    assert np.abs(h.values[:, :7] - ref[:, :7]).max() < 1e-8 and np.abs(h.values[:, 14:] - ref[:, 14:]).max() < 1e-12
    assert env.steps_beyond_done == 1


def test_auto_reset_and_sharding_bitwise():
    n, steps = 256, 9
    rng = np.random.default_rng(23)
    acts = rng.uniform(-3500, 3500, (steps, n, 4))
    mk = lambda m, id0: BlueROV2Heavy3DoFVecEnv(m, action_mode="rpm", dtype=torch.float64, device=DEV, maxSteps=4, auto_reset=True,
                                                 seed=77, env_id0=id0)
    full, a, b = mk(n, 0), mk(n // 2, 0), mk(n // 2, n // 2)
    ref = o.Rov3EnvOracle(n, mode=o.MODE_RPM, max_steps=4, auto_reset=True, seed=77)
    o0 = full.reset().cpu().numpy(); a.reset(); b.reset()
    assert np.abs(o0 - ref.reset()).max() < 1e-12
    for k in range(steps):
        act = torch.as_tensor(acts[k], device=DEV)
        obs, rew, done, info = full.step(act)
        oa, _, da, _ = a.step(act[: n // 2]); ob, _, db, _ = b.step(act[n // 2:])
        assert torch.equal(obs, torch.cat([oa, ob])) and torch.equal(full.systemState, torch.cat([a.systemState, b.systemState]))
        ro, rr, rd, rinfo = ref.step(acts[k])
        assert np.array_equal(done.cpu().numpy(), rd) and np.abs(obs.cpu().numpy() - ro).max() < 1e-9
        if rd.any():
            assert np.abs(info["terminal_observation"].cpu().numpy()[rd] - rinfo["terminal_observation"][rd]).max() < 1e-9
            assert np.abs(full.path.cpu().numpy().reshape(n, 4) - ref.path).max() < 1e-12
    st = full.episode_stats()
    assert st["episodes"] == n * (steps // 4) and st["mean_length"] == 4.0 and st["nonfinite"] == 0
    # no range or host step for the 3DoF env: EnvBlocks refuses it when it is built
    assert not hasattr(full, "step_range_async") and not hasattr(full, "step_host")
    with pytest.raises(TypeError):
        vec_tools.EnvBlocks(full, 2)


def test_los_navigation_vs_reference_golden():
    """lineOfSight / LOSNavigation.predict (3DoF.py:517-607) through mvrl_los_navigation."""
    g = load_golden("agents")
    nav = m3.LOSNavigation()
    nav_obs = g["nav_obs"]
    act, states = nav.predict(nav_obs)
    assert act.shape == (500, 3) and np.abs(act - g["nav_action"]).max() < 1e-13 and states is nav_obs
    a1, _ = nav.predict(g["nav_obs"][7])
    assert a1.shape == (3,) and np.abs(a1 - g["nav_action"][7]).max() < 1e-13
    for i in (0, 60, 90, 170, 210, 300, 2999):   # each branch family of the generator
        t = m3.lineOfSight(g["los_p0"][i], g["los_p1"][i], float(g["los_rnav"][i]))
        assert np.abs(t - g["los_target"][i]).max() < 1e-13, i
    # batched on the device, all 3000 cases at Rnav = 0.5 vs the oracle, fp64 and fp32
    obs = np.concatenate([g["los_p0"], g["los_p1"], np.zeros((3000, 1))], axis=1)
    want = o.los_navigation_predict(obs, 0.5)
    got, _ = nav.predict(torch.as_tensor(obs, device=DEV))
    assert np.abs(got.cpu().numpy() - want).max() < 1e-12
    got32, _ = nav.predict(torch.as_tensor(obs, device=DEV, dtype=torch.float32))
    close = np.abs(got32.cpu().numpy() - want).max(axis=1) < 1e-4      # fp32 may take the other branch at a tie
    assert close.mean() > 0.995
    # closing the loop: the heuristic drives the batched 3DoF env along its path
    env = BlueROV2Heavy3DoFVecEnv(64, action_mode="setpoint", dtype=torch.float64, device=DEV, maxSteps=200, auto_reset=False, seed=2)
    ob = env.reset()
    d0 = torch.linalg.norm(env.path[:, 1] - env.systemState[:, :2], dim=1)
    for _ in range(200):
        a, _ = nav.predict(ob)
        ob, _, _, _ = env.step(a)
    d1 = torch.linalg.norm(env.path[:, 1] - env.systemState[:, :2], dim=1)
    assert (d1 < 0.5 * d0).float().mean() > 0.9
