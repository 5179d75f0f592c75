"""GPU: the squashed head's weight sync from a learner's CUDA tensors (``load_state_dict(sd, share=True)`` ->
``mvrl_policy_set_weights_squashed_device``, one packing kernel on the caller's stream) against the host entry that the
same kernel serves through a staging buffer.  Both must give the same packed blocks, so every output is compared bit for
bit."""
import ctypes as C
import math

import pytest
import torch

pytestmark = pytest.mark.gpu

if torch.cuda.is_available():
    from marinevehiclereinforcementlearning_b200 import BlueROV2Heavy6DoFVecEnv, SquashedGaussianPolicy, _lib
    from marinevehiclereinforcementlearning_b200.vec_tools import EnvBlocks

DEV = "cuda:0"
SHAPES = [(9, 6), (11, 3), (1, 1), (16, 8)]
KERNELS = [("bf16", False), ("fp32", False), ("bf16", True)]   # (precision, MVRL_POLICY_MMA_SYNC=1)
OUTPUTS = ("act", "mean", "log_std", "eps", "logp")


def actor_sd(obs_dim, act_dim, seed=5):
    """SB3-named Actor parameters (fp32, CPU) with non-zero biases and log_std biases on both sides of the [-20, 2] clamp."""
    g = torch.Generator().manual_seed(seed)
    sd = {}
    for name, fan_in, fan_out in (("latent_pi.0", obs_dim, 128), ("latent_pi.2", 128, 128), ("latent_pi.4", 128, 128),
                                  ("mu", 128, act_dim), ("log_std", 128, act_dim)):
        sd[name + ".weight"] = torch.randn(fan_out, fan_in, generator=g) / math.sqrt(fan_in)
        sd[name + ".bias"] = torch.rand(fan_out, generator=g) * 0.6 - 0.3
    sd["log_std.bias"] = torch.linspace(-26.0, 5.0, act_dim) if act_dim > 1 else torch.tensor([3.0])
    return sd


def offset_views(sd):
    """CUDA copies of ``sd`` that start one float into a larger allocation: a storage offset, 4-byte alignment only."""
    out = {}
    for k, v in sd.items():
        big = torch.empty(v.numel() + 1, device=DEV)
        t = big[1:].view(v.shape)
        t.copy_(v)
        assert t.storage_offset() == 1
        out[k] = t
    return out


def buffers(obs_dim, act_dim, n, seed=0):
    ld = (n + 31) // 32 * 32
    g = torch.Generator(device=DEV).manual_seed(seed)
    obs = torch.zeros((obs_dim, ld), device=DEV)
    obs[:, :n] = torch.rand((obs_dim, n), generator=g, device=DEV) * 4 - 2
    z = lambda k: torch.full((k, ld), 7.0, device=DEV)
    return dict(obs=obs, act=z(act_dim), mean=z(act_dim), log_std=z(act_dim), eps=z(act_dim), logp=torch.full((ld,), 7.0, device=DEV))


def run(pol, b, n, step=4, deterministic=False):
    pol.act_into(b["obs"], b["act"], n, logp=b["logp"], mean=b["mean"], eps=b["eps"], log_std=b["log_std"], env_id0=11, step=step,
                 deterministic=deterministic)
    torch.cuda.synchronize()
    return {k: b[k].clone() for k in OUTPUTS}


def assert_bitwise(x, y, what=""):
    for k in OUTPUTS:
        assert torch.equal(x[k].view(torch.int32), y[k].view(torch.int32)), (what, k)


def policy(obs_dim, act_dim, precision, noise=None, seed=3):
    return SquashedGaussianPolicy(obs_dim, act_dim, device=DEV, seed=seed, action_noise_std=noise, precision=precision)


@pytest.mark.parametrize("noise", [None, 0.3])
@pytest.mark.parametrize("obs_dim,act_dim", SHAPES)
@pytest.mark.parametrize("precision,mma_sync", KERNELS)
def test_device_path_matches_host_path_bitwise(monkeypatch, precision, mma_sync, obs_dim, act_dim, noise):
    if mma_sync:
        monkeypatch.setenv("MVRL_POLICY_MMA_SYNC", "1")
    sd = actor_sd(obs_dim, act_dim)
    host = policy(obs_dim, act_dim, precision, noise).load_state_dict(sd)
    dev = policy(obs_dim, act_dim, precision, noise).load_state_dict(offset_views(sd), share=True)
    for n in (1, 129, 131072):
        b = buffers(obs_dim, act_dim, n)
        for det in (False, True):
            assert_bitwise(run(host, b, n, deterministic=det), run(dev, b, n, deterministic=det), (n, det))
    if act_dim > 1:   # the clamp is exercised on both sides
        ls = run(dev, buffers(obs_dim, act_dim, 129), 129)["log_std"][:, :129]
        assert (ls == -20.0).any() and (ls == 2.0).any()


@pytest.mark.parametrize("precision", ["bf16", "fp32"])
def test_in_place_learner_updates_are_seen(precision):
    obs_dim, act_dim, n = 9, 6, 4096
    shared = {k: v.to(DEV) for k, v in actor_sd(obs_dim, act_dim).items()}
    pol = policy(obs_dim, act_dim, precision, 0.1).load_state_dict(shared, share=True)
    b = buffers(obs_dim, act_dim, n)
    before = run(pol, b, n)
    for i, v in enumerate(shared.values()):   # what an optimiser step does: in-place updates of the same storage
        v.mul_(1.0 - 0.01 * (i + 1)).add_(0.002 * (i + 1))
    pol.sync_weights()
    after = run(pol, b, n)
    fresh = policy(obs_dim, act_dim, precision, 0.1).load_state_dict({k: v.cpu() for k, v in shared.items()})
    assert_bitwise(after, run(fresh, b, n))
    assert not torch.equal(before["mean"], after["mean"])


def test_device_sync_does_not_block_the_host():
    obs_dim, act_dim, n = 9, 6, 4096
    shared = {k: v.to(DEV) for k, v in actor_sd(obs_dim, act_dim).items()}
    pol = policy(obs_dim, act_dim, "bf16").load_state_dict(shared, share=True)
    for v in shared.values():
        v.mul_(0.5)
    torch.cuda.synchronize()
    b = buffers(obs_dim, act_dim, n)
    side = torch.cuda.Stream(device=DEV)
    with torch.cuda.stream(side):
        torch.cuda._sleep(100_000_000)    # ~50 ms of device time ahead of the packing kernel
        pol.sync_weights()
        assert not side.query()           # returned while the stream is still busy: no synchronisation
        pol.act_into(b["obs"], b["act"], n, logp=b["logp"], mean=b["mean"], eps=b["eps"], log_std=b["log_std"], env_id0=11, step=4)
    side.synchronize()
    got = {k: b[k].clone() for k in OUTPUTS}
    fresh = policy(obs_dim, act_dim, "bf16").load_state_dict({k: v.cpu() for k, v in shared.items()})
    assert_bitwise(got, run(fresh, buffers(obs_dim, act_dim, n), n))


def test_cuda_graph_of_update_sync_act_step():
    """T iterations of (in-place parameter update, sync_weights, act, env step) captured as one CUDA graph and replayed, against
    the same sequence run eagerly through the host entry from the same start state."""
    n, T = 4096, 4
    env = BlueROV2Heavy6DoFVecEnv(n, action_mode="setpoint", dtype=torch.float32, device=DEV, seed=7, auto_reset=True, maxSteps=3)
    env.reset()
    start_env = env.state_dict()
    start = {k: v.to(DEV) for k, v in actor_sd(9, 6).items()}
    shared = {k: v.clone() for k, v in start.items()}
    pol = policy(9, 6, "bf16", 0.2).load_state_dict(shared, share=True)
    acts = torch.zeros((T, 6, env.ld), device=DEV)
    obs = torch.zeros((T, 9, env.ld), device=DEV)

    def update(params):
        for v in params.values():
            v.mul_(0.97).add_(0.001)

    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        for t in range(T):
            update(shared)
            pol.sync_weights()
            pol.act(env, step=100 + t)
            env.step_async()
            acts[t].copy_(env._action)
            obs[t].copy_(env._obs)
    graph.replay()
    torch.cuda.synchronize()

    env.load_state_dict(start_env)
    eager = {k: v.clone() for k, v in start.items()}
    ref = policy(9, 6, "bf16", 0.2)
    for t in range(T):
        update(eager)
        ref.load_state_dict({k: v.cpu() for k, v in eager.items()})
        ref.act(env, step=100 + t)
        env.step_async()
        torch.cuda.synchronize()
        assert torch.equal(acts[t].view(torch.int32), env._action.view(torch.int32)), t
        assert torch.equal(obs[t].view(torch.int32), env._obs.view(torch.int32)), t
    assert torch.equal(torch.cat([v.flatten() for v in shared.values()]), torch.cat([v.flatten() for v in eager.values()]))


def test_env_blocks_act_after_device_sync():
    """sync_weights() on the caller's stream; the per-block acts on the EnvBlocks streams (forked from it) see the new weights."""
    n = 4096
    env = BlueROV2Heavy6DoFVecEnv(n, action_mode="setpoint", dtype=torch.float32, device=DEV, seed=7)
    env.reset()
    shared = {k: v.to(DEV) for k, v in actor_sd(9, 6).items()}
    pol = policy(9, 6, "bf16", 0.2).load_state_dict(shared, share=True)
    torch.cuda.synchronize()
    blocks = EnvBlocks(env, 4, align=128)
    ld = env.ld
    out = {k: torch.full((6, ld), 7.0, device=DEV) for k in ("act", "mean", "log_std", "eps")}
    out["logp"] = torch.full((ld,), 7.0, device=DEV)
    for v in shared.values():
        v.mul_(0.9)
    torch.cuda._sleep(20_000_000)   # the update and the sync are still queued when the blocks are forked
    pol.sync_weights()
    with blocks:
        for lo, cnt, s in blocks:
            with torch.cuda.stream(s):
                p = lambda k: C.c_void_p(out[k].data_ptr() + 4 * lo)
                _lib.check(pol.lib.mvrl_policy_act_ex(pol._h, cnt, ld, C.c_void_p(env._obs.data_ptr() + 4 * lo), p("act"), p("logp"), p("mean"),
                                                      p("log_std"), p("eps"), pol.seed, lo, 9, 0, _lib.current_stream(DEV)))
    torch.cuda.synchronize()
    whole = {k: torch.full_like(v, 7.0) for k, v in out.items()}
    pol.act_into(env._obs, whole["act"], n, logp=whole["logp"], mean=whole["mean"], eps=whole["eps"], log_std=whole["log_std"], step=9)
    torch.cuda.synchronize()
    assert_bitwise(out, whole)
    fresh = policy(9, 6, "bf16", 0.2).load_state_dict({k: v.cpu() for k, v in shared.items()})
    again = {k: torch.full_like(v, 7.0) for k, v in out.items()}
    fresh.act_into(env._obs, again["act"], n, logp=again["logp"], mean=again["mean"], eps=again["eps"], log_std=again["log_std"], step=9)
    torch.cuda.synchronize()
    assert_bitwise(out, again)


def test_rejections():
    sd = actor_sd(9, 6)
    pol = policy(9, 6, "bf16")
    cuda = {k: v.to(DEV) for k, v in sd.items()}
    bad = [dict(sd),                                                                       # CPU
           dict(cuda, **{"mu.weight": cuda["mu.weight"].double()}),                        # float64
           dict(cuda, **{"latent_pi.2.weight": cuda["latent_pi.2.weight"].T.contiguous().T})]   # non-contiguous
    if torch.cuda.device_count() > 1:
        bad.append(dict(cuda, **{"mu.bias": cuda["mu.bias"].to("cuda:1")}))                # another device
    for b in bad:
        with pytest.raises(ValueError, match="share=True"):
            pol.load_state_dict(b, share=True)

    lib = _lib.load()
    names = list(sd)
    ptrs = [C.c_void_p(cuda[k].data_ptr()) for k in names]
    stream = _lib.current_stream(DEV)
    fn = lib.mvrl_policy_set_weights_squashed_device
    assert fn(pol._h, *ptrs, None, stream) == 0

    def rejected(rc, text):
        assert rc == -1 and text in lib.mvrl_last_error().decode(), lib.mvrl_last_error()

    fixed = C.c_void_p()
    _lib.check(lib.mvrl_policy_create_head(C.byref(fixed), 0, 9, 6, _lib.POLICY_HEAD_FIXED_STD))
    try:
        rejected(fn(fixed, *ptrs, None, stream), "fixed-std head")
    finally:
        lib.mvrl_policy_destroy(fixed)
    rejected(fn(None, *ptrs, None, stream), "null")
    c_names = ["W1", "b1", "W2", "b2", "W3", "b3", "W_mu", "b_mu", "W_log_std", "b_log_std"]
    for i in range(10):
        rejected(fn(pol._h, *(ptrs[:i] + [None] + ptrs[i + 1:]), None, stream), "null argument " + c_names[i])
    host_w = sd["latent_pi.2.weight"].contiguous()
    rejected(fn(pol._h, *(ptrs[:2] + [C.c_void_p(host_w.data_ptr())] + ptrs[3:]), None, stream), "W2 is not device memory")
    for v in (float("nan"), -0.5, float("inf")):
        noise = (C.c_float * 6)(0.1, 0.1, v, 0.1, 0.1, 0.1)
        rejected(fn(pol._h, *ptrs, noise, stream), "noise_std[2]")
    torch.cuda.synchronize()
