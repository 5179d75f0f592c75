"""Rollout actor next to the env: the SB3 ``MlpPolicy`` of the reference's training scripts
(tag_00_Dec2023_simpleControlTurbulence/main_00_sbl.py:100-105: ``net_arch=[128, 128, 128]``, GELU) with a Gaussian action
head, evaluated by ONE tensor-core kernel (``mvrl_policy_act``, csrc/mvrl_policy.cu) directly on the batched env's
structure-of-arrays observation / action buffers - so that collecting a rollout step is two launches: actor, env step.

Two heads: ``MlpGaussianPolicy`` (a generic state-independent-std head) and ``SquashedGaussianPolicy`` (the Actor of SB3
SAC / sb3_contrib TQC, loadable from their state dicts).  Two precisions for either, chosen at construction: ``"bf16"`` (the
default and the fast mode: bf16 operands, GELU in its tanh form) and ``"fp32"`` (SB3's fp32 network: split-bf16 tensor-core
products, GELU in its erf form; within 5e-5 of the network in fp64).

The parameters live in ordinary fp32 torch tensors (a learner may update them in place); ``sync_weights()`` repacks them
into the kernel's operand layout (bf16, or bf16 hi / lo pairs for precision="fp32"; canonical K-major core matrices for
tcgen05.mma) with one packing kernel.  ``SquashedGaussianPolicy.load_state_dict(sd, share=True)`` keeps references to a
learner's CUDA tensors; its ``sync_weights()`` then packs them in place on the current stream, without a host copy or a
synchronisation, and can be captured in a CUDA graph.

``CriticTarget`` is the one piece of the SAC / TQC learner that needs no gradients: the critic target of a replay sample
(next action and log-prob by the fp32 actor, the target critics, TQC's truncated quantiles or SAC's minimum, the entropy and
discount terms) as one fp32 tensor-core kernel (``mvrl_critic_target``, DESIGN.md K10).  ``quantile_huber_loss`` is TQC's
critic loss on that target, sb3_contrib's function with its gradient fused into one kernel behind autograd
(``mvrl_quantile_huber_loss``, DESIGN.md K11).  ``Critic`` is the critics' forward pass on the learner's own parameters
with its backward pass to those parameters and to the actions (``mvrl_critic_forward`` / ``mvrl_critic_backward``,
DESIGN.md K12), behind autograd.  ``Actor`` is the learner's ``actor.action_log_prob`` on the actor's own parameters with
its backward pass to those parameters (``mvrl_actor_forward`` / ``mvrl_actor_backward``, DESIGN.md K13), behind autograd.
So every network pass of a SAC / TQC gradient step runs on the library's kernels; the scalar actor and entropy losses,
the optimisers and the Polyak update stay in PyTorch."""
import ctypes as C
import math

import torch

from . import _lib
from .rov6 import _device_index

HIDDEN = 128
PRECISIONS = {"bf16": _lib.POLICY_PRECISION_BF16, "fp32": _lib.POLICY_PRECISION_FP32}


def _check_precision(precision):
    if precision not in PRECISIONS:
        raise ValueError("precision must be one of %s, got %r" % (sorted(PRECISIONS), precision))
    return precision


class _FusedActor(_lib.Handle):
    """The plumbing both heads share: the library handle, sampling into feature-major buffers, SB3 ``predict``."""

    def _open(self, device, obs_dim, act_dim, seed, head):
        self.device = torch.device("cuda", _device_index(device))
        self.obs_dim, self.act_dim, self.seed = int(obs_dim), int(act_dim), int(seed)
        self.step = 0
        super().__init__("mvrl_policy", self.device.index, self.obs_dim, self.act_dim, head, PRECISIONS[self.precision],
                         create="create_ex")

    def act_into(self, obs_fm, act_fm, n, logp=None, mean=None, eps=None, env_id0=0, step=None, deterministic=False, log_std=None):
        """obs_fm float32 [obs_dim, ld] -> act_fm float32 [act_dim, ld] (feature-major, as the envs hold them); no sync.
        ``log_std`` [act_dim, ld] is an output of the squashed head only."""
        if step is None:
            step, self.step = self.step, self.step + 1
        ld = obs_fm.shape[1]
        for t, rows in ((obs_fm, self.obs_dim), (act_fm, self.act_dim), (mean, self.act_dim), (eps, self.act_dim), (log_std, self.act_dim)):
            if t is not None and (t.dtype != torch.float32 or t.device != self.device or t.shape[0] < rows or t.shape[1] != ld or not t.is_contiguous()):
                raise ValueError("feature-major float32 tensors [k, %d] on %s expected" % (ld, self.device))
        _lib.check(self.lib.mvrl_policy_act_ex(self._h, int(n), int(ld), _lib.ptr(obs_fm), _lib.ptr(act_fm), _lib.ptr(logp), _lib.ptr(mean),
                                               _lib.ptr(log_std), _lib.ptr(eps), self.seed & (2 ** 64 - 1), int(env_id0), int(step) & 0xffffffff,
                                               int(bool(deterministic)), _lib.current_stream(self.device)))

    def act(self, env, logp=None, deterministic=False, step=None):
        """Sample actions for a batched env straight into its action buffer (the next ``env.step_async()`` reads them)."""
        self.act_into(env._obs, env._action, env.num_envs, logp=logp, env_id0=env.env_id0, step=step, deterministic=deterministic)
        return env.actions_fm

    def predict(self, obs, state=None, episode_start=None, deterministic=False):
        """SB3 ``predict``: numpy / tensor observations [obs_dim] or [N, obs_dim] -> (actions, None)."""
        x = torch.as_tensor(obs, dtype=torch.float32)
        single = x.dim() == 1
        x = x.reshape(-1, self.obs_dim).to(self.device)
        n = x.shape[0]
        ld = max(32, (n + 31) // 32 * 32)
        o = torch.zeros((self.obs_dim, ld), dtype=torch.float32, device=self.device)
        o[:, :n] = x.T
        a = torch.zeros((self.act_dim, ld), dtype=torch.float32, device=self.device)
        self.act_into(o, a, n, deterministic=deterministic)
        out = a[:, :n].T.cpu().numpy()
        return (out[0] if single else out), None


class MlpGaussianPolicy(_FusedActor):
    """obs_dim -> 128 -> 128 -> 128 -> act_dim, GELU (tanh form), tanh-squashed mean, state-independent ``log_std``.

    ``act(env)`` / ``act_into(obs_fm, act_fm, ...)`` sample ``a = clip(mean + std * eps, -1, 1)`` with ``eps`` from Philox
    keyed on (seed, global env id, step): the draw of an environment does not depend on the batch layout or the number
    of GPUs.  ``predict(obs, deterministic)`` is the SB3-shaped entry point (numpy in / out) the reference's
    ``evaluate_agent`` loop calls (resources.py:145-198).  This head is generic, not the one SB3 trains: for an agent
    trained with SAC / TQC use ``SquashedGaussianPolicy``.

    ``precision="bf16"`` (default) is the fast mode: bf16 operands, GELU in its tanh form, ``tanh.approx`` for the mean.
    ``precision="fp32"`` evaluates the network in fp32 as PyTorch does (split-bf16 tensor-core products, ``nn.GELU()``'s
    erf form, accurate ``tanh``); the noise is the same bit for bit."""

    def __init__(self, obs_dim, act_dim, device="cuda", seed=0, log_std_init=-0.5, precision="bf16"):
        self.precision = _check_precision(precision)
        g = torch.Generator().manual_seed(int(seed))
        dims = [int(obs_dim), HIDDEN, HIDDEN, HIDDEN, int(act_dim)]
        self.weights = [torch.randn(dims[i + 1], dims[i], generator=g) / math.sqrt(dims[i]) for i in range(4)]   # nn.Linear layout [out, in]
        self.biases = [torch.zeros(dims[i + 1]) for i in range(4)]
        self.log_std = torch.full((int(act_dim),), float(log_std_init))
        self._open(device, obs_dim, act_dim, seed, _lib.POLICY_HEAD_FIXED_STD)
        self.sync_weights()

    def sync_weights(self):
        """Repack the fp32 parameters (any device) into the kernel's operand layout.  Call after a learner update."""
        host = [t.detach().to("cpu", torch.float32).contiguous() for t in
                (self.weights[0], self.biases[0], self.weights[1], self.biases[1], self.weights[2], self.biases[2],
                 self.weights[3], self.biases[3], self.log_std)]
        _lib.check(self.lib.mvrl_policy_set_weights(self._h, *[C.c_void_p(t.data_ptr()) for t in host]))

    @property
    def logp_const(self):
        return float(-self.log_std.sum())


def squashed_param_shapes(obs_dim, act_dim):
    """SB3 names and shapes of the SAC / TQC ``Actor`` parameters (net_arch [128, 128, 128], no gSDE), in upload order."""
    return {"latent_pi.0.weight": (HIDDEN, obs_dim), "latent_pi.0.bias": (HIDDEN,),
            "latent_pi.2.weight": (HIDDEN, HIDDEN), "latent_pi.2.bias": (HIDDEN,),
            "latent_pi.4.weight": (HIDDEN, HIDDEN), "latent_pi.4.bias": (HIDDEN,),
            "mu.weight": (act_dim, HIDDEN), "mu.bias": (act_dim,),
            "log_std.weight": (act_dim, HIDDEN), "log_std.bias": (act_dim,)}


def actor_params_from_state_dict(sd, obs_dim, act_dim):
    """The Actor parameters of an SB3 state dict -> {SB3 name: fp32 CPU tensor}.  ``sd`` is an ``Actor`` state dict or a
    whole SAC / TQC policy state dict (keys ``actor.*``; critic and other keys are ignored).  Raises ``ValueError`` for a
    missing key, a shape mismatch, or a gSDE actor (``log_std`` a Parameter, not a Linear)."""
    return {k: t.to("cpu", torch.float32).clone().contiguous() for k, t in _actor_tensors(sd, obs_dim, act_dim).items()}


def _strip_prefix(sd, prefixes):
    """The entries of ``sd`` under the first of ``prefixes`` that any key starts with, that prefix removed; else ``sd``."""
    for prefix in prefixes:
        if any(k.startswith(prefix) for k in sd):
            return {k[len(prefix):]: v for k, v in sd.items() if k.startswith(prefix)}
    return sd


def _check_shared(params, device):
    """``share=True``: every tensor of ``params`` {name: tensor} float32, contiguous and on ``device``, else ``ValueError``."""
    for name, t in params.items():
        if t.dtype != torch.float32 or not t.is_contiguous() or t.device != device:
            raise ValueError("share=True needs float32 contiguous tensors on %s; %r is %s%s on %s"
                             % (device, name, t.dtype, "" if t.is_contiguous() else " (non-contiguous)", t.device))
    return params


def _actor_tensors(sd, obs_dim, act_dim, detach=True):
    """The checks of ``actor_params_from_state_dict``; the tensors as given (detached unless ``detach=False``: they share
    storage with ``sd``'s)."""
    sd = _strip_prefix(sd, ("actor.",))
    if "log_std" in sd:
        raise ValueError("the state dict is of a gSDE actor (use_sde=True: log_std is a Parameter, not a Linear layer); "
                         "gSDE is not supported")
    out = {}
    for name, shape in squashed_param_shapes(obs_dim, act_dim).items():
        if name not in sd:
            raise ValueError("actor state dict has no %r" % name)
        t = torch.as_tensor(sd[name])
        t = t.detach() if detach else t
        if tuple(t.shape) != shape:
            raise ValueError("%r has shape %s, expected %s (obs_dim %d, act_dim %d, net_arch [128, 128, 128])"
                             % (name, tuple(t.shape), shape, obs_dim, act_dim))
        out[name] = t
    return out


class SquashedGaussianPolicy(_FusedActor):
    """The Actor of SB3 SAC / sb3_contrib TQC (``MlpPolicy``, net_arch [128, 128, 128], GELU) with its squashed Gaussian head: ``mu`` and ``log_std`` (clamped to [-20, 2]) are two Linear layers on the
    last hidden layer, ``a = tanh(mu + exp(log_std) * eps)``, and ``logp`` is the log-prob of ``a`` with the tanh Jacobian,
    as SB3's ``SquashedDiagGaussianDistribution`` computes it.  ``eps`` comes from the same Philox stream as
    ``MlpGaussianPolicy``'s.

    ``action_noise_std`` (a float or one per action dimension; None = off) adds SB3's ``NormalActionNoise`` of off-policy
    collection: ``act = clip(a + action_noise_std * xi, -1, 1)`` with ``xi`` from its own Philox stream; ``eps`` and
    ``logp`` do not change with it.  It applies to every non-deterministic call, ``predict`` included.
    ``deterministic=True`` gives ``tanh(mu)`` (SB3 ``predict(obs, deterministic=True)``).  ``act_into(mean=)`` returns
    ``mu`` (before tanh), ``act_into(log_std=)`` the clamped log std.

    Parameters are held under SB3's names (``params``); ``load_state_dict`` takes a trained agent's actor or policy state
    dict, e.g. ``SquashedGaussianPolicy(9, 6, precision="fp32").load_state_dict(TQC.load(path).policy.state_dict())``.

    ``precision``: ``"bf16"`` (default) is the fast mode for rollout collection - bf16 operands and GELU in its tanh form,
    ``mu`` within ~4e-3 of SB3's network.  ``"fp32"`` is the one that reproduces ``agent.predict``: the network in fp32 with
    ``nn.GELU()``'s erf form, as SB3 evaluates it (split-bf16 tensor-core products, within 5e-5 of the fp64 network), at
    about 7x the kernel time (166 vs 24 us at 131 072 environments on a B200; PyTorch's fp32 evaluation takes 547 us).  ``eps``, the action noise, the clamp and ``logp`` are the same in both."""

    def __init__(self, obs_dim, act_dim, device="cuda", seed=0, action_noise_std=None, precision="bf16"):
        self.precision = _check_precision(precision)
        g = torch.Generator().manual_seed(int(seed))
        self.params = {}
        for name, shape in squashed_param_shapes(int(obs_dim), int(act_dim)).items():
            self.params[name] = torch.randn(shape, generator=g) / math.sqrt(shape[1]) if len(shape) == 2 else torch.zeros(shape)
        self.action_noise_std = action_noise_std
        self._open(device, obs_dim, act_dim, seed, _lib.POLICY_HEAD_SQUASHED)
        self.sync_weights()

    def state_dict(self):
        """{SB3 Actor name: fp32 tensor} (copies)."""
        return {k: v.detach().clone() for k, v in self.params.items()}

    def load_state_dict(self, sd, share=False):
        """Take the Actor parameters of an SB3 SAC / TQC state dict (see ``actor_params_from_state_dict``) and upload them.

        ``share=False`` keeps fp32 CPU copies.  ``share=True`` keeps REFERENCES to the given tensors, e.g. those of
        ``agent.actor.state_dict()`` or of a SAC / TQC policy state dict (``actor.*`` keys), which share storage with the
        learner's parameters: an in-place ``optimizer.step()`` is then seen by the next ``sync_weights()``, which packs them
        on the device (see there).  Every tensor must be float32, contiguous and on this policy's device; otherwise
        ``ValueError``."""
        if share:
            self.params = _check_shared(_actor_tensors(sd, self.obs_dim, self.act_dim), self.device)
        else:
            self.params = actor_params_from_state_dict(sd, self.obs_dim, self.act_dim)
        self.sync_weights()
        return self

    def sync_weights(self):
        """Repack the fp32 parameters and the action noise into the kernel's layout.  Call after an update.

        If every parameter is a float32 contiguous CUDA tensor on this policy's device (``load_state_dict(sd, share=True)``),
        they are packed where they are, on ``torch.cuda.current_stream()``: no host copy, no device synchronisation and no
        allocation of device memory, so the call can be captured in ``torch.cuda.graph(...)`` along with the learner
        update and ``act``.  An act queued on that stream afterwards sees the new weights; one on another stream must be
        ordered by the caller (``wait_stream`` / events).  ``action_noise_std`` stays a host value: a captured graph keeps
        the noise it had at capture time.  Otherwise (CPU tensors, the default) the parameters are copied to the host and
        uploaded by the synchronising host entry."""
        params = [self.params[k] for k in squashed_param_shapes(self.obs_dim, self.act_dim)]
        noise = None
        if self.action_noise_std is not None:
            noise = torch.as_tensor(self.action_noise_std, dtype=torch.float32).flatten()
            noise = (noise.expand(self.act_dim) if noise.numel() == 1 else noise).contiguous()
            if noise.numel() != self.act_dim:
                raise ValueError("action_noise_std: a float or %d values expected" % self.act_dim)
        noise_ptr = None if noise is None else C.c_void_p(noise.data_ptr())
        if all(t.device == self.device and t.dtype == torch.float32 and t.is_contiguous() for t in params):
            _lib.check(self.lib.mvrl_policy_set_weights_squashed_device(self._h, *[C.c_void_p(t.data_ptr()) for t in params], noise_ptr,
                                                                        _lib.current_stream(self.device)))
            return
        host = [t.detach().to("cpu", torch.float32).contiguous() for t in params]
        _lib.check(self.lib.mvrl_policy_set_weights_squashed(self._h, *[C.c_void_p(t.data_ptr()) for t in host], noise_ptr))

    @property
    def logp_const(self):
        return -0.5 * self.act_dim * math.log(2.0 * math.pi)


MAX_CRITICS, MAX_QUANTILES = 5, 32
CRITIC_KINDS = {"sac": _lib.CRITIC_SAC, "tqc": _lib.CRITIC_TQC}


def critic_param_shapes(obs_dim, act_dim, n_critics, n_out):
    """SB3 names and shapes of the critics of a SAC ``ContinuousCritic`` / TQC ``Critic`` (``create_mlp`` with net_arch
    [128, 128, 128]: ``qf{i}.{0,2,4,6}``), in upload order; ``n_out`` is 1 for SAC and ``n_quantiles`` for TQC."""
    shapes = {}
    for i in range(n_critics):
        for j, (fan_out, fan_in) in zip((0, 2, 4, 6), ((HIDDEN, obs_dim + act_dim), (HIDDEN, HIDDEN), (HIDDEN, HIDDEN), (n_out, HIDDEN))):
            shapes["qf%d.%d.weight" % (i, j)], shapes["qf%d.%d.bias" % (i, j)] = (fan_out, fan_in), (fan_out,)
    return shapes


def critic_target_config(kind, n_critics, n_quantiles, top_quantiles_to_drop_per_net, obs_dim, act_dim):
    """The checks of ``CriticTarget``'s configuration -> (n_out per critic, drop per critic, n_target); ``ValueError``
    for anything the kernel does not take.  SAC ignores ``n_quantiles`` and ``top_quantiles_to_drop_per_net``."""
    if kind not in CRITIC_KINDS:
        raise ValueError("kind must be one of %s, got %r" % (sorted(CRITIC_KINDS), kind))
    if not 1 <= n_critics <= MAX_CRITICS:
        raise ValueError("n_critics must be 1..%d, got %d" % (MAX_CRITICS, n_critics))
    if obs_dim + act_dim > 16:
        raise ValueError("obs_dim + act_dim must be <= 16 (the critics' first layer is one K = 16 step), got %d + %d" % (obs_dim, act_dim))
    if kind == "sac":
        return 1, 0, 1
    if not 1 <= n_quantiles <= MAX_QUANTILES:
        raise ValueError("n_quantiles must be 1..%d, got %d" % (MAX_QUANTILES, n_quantiles))
    if not 0 <= top_quantiles_to_drop_per_net < n_quantiles:
        raise ValueError("top_quantiles_to_drop_per_net must be in [0, n_quantiles) to keep a quantile, got %d of %d"
                         % (top_quantiles_to_drop_per_net, n_quantiles))
    return n_quantiles, top_quantiles_to_drop_per_net, n_critics * (n_quantiles - top_quantiles_to_drop_per_net)


def _critic_tensors(sd, obs_dim, act_dim, n_critics, n_out, prefixes=("critic_target.", "critic."), detach=True):
    """The critic parameters of a critic / critic-target module state dict or of a whole SAC / TQC policy state dict
    (the keys under the first of ``prefixes`` present), as given (detached unless ``detach=False``); ``ValueError`` for a
    missing key, a shape other than [128, 128, 128] hidden with ``n_out`` outputs or another number of critics
    (obs_dim + act_dim <= 16 is ``critic_target_config``'s check)."""
    sd = _strip_prefix(sd, prefixes)
    found = {k.split(".")[0] for k in sd if k.startswith("qf") and k.split(".")[0][2:].isdigit()}
    if found != {"qf%d" % i for i in range(n_critics)}:
        raise ValueError("expected the %d critics qf0 .. qf%d, the state dict has %s" % (n_critics, n_critics - 1, sorted(found) or "none"))
    shapes = critic_param_shapes(obs_dim, act_dim, n_critics, n_out)
    extra = sorted(k for k in sd if k.startswith("qf") and k not in shapes)
    if extra:
        raise ValueError("critic layers beyond net_arch [128, 128, 128]: %s" % extra)
    out = {}
    for name, shape in shapes.items():
        if name not in sd:
            raise ValueError("critic state dict has no %r" % name)
        t = torch.as_tensor(sd[name])
        t = t.detach() if detach else t
        if tuple(t.shape) != shape:
            raise ValueError("%r has shape %s, expected %s (obs_dim %d + act_dim %d inputs, net_arch [128, 128, 128], %d outputs)"
                             % (name, tuple(t.shape), shape, obs_dim, act_dim, n_out))
        out[name] = t
    return out


class CriticTarget(_lib.Handle):
    """The critic target of SB3 SAC / sb3_contrib TQC for one gradient step, as one fp32 tensor-core kernel
    (``mvrl_critic_target``): on a replay sample, under SB3's ``th.no_grad()`` block,

        next_actions, next_log_prob = actor.action_log_prob(next_observations)
        q = critic_target(next_observations, next_actions)              # [B, n_critics, n_quantiles]; SAC [B, n_critics]
        TQC: q = sort(q.reshape(B, -1))[:, :n_critics * (n_quantiles - top_quantiles_to_drop_per_net)]
        SAC: q = min over the critics, [B, 1]
        target = rewards + (1 - dones) * gamma * (q - ent_coef * next_log_prob)

    ``actor`` is a ``SquashedGaussianPolicy(precision="fp32")`` on the same device; its packed fp32 parameters are read by
    the kernel, so ``actor.sync_weights()`` after the actor's optimiser step updates both the collection of that handle
    and the next action here.  The critics are ``n_critics`` [128, 128, 128] GELU MLPs on ``[next_obs, action]`` with SB3's
    key names (``load_state_dict``); ``sync_weights()`` repacks them after the Polyak update.  Everything is in fp32 as SB3
    evaluates it (split-bf16 tensor-core products, erf GELU); the gradient steps, optimisers and the Polyak update stay
    with the learner.

    ``eps`` of the next action comes from Philox4x32-10 stream 10 keyed on (``seed``, sampled row, call number); the call
    number is the device counter ``calls`` (int64 [2]: the count and a block ticket that is 0 between launches), so a CUDA
    graph of T calls replayed R times draws like T * R eager calls.  ``kind="sac"`` ignores ``n_quantiles`` and
    ``top_quantiles_to_drop_per_net``.  Limits: obs_dim + act_dim <= 16, n_critics 1..5, n_quantiles 1..32."""

    def __init__(self, actor, kind="tqc", n_critics=2, n_quantiles=25, top_quantiles_to_drop_per_net=2, gamma=0.99, seed=0):
        if not isinstance(actor, SquashedGaussianPolicy) or getattr(actor, "precision", None) != "fp32":
            raise ValueError("actor must be a SquashedGaussianPolicy with precision='fp32', got %r" % (actor,))
        self.actor, self.kind = actor, kind
        self.obs_dim, self.act_dim, self.device = actor.obs_dim, actor.act_dim, actor.device
        self.n_critics = int(n_critics)
        self.n_out, self.drop, self.n_target = critic_target_config(kind, self.n_critics, int(n_quantiles), int(top_quantiles_to_drop_per_net),
                                                                    self.obs_dim, self.act_dim)
        self.n_quantiles = self.n_out
        self.gamma, self.seed = float(gamma), int(seed)
        super().__init__("mvrl_critic", self.device.index, self.obs_dim, self.act_dim, CRITIC_KINDS[kind], self.n_critics, self.n_out)
        self.calls = torch.zeros(2, dtype=torch.int64, device=self.device)
        self._ent_coef = torch.zeros(1, dtype=torch.float32, device=self.device)
        g = torch.Generator().manual_seed(self.seed)
        self.params = {}
        for name, shape in critic_param_shapes(self.obs_dim, self.act_dim, self.n_critics, self.n_out).items():
            t = torch.randn(shape, generator=g) / math.sqrt(shape[1]) if len(shape) == 2 else torch.zeros(shape)
            self.params[name] = t.to(self.device)
        self.sync_weights()

    def state_dict(self):
        """{SB3 critic name: fp32 tensor} and ``calls`` (copies)."""
        d = {k: v.detach().clone() for k, v in self.params.items()}
        d["calls"] = self.calls.clone()
        return d

    def load_state_dict(self, sd, share=False):
        """Take the critics of a critic / critic-target state dict (keys ``qf{i}.{0,2,4,6}.{weight,bias}``) or of a whole
        SAC / TQC policy state dict (``critic_target.*`` if present, else ``critic.*``) and pack them; a ``calls`` entry
        (from ``state_dict()``) is copied into the counter.  ``share=False`` keeps fp32 copies on this device.
        ``share=True`` keeps REFERENCES, e.g. to ``agent.critic_target.state_dict()``: the Polyak update in place is then
        seen by the next ``sync_weights()``; every tensor must be float32, contiguous and on this device, else
        ``ValueError``."""
        params = _critic_tensors(sd, self.obs_dim, self.act_dim, self.n_critics, self.n_out)
        if share:
            self.params = _check_shared(params, self.device)
        else:
            self.params = {k: t.to(self.device, torch.float32).clone().contiguous() for k, t in params.items()}
        if "calls" in sd:
            calls = torch.as_tensor(sd["calls"]).reshape(-1)
            if calls.numel() != 2 or int(calls[0]) < 0 or int(calls[1]) != 0:
                raise ValueError("calls must be [call number >= 0, 0], got %s" % calls.tolist())
            self.calls.copy_(calls)
        self.sync_weights()
        return self

    def sync_weights(self):
        """Pack the critic parameters on ``torch.cuda.current_stream()``: no host copy, no synchronisation, capturable in a
        CUDA graph with the learner update; a call queued on the same stream afterwards sees the new weights."""
        params = list(self.params[k] for k in critic_param_shapes(self.obs_dim, self.act_dim, self.n_critics, self.n_out))
        arr = (C.c_void_p * len(params))(*[t.data_ptr() for t in params])
        _lib.check(self.lib.mvrl_critic_set_weights_device(self._h, arr, _lib.current_stream(self.device)))

    def __call__(self, batch, ent_coef, next_actions=None, next_log_prob=None, eps=None):
        """The target of a ``ReplayBufferSamples`` (float32; ``next_observations``, ``rewards``, ``dones`` are read):
        ``[B, n_target]`` sorted ascending (TQC) or ``[B, 1]`` (SAC), a new tensor.  ``ent_coef``: a float, or a 1-element
        float32 tensor on this device read by the kernel (e.g. ``log_ent_coef.exp()``).  Optional outputs ``next_actions``
        / ``eps`` ``[B, act_dim]`` and ``next_log_prob`` ``[B]`` (float32, contiguous).  One launch on the current stream."""
        obs, rew, done = batch.next_observations, batch.rewards, batch.dones
        b = int(obs.shape[0]) if obs.dim() == 2 else -1
        for name, t, shape in (("next_observations", obs, (b, self.obs_dim)), ("rewards", rew, (b, 1)), ("dones", done, (b, 1))):
            if t.dtype != torch.float32:
                raise ValueError("%s must be float32 (cast the batch of an fp64 env), got %s" % (name, t.dtype))
            if t.device != self.device or tuple(t.reshape(-1, shape[1]).shape) != shape or b < 1:
                raise ValueError("%s: [%d, %d] on %s expected, got %s on %s" % (name, b, shape[1], self.device, tuple(t.shape), t.device))
        if isinstance(ent_coef, torch.Tensor):
            if ent_coef.dtype != torch.float32 or ent_coef.numel() != 1 or ent_coef.device != self.device:
                raise ValueError("ent_coef: a float or a 1-element float32 tensor on %s, got %s %s on %s"
                                 % (self.device, ent_coef.dtype, tuple(ent_coef.shape), ent_coef.device))
            alpha = ent_coef.reshape(1).contiguous()
        else:
            alpha = self._ent_coef.fill_(float(ent_coef))
        for name, t, shape in (("next_actions", next_actions, (b, self.act_dim)), ("eps", eps, (b, self.act_dim)), ("next_log_prob", next_log_prob, (b,))):
            if t is not None and (t.dtype != torch.float32 or t.device != self.device or tuple(t.shape) != shape or not t.is_contiguous()):
                raise ValueError("%s: contiguous float32 %s on %s expected" % (name, list(shape), self.device))
        out = torch.empty((b, self.n_target), dtype=torch.float32, device=self.device)
        _lib.check(self.lib.mvrl_critic_target(
            self._h, self.actor._h, b, _lib.ptr(obs.contiguous()), _lib.ptr(rew.contiguous()), _lib.ptr(done.contiguous()), _lib.ptr(alpha),
            self.gamma, self.drop, self.seed & (2 ** 64 - 1), _lib.ptr(self.calls), _lib.ptr(out), _lib.ptr(next_actions),
            _lib.ptr(next_log_prob), _lib.ptr(eps), _lib.current_stream(self.device)))
        return out


_SB3_LOSS = "sb3_contrib.common.utils.quantile_huber_loss"


def _quantile_loss_shapes(current, target, cum_prob):
    """The checks of ``quantile_huber_loss`` decided from the tensors' metadata -> (B, n_critics, n_quantiles, n_target);
    ``ValueError`` for anything the kernel does not take."""
    if cum_prob is not None:
        raise ValueError("cum_prob: only the default (i + 0.5) / n_quantiles is computed here; use %s for another" % _SB3_LOSS)
    for name, t in (("current_quantiles", current), ("target_quantiles", target)):
        if not isinstance(t, torch.Tensor) or t.dtype != torch.float32:
            raise ValueError("%s must be a float32 tensor, got %s" % (name, getattr(t, "dtype", type(t).__name__)))
    if current.dim() not in (2, 3) or target.dim() != current.dim():
        raise ValueError("current_quantiles and target_quantiles must both be 2-D ([B, n_quantiles], [B, n_target]) or 3-D "
                         "([B, n_critics, n_quantiles], [B, 1, n_target]), got %s and %s" % (tuple(current.shape), tuple(target.shape)))
    if current.shape[0] != target.shape[0] or current.shape[0] < 1:
        raise ValueError("current_quantiles and target_quantiles need the same batch size >= 1, got %s and %s"
                         % (tuple(current.shape), tuple(target.shape)))
    if current.dim() == 3 and target.shape[1] != 1:
        raise ValueError("a 3-D target_quantiles must be [B, 1, n_target] (one target shared by the critics), got %s; use %s "
                         "for per-critic targets" % (tuple(target.shape), _SB3_LOSS))
    if target.requires_grad:
        raise ValueError("target_quantiles requires grad: the gradient is computed for current_quantiles only (detach the "
                         "target, as TQC computes it under th.no_grad(), or use %s)" % _SB3_LOSS)
    b, nq, t = int(current.shape[0]), int(current.shape[-1]), int(target.shape[-1])
    c = int(current.shape[1]) if current.dim() == 3 else 1
    if min(c, nq, t) < 1:
        raise ValueError("empty quantile dimension: current_quantiles %s, target_quantiles %s" % (tuple(current.shape), tuple(target.shape)))
    return b, c, nq, t


class _QuantileHuberLoss(torch.autograd.Function):
    """Forward: one ``mvrl_quantile_huber_loss`` call, which also writes d loss / d current when ``with_grad``; backward:
    that gradient times the incoming scalar."""

    @staticmethod
    def forward(ctx, current, target, dims, sum_over_quantiles, with_grad):
        b, c, nq, t = dims
        lib = _lib.load()
        dev = current.device
        cur, tgt = current.detach().contiguous(), target.detach().contiguous()
        loss = torch.empty((), dtype=torch.float32, device=dev)
        grad = torch.empty_like(cur) if with_grad else None
        scratch = torch.empty(int(lib.mvrl_quantile_huber_scratch(b * c * nq)), dtype=torch.uint8, device=dev)
        _lib.check(lib.mvrl_quantile_huber_loss(b, c, nq, t, _lib.ptr(cur), _lib.ptr(tgt), int(bool(sum_over_quantiles)),
                                                _lib.ptr(loss), _lib.ptr(grad), _lib.ptr(scratch), _lib.current_stream(dev)))
        if grad is not None:
            ctx.save_for_backward(grad.view(current.shape))
        return loss

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, grad_output):
        (grad,) = ctx.saved_tensors
        return grad_output * grad, None, None, None, None


def quantile_huber_loss(current_quantiles, target_quantiles, cum_prob=None, sum_over_quantiles=True):
    """sb3_contrib's ``quantile_huber_loss`` (``common/utils.py``) as one fused kernel with its gradient: the loss TQC's
    critic update calls as ``quantile_huber_loss(current_quantiles, target_quantiles, sum_over_quantiles=False)``.

    ``current_quantiles`` ``[B, n_critics, n_quantiles]`` (QR-DQN: ``[B, n_quantiles]``), ``target_quantiles`` ``[B, 1,
    n_target]`` (QR-DQN: ``[B, n_target]``), float32 on one CUDA device; non-contiguous inputs are copied.  Returns a 0-dim
    float32 tensor, with a ``grad_fn`` when ``current_quantiles`` requires grad under grad mode: the forward launch then
    also writes d loss / d current_quantiles, and ``backward`` scales it by the incoming gradient (no double backward).
    The same inputs give the same bits (fixed-order sums, no atomics); the call allocates its outputs on the current
    stream and does not synchronise, so it can be captured in a CUDA graph with the rest of the learner step.

    ``ValueError`` for what sb3_contrib accepts but no TQC / QR-DQN caller passes - a ``cum_prob``, per-critic targets
    ``[B, n_critics, n_target]``, a target that requires grad - and for another dtype, mismatched shapes or devices."""
    dims = _quantile_loss_shapes(current_quantiles, target_quantiles, cum_prob)
    _lib.require_cuda()
    dev = current_quantiles.device
    if dev.type != "cuda" or target_quantiles.device != dev:
        raise ValueError("current_quantiles and target_quantiles must be on the same CUDA device, got %s and %s"
                         % (dev, target_quantiles.device))
    with_grad = current_quantiles.requires_grad and torch.is_grad_enabled()
    return _QuantileHuberLoss.apply(current_quantiles, target_quantiles, dims, bool(sum_over_quantiles), with_grad)


class _CriticFn(torch.autograd.Function):
    """Forward: one ``mvrl_critic_forward`` launch, which also stores the pre-activations when a gradient will be needed;
    backward: ``mvrl_critic_backward`` for what autograd asks (weight gradients, the action gradient, or both).  The
    parameters are inputs saved for backward, so an in-place change between the two passes raises torch's version error
    (the packed block the backward pass reads is a function of them)."""

    @staticmethod
    def forward(ctx, critic, want_grad, obs, actions, *params):
        b = obs.shape[0]
        dev = obs.device
        lib = critic.lib
        q = torch.empty((b, critic.n_critics, critic.n_out), dtype=torch.float32, device=dev)
        saved = torch.empty(int(lib.mvrl_critic_saved_bytes(critic._h, b)), dtype=torch.uint8, device=dev) if want_grad else None
        _lib.check(lib.mvrl_critic_forward(critic._h, b, _lib.ptr(obs), _lib.ptr(actions), _lib.ptr(q), _lib.ptr(saved),
                                           _lib.current_stream(dev)))
        if want_grad:
            ctx.critic, ctx.workspace = critic, saved
            ctx.save_for_backward(obs, actions, *params)
        return q

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, grad_q):
        obs, actions, *params = ctx.saved_tensors
        critic = ctx.critic
        lib, dev, b = critic.lib, obs.device, obs.shape[0]
        need_act, need_w = ctx.needs_input_grad[3], any(ctx.needs_input_grad[4:])
        grad_q = grad_q.contiguous()
        grads = [torch.empty_like(p) for p in params] if need_w else None
        grad_act = torch.empty_like(actions) if need_act else None
        scratch = torch.empty(int(lib.mvrl_critic_grad_scratch(critic._h, b)), dtype=torch.uint8, device=dev)
        arr = (C.c_void_p * len(params))(*[g.data_ptr() for g in grads]) if need_w else None
        _lib.check(lib.mvrl_critic_backward(critic._h, b, _lib.ptr(obs), _lib.ptr(actions), _lib.ptr(ctx.workspace), _lib.ptr(grad_q),
                                            arr, _lib.ptr(grad_act), _lib.ptr(scratch), _lib.current_stream(dev)))
        ctx.workspace = None
        gp = [g if n else None for g, n in zip(grads, ctx.needs_input_grad[4:])] if need_w else [None] * len(params)
        return (None, None, None, grad_act, *gp)


class Critic(_lib.Handle):
    """The critics of SB3 SAC (``ContinuousCritic``) / sb3_contrib TQC (``Critic``): ``n_critics`` [128, 128, 128] GELU MLPs
    on ``[obs, actions]`` (``qf{i}.{0,2,4,6}``), evaluated by the library on the learner's own parameters, with a backward
    pass that reaches those parameters' ``.grad`` and the actions:

        critic = Critic(agent.critic, obs_dim, act_dim, kind="tqc", n_critics=2, n_quantiles=25)
        q = critic(batch.observations, batch.actions)        # TQC: [B, n_critics, n_quantiles]; SAC: n_critics tensors [B, 1]
        loss = quantile_huber_loss(q, target.unsqueeze(1), sum_over_quantiles=False)
        agent.critic.optimizer.zero_grad(); loss.backward(); agent.critic.optimizer.step()

    ``params``: a module (its ``named_parameters()``, an optional ``critic.`` prefix stripped) or a {name: Parameter}
    mapping.  References to the tensors themselves are kept, never copies: float32, contiguous, on one CUDA device.  Every
    call packs the current parameters first (``mvrl_critic_set_weights_device`` on the current stream), so it sees each
    ``optimizer.step()`` and can be captured in a CUDA graph with the whole update.  The backward pass computes the weight
    gradients only if a parameter requires grad and the action gradient only if ``actions`` does (the actor loss's
    ``critic(obs, actions_pi)``); under ``no_grad`` nothing is saved.  Everything is fp32 as SB3 computes it (split-bf16
    tensor-core products, erf GELU; DESIGN.md K12); the same inputs give the same bits.  All memory is allocated by torch
    on the current stream; nothing synchronises.  Limits: obs_dim + act_dim <= 16, n_critics 1..5, n_quantiles 1..32."""

    def __init__(self, params, obs_dim, act_dim, kind="tqc", n_critics=2, n_quantiles=25):
        self.obs_dim, self.act_dim, self.kind, self.n_critics = int(obs_dim), int(act_dim), kind, int(n_critics)
        self.n_out = critic_target_config(kind, self.n_critics, int(n_quantiles), 0, self.obs_dim, self.act_dim)[0]
        named = dict(params.named_parameters()) if isinstance(params, torch.nn.Module) else dict(params)
        tensors = _critic_tensors(named, self.obs_dim, self.act_dim, self.n_critics, self.n_out, prefixes=("critic.",), detach=False)
        first = next(iter(tensors.values()))
        if first.device.type != "cuda":
            raise ValueError("the critic parameters must be on a CUDA device, got %s" % first.device)
        self.device = first.device
        self.params = _check_shared(tensors, self.device)
        self._order = list(critic_param_shapes(self.obs_dim, self.act_dim, self.n_critics, self.n_out))
        super().__init__("mvrl_critic", self.device.index, self.obs_dim, self.act_dim, CRITIC_KINDS[kind], self.n_critics, self.n_out)

    def _check_inputs(self, obs, actions):
        for name, t, width in (("obs", obs, self.obs_dim), ("actions", actions, self.act_dim)):
            if not isinstance(t, torch.Tensor) or t.dtype != torch.float32:
                raise ValueError("%s must be a float32 tensor (cast the batch of an fp64 env), got %s" % (name, getattr(t, "dtype", type(t).__name__)))
            if t.device != self.device:
                raise ValueError("%s is on %s, the critic parameters on %s" % (name, t.device, self.device))
            if t.dim() != 2 or t.shape[1] != width:
                raise ValueError("%s: [B, %d] expected, got %s" % (name, width, tuple(t.shape)))
        if obs.shape[0] != actions.shape[0] or obs.shape[0] < 1:
            raise ValueError("obs and actions need the same batch size >= 1, got %s and %s" % (tuple(obs.shape), tuple(actions.shape)))
        if obs.requires_grad:
            raise ValueError("obs requires grad: the gradient is computed for the parameters and the actions only (detach the "
                             "observations, or use the PyTorch critic for d q / d obs)")

    def __call__(self, obs, actions):
        """``q`` of the batch: ``[B, n_critics, n_quantiles]`` for TQC, a tuple of ``n_critics`` ``[B, 1]`` for SAC
        (``ContinuousCritic.forward``).  ``obs`` and ``actions`` float32 ``[B, obs_dim]`` / ``[B, act_dim]`` on the
        parameters' device; non-contiguous inputs are copied."""
        self._check_inputs(obs, actions)
        params = [self.params[k] for k in self._order]
        arr = (C.c_void_p * len(params))(*[t.data_ptr() for t in params])
        _lib.check(self.lib.mvrl_critic_set_weights_device(self._h, arr, _lib.current_stream(self.device)))
        want_grad = torch.is_grad_enabled() and (actions.requires_grad or any(p.requires_grad for p in params))
        q = _CriticFn.apply(self, want_grad, obs.contiguous(), actions.contiguous(), *params)
        if self.kind == "sac":
            return tuple(q[:, i] for i in range(self.n_critics))
        return q


class _ActorFn(torch.autograd.Function):
    """Forward: one ``mvrl_actor_forward`` launch, which also stores what the backward pass reads when a gradient will be
    needed; backward: ``mvrl_actor_backward`` from the gradients of either or both outputs.  The parameters are inputs
    saved for backward, so an in-place change between the two passes raises torch's version error."""

    @staticmethod
    def forward(ctx, actor, want_grad, eps_out, obs, *params):
        ctx.set_materialize_grads(False)
        b, dev = obs.shape[0], obs.device
        lib = actor.lib
        actions = torch.empty((b, actor.act_dim), dtype=torch.float32, device=dev)
        log_prob = torch.empty((b,), dtype=torch.float32, device=dev)
        saved = torch.empty(int(lib.mvrl_actor_saved_bytes(actor._policy._h, b)), dtype=torch.uint8, device=dev) if want_grad else None
        _lib.check(lib.mvrl_actor_forward(actor._policy._h, b, _lib.ptr(obs), _lib.ptr(actions), _lib.ptr(log_prob), _lib.ptr(eps_out[0]),
                                          _lib.ptr(saved), actor.seed & (2 ** 64 - 1), _lib.ptr(actor.calls), _lib.current_stream(dev)))
        if want_grad:
            ctx.actor, ctx.workspace = actor, saved
            ctx.save_for_backward(obs, *params)
        return actions, log_prob

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, grad_actions, grad_log_prob):
        obs, *params = ctx.saved_tensors
        needs = ctx.needs_input_grad[4:]
        if (grad_actions is None and grad_log_prob is None) or not any(needs):
            return (None,) * (4 + len(params))
        actor = ctx.actor
        lib, dev, b = actor.lib, obs.device, obs.shape[0]
        grads = [torch.empty_like(p) for p in params]
        scratch = torch.empty(int(lib.mvrl_actor_grad_scratch(actor._policy._h, b)), dtype=torch.uint8, device=dev)
        arr = (C.c_void_p * len(grads))(*[g.data_ptr() for g in grads])
        ga = None if grad_actions is None else grad_actions.contiguous()
        gl = None if grad_log_prob is None else grad_log_prob.contiguous()
        _lib.check(lib.mvrl_actor_backward(actor._policy._h, b, _lib.ptr(obs), _lib.ptr(ctx.workspace), _lib.ptr(ga), _lib.ptr(gl), arr,
                                           _lib.ptr(scratch), _lib.current_stream(dev)))
        ctx.workspace = None
        return (None, None, None, None, *[g if n else None for g, n in zip(grads, needs)])


class Actor:
    """The actor of SB3 SAC / sb3_contrib TQC (``Actor``, net_arch [128, 128, 128], GELU, no gSDE) in the learner's gradient
    step, evaluated by the library on the learner's own parameters, with a backward pass that reaches those parameters'
    ``.grad``:

        actor = Actor(agent.actor, obs_dim, act_dim)
        actions_pi, log_prob = actor.action_log_prob(batch.observations)
        q = critic(batch.observations, actions_pi)              # Critic: TQC [B, n_critics, n_quantiles]
        actor_loss = (ent_coef * log_prob - q.mean(2).mean(1, keepdim=True)).mean()
        agent.actor.optimizer.zero_grad(); actor_loss.backward(); agent.actor.optimizer.step()

    ``params``: a module (its ``named_parameters()``, an optional ``actor.`` prefix stripped, so ``agent.policy`` works too)
    or a {name: Parameter} mapping under SB3's names.  References to the tensors themselves are kept, never copies: float32,
    contiguous, on one CUDA device.  Every call packs the current parameters first, on the current stream, into an
    internal fp32 ``SquashedGaussianPolicy`` handle, so it sees each ``optimizer.step()`` and can be captured in a CUDA
    graph with the whole gradient step.  ``eps`` is drawn from Philox4x32-10 stream 11 keyed on (``seed``, row, call
    number); ``calls`` is the int64 [2] device counter (call number, block ticket), so a graph of T calls replayed R times
    draws like T * R eager calls.  Everything is fp32 as SB3 computes it (split-bf16 tensor-core products, erf GELU;
    DESIGN.md K13); the same inputs and call number give the same bits.  All memory is allocated by torch on the current
    stream; nothing synchronises.  Limits: obs_dim <= 16, act_dim <= 8.  This actor's packed block is its own: a
    ``CriticTarget``'s actor handle still needs its ``sync_weights()`` after the actor's optimiser step."""

    def __init__(self, params, obs_dim, act_dim, seed=0):
        self.obs_dim, self.act_dim, self.seed = int(obs_dim), int(act_dim), int(seed)
        if not (1 <= self.obs_dim <= 16 and 1 <= self.act_dim <= 8):
            raise ValueError("Actor needs 1 <= obs_dim <= 16 and 1 <= act_dim <= 8 (one K = 16 step, one head tile), got %d, %d"
                             % (self.obs_dim, self.act_dim))
        named = dict(params.named_parameters()) if isinstance(params, torch.nn.Module) else dict(params)
        tensors = _actor_tensors(named, self.obs_dim, self.act_dim, detach=False)
        first = next(iter(tensors.values()))
        if first.device.type != "cuda":
            raise ValueError("the actor parameters must be on a CUDA device, got %s" % first.device)
        self.device = first.device
        self.params = _check_shared(tensors, self.device)
        self._order = list(squashed_param_shapes(self.obs_dim, self.act_dim))
        self._policy = SquashedGaussianPolicy(self.obs_dim, self.act_dim, device=self.device, seed=self.seed, precision="fp32")
        self._policy.load_state_dict(self.params, share=True)
        self.lib = self._policy.lib
        self.calls = torch.zeros(2, dtype=torch.int64, device=self.device)

    def action_log_prob(self, obs, eps=None):
        """SB3's ``actor.action_log_prob(obs)``: ``(actions [B, act_dim], log_prob [B])``, new tensors with a ``grad_fn``
        when a parameter requires grad under grad mode.  ``obs`` float32 ``[B, obs_dim]`` on the parameters' device (copied
        if non-contiguous; it must not require grad: no gradient with respect to obs is computed).  ``eps`` (optional):
        a contiguous float32 ``[B, act_dim]`` tensor that receives the standard normals of the draw."""
        if not isinstance(obs, torch.Tensor) or obs.dtype != torch.float32:
            raise ValueError("obs must be a float32 tensor (cast the batch of an fp64 env), got %s" % getattr(obs, "dtype", type(obs).__name__))
        if obs.device != self.device:
            raise ValueError("obs is on %s, the actor parameters on %s" % (obs.device, self.device))
        if obs.dim() != 2 or obs.shape[1] != self.obs_dim or obs.shape[0] < 1:
            raise ValueError("obs: [B, %d] with B >= 1 expected, got %s" % (self.obs_dim, tuple(obs.shape)))
        if obs.requires_grad:
            raise ValueError("obs requires grad: the gradient is computed for the actor parameters only (detach the observations)")
        b = int(obs.shape[0])
        if eps is not None and (eps.dtype != torch.float32 or eps.device != self.device or tuple(eps.shape) != (b, self.act_dim)
                                or not eps.is_contiguous()):
            raise ValueError("eps: contiguous float32 [%d, %d] on %s expected" % (b, self.act_dim, self.device))
        params = [self.params[k] for k in self._order]
        self._policy.sync_weights()
        want_grad = torch.is_grad_enabled() and any(p.requires_grad for p in params)
        return _ActorFn.apply(self, want_grad, (eps,), obs.contiguous(), *params)
