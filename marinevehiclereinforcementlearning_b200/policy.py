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
synchronisation, and can be captured in a CUDA graph.  The learner side (losses, optimiser) is out of scope, like in
SURVEY.md 8(e)."""
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


class _FusedActor:
    """The plumbing both heads share: the library handle, sampling into feature-major buffers, SB3 ``predict``."""

    def _open(self, device, obs_dim, act_dim, seed, head):
        self.device = torch.device("cuda", _device_index(device))
        self.obs_dim, self.act_dim, self.seed = int(obs_dim), int(act_dim), int(seed)
        self.step = 0
        self.lib = _lib.load()
        _lib.require_cuda()
        self._h = C.c_void_p()
        _lib.check(self.lib.mvrl_policy_create_ex(C.byref(self._h), self.device.index, self.obs_dim, self.act_dim, head,
                                                  PRECISIONS[self.precision]))

    def __del__(self):
        h = getattr(self, "_h", None)
        if h:
            try:
                self.lib.mvrl_policy_destroy(h)
            except Exception:
                pass
            self._h = None

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


def _actor_tensors(sd, obs_dim, act_dim):
    """The checks of ``actor_params_from_state_dict``; the tensors as given (detached: they share storage with ``sd``'s)."""
    keys = list(sd.keys())
    if any(k.startswith("actor.") for k in keys):
        sd = {k[len("actor."):]: sd[k] for k in keys if k.startswith("actor.")}
    if "log_std" in sd:
        raise ValueError("the state dict is of a gSDE actor (use_sde=True: log_std is a Parameter, not a Linear layer); "
                         "gSDE is not supported")
    out = {}
    for name, shape in squashed_param_shapes(obs_dim, act_dim).items():
        if name not in sd:
            raise ValueError("actor state dict has no %r" % name)
        t = torch.as_tensor(sd[name]).detach()
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
            params = _actor_tensors(sd, self.obs_dim, self.act_dim)
            for name, t in params.items():
                if t.dtype != torch.float32 or not t.is_contiguous() or t.device != self.device:
                    raise ValueError("share=True needs float32 contiguous tensors on %s; %r is %s%s on %s"
                                     % (self.device, name, t.dtype, "" if t.is_contiguous() else " (non-contiguous)", t.device))
            self.params = params
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
