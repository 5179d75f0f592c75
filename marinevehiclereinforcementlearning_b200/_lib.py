"""ctypes binding of libmvrl.so (C ABI declared in include/mvrl.h).

There is deliberately no CPU implementation behind this module: if the shared
library is missing, or no CUDA device is present, every compute entry point
raises ``RuntimeError``.
"""
import ctypes as C
import os
import subprocess

_PKG_DIR = os.path.dirname(os.path.abspath(__file__))
# MVRL_LIB selects an alternative build of the same sources (kernel-tuning experiments)
LIB_PATH = os.environ.get("MVRL_LIB") or os.path.join(_PKG_DIR, "libmvrl.so")
CSRC_DIR = os.path.join(_PKG_DIR, "csrc")

F32, F64 = 0, 1
ACT_RPM, ACT_FORCE, ACT_SETPOINT = 0, 1, 2

_d = C.c_double


class MvrlRov6Params(C.Structure):
    _fields_ = [
        ("rho_f", _d), ("m", _d), ("Length", _d),
        ("CG", _d * 3), ("CB", _d * 3), ("I", _d * 9),
        ("Xudot", _d), ("Yvdot", _d), ("Zwdot", _d), ("Kpdot", _d), ("Mqdot", _d), ("Nrdot", _d),
        ("Xu", _d), ("Yv", _d), ("Yp", _d), ("Yr", _d), ("Zw", _d), ("Zq", _d), ("Kv", _d),
        ("Kp", _d), ("Kr", _d), ("Mw", _d), ("Mq", _d), ("Nv", _d), ("Np", _d), ("Nr", _d),
        ("Xuu", _d), ("Yvv", _d), ("Ypp", _d), ("Yrr", _d), ("Zww", _d), ("Zqq", _d), ("Kvv", _d),
        ("Kpp", _d), ("Krr", _d), ("Mww", _d), ("Mqq", _d), ("Nvv", _d), ("Npp", _d), ("Nrr", _d),
        ("W", _d), ("B", _d), ("thrust_coef", _d), ("rpm_max", _d), ("rpm_deadband", _d),
        ("M", _d * 36), ("Minv", _d * 36), ("A", _d * 48), ("Ainv", _d * 48),
        ("pid_Kp", _d * 6), ("pid_Ki", _d * 6), ("pid_Kd", _d * 6), ("pid_windup", _d * 6), ("pid_max", _d * 6),
        ("disable_thrusters", C.c_int),
    ]


class MvrlRov6Config(C.Structure):
    _fields_ = [
        ("dtype", C.c_int), ("action_mode", C.c_int), ("n_sub", C.c_int), ("max_steps", C.c_int),
        ("dt", _d), ("seed", C.c_uint64), ("env_id0", C.c_uint64),
        ("auto_reset", C.c_int), ("fixed_sp", C.c_int), ("device", C.c_int), ("fast_math", C.c_int),
    ]


class MvrlRov6Buffers(C.Structure):
    _fields_ = [
        ("state", C.c_void_p), ("action", C.c_void_p), ("obs", C.c_void_p), ("reward", C.c_void_p),
        ("done", C.c_void_p), ("istep", C.c_void_p), ("setpoint", C.c_void_p), ("path", C.c_void_p),
        ("ctrl", C.c_void_p), ("episode", C.c_void_p), ("terminal_obs", C.c_void_p), ("aux", C.c_void_p),
        ("ep_stats", C.c_void_p),
    ]


class MvrlRov3Params(C.Structure):
    _fields_ = [(n, _d) for n in ("rho_f", "m", "Length", "dispVol", "xg", "yg", "Izz", "Xudot", "Yvdot", "Nrdot",
                                  "Xu", "Yv", "Yr", "Nv", "Nr", "Xuu", "Yvv", "Yrr", "Nvv", "Nrr",
                                  "D_thruster", "thrust_coef", "alphaThruster", "l_x", "l_y", "rpm_max", "rpm_deadband")] + \
        [("M", _d * 9), ("Minv", _d * 9), ("Ainv", _d * 12),
         ("pid_Kp", _d * 3), ("pid_Ki", _d * 3), ("pid_Kd", _d * 3), ("pid_windup", _d * 3), ("pid_max", _d * 3)]


MvrlRov3Config = MvrlRov6Config
MvrlRov3Buffers = MvrlRov6Buffers  # same members, different leading dimensions per array


AUV_PLAIN, AUV_CYL = 0, 1


class MvrlAuvParams(C.Structure):
    _fields_ = [(n, _d) for n in ("m", "Izz", "Xuu", "Yvv", "Nrr", "Xu", "Yv", "Nr", "maxForce", "maxMoment",
                                  "xMin", "xMax", "yMin", "yMax", "noiseMagCoeffs", "noiseMagActuation", "wp_threshold")] + \
        [("waypoints", _d * 96), ("variant", C.c_int), ("n_waypoints", C.c_int)]


class MvrlAuvConfig(C.Structure):
    _fields_ = [("dtype", C.c_int), ("max_steps", C.c_int), ("dt", _d), ("seed", C.c_uint64), ("env_id0", C.c_uint64),
                ("auto_reset", C.c_int), ("stop_on_bounds", C.c_int), ("apply_noise", C.c_int), ("device", C.c_int)]


class MvrlAuvBuffers(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in ("state", "action", "obs", "reward", "done", "istep", "mults", "target", "err_o",
                                          "recent", "ep_return", "iwp", "episode", "terminal_obs", "aux", "ep_stats")]


REPLAY_MAX_DIM = 16


class MvrlReplayStorage(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in ("observations", "next_observations", "actions", "rewards", "dones", "timeouts",
                                          "last_obs", "cursor")]


_vp, _i64, _int = C.c_void_p, C.c_int64, C.c_int

# name -> (restype, argtypes); every symbol include/mvrl.h declares
PROTOTYPES = {
    "mvrl_version": (_int, []),
    "mvrl_last_error": (C.c_char_p, []),
    "mvrl_device_count": (_int, []),
    "mvrl_rov6_default_params": (_int, [C.POINTER(MvrlRov6Params)]),
    "mvrl_rov6_create": (_int, [C.POINTER(_vp), C.POINTER(MvrlRov6Params), C.POINTER(MvrlRov6Config)]),
    "mvrl_rov6_destroy": (_int, [_vp]),
    "mvrl_rov6_is_specialised": (_int, [_vp]),
    "mvrl_rov6_dev_constants_f32": (_int, [C.POINTER(MvrlRov6Params), C.POINTER(C.c_float), _int]),
    "mvrl_rov6_derivs": (_int, [_vp, _i64, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "mvrl_rov6_step": (_int, [_vp, _i64, _i64, C.POINTER(MvrlRov6Buffers), _vp]),
    "mvrl_rov6_step_range": (_int, [_vp, _i64, _i64, _i64, C.POINTER(MvrlRov6Buffers), _vp]),
    "mvrl_host_chunk_count": (_int, [_i64, _int]),
    "mvrl_rov6_step_host": (_int, [_vp, _i64, _i64, C.POINTER(MvrlRov6Buffers), _vp, _vp, _vp, _vp, _int, _vp]),
    "mvrl_rov6_reset": (_int, [_vp, _i64, _i64, C.POINTER(MvrlRov6Buffers), _vp, C.POINTER(_d), _vp]),
    "mvrl_rov6_pid": (_int, [_vp, _i64, _i64, _vp, _vp, _vp, _vp, _vp, _vp]),
    "mvrl_coordinate_transform": (_int, [_int, _int, _i64, _i64, _vp, _vp, _vp, _vp, _vp]),
    "mvrl_angle_error": (_int, [_int, _i64, _vp, _vp, _vp, _vp]),
    "mvrl_body_axes": (_int, [_int, _i64, _i64, _vp, _vp, _vp]),
    "mvrl_measure_fma_peak": (_int, [_int, _int, _int, C.POINTER(_d), C.POINTER(_d)]),
    "mvrl_rov6_thruster_model": (_int, [_vp, _i64, _vp, _vp, _vp]),
    "mvrl_frame_rotate": (_int, [_int, _i64, _i64, _vp, _vp, _vp, _int, _vp]),
    "mvrl_rov3_default_params": (_int, [C.POINTER(MvrlRov3Params)]),
    "mvrl_rov3_create": (_int, [C.POINTER(_vp), C.POINTER(MvrlRov3Params), C.POINTER(MvrlRov3Config)]),
    "mvrl_rov3_destroy": (_int, [_vp]),
    "mvrl_rov3_derivs": (_int, [_vp, _i64, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "mvrl_rov3_step": (_int, [_vp, _i64, _i64, C.POINTER(MvrlRov3Buffers), _vp]),
    "mvrl_rov3_reset": (_int, [_vp, _i64, _i64, C.POINTER(MvrlRov3Buffers), _vp, C.POINTER(_d), _vp]),
    "mvrl_rov3_thruster_model": (_int, [_vp, _i64, _vp, _vp, _vp, _vp, _vp]),
    "mvrl_los_navigation": (_int, [_int, _i64, _i64, _vp, _vp, _d, _vp]),
    "mvrl_auv_default_params": (_int, [C.POINTER(MvrlAuvParams)]),
    "mvrl_auv_create": (_int, [C.POINTER(_vp), C.POINTER(MvrlAuvParams), C.POINTER(MvrlAuvConfig)]),
    "mvrl_auv_destroy": (_int, [_vp]),
    "mvrl_auv_set_apply_noise": (_int, [_vp, _int]),
    "mvrl_auv_set_flow": (_int, [_vp, _vp, _int, _int, _int, _int, _d, _d, _d]),
    "mvrl_auv_step": (_int, [_vp, _i64, _i64, C.POINTER(MvrlAuvBuffers), _vp]),
    "mvrl_auv_reset": (_int, [_vp, _i64, _i64, C.POINTER(MvrlAuvBuffers), _vp, _vp, _vp]),
    "mvrl_flow_interp": (_int, [_int, _vp, _int, _int, _int, _int, _d, _d, _d, _i64, _i64, _vp, _vp, _vp, _vp]),
    "mvrl_replay_add_symmetric": (_int, [_int, _i64, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _i64, _int, _vp]),
    "mvrl_replay_add": (_int, [_int, _i64, _i64, _int, _int, _i64, C.POINTER(MvrlReplayStorage), _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "mvrl_replay_sample": (_int, [_int, _i64, _int, _int, _i64, C.POINTER(MvrlReplayStorage), _i64, C.c_uint64, _vp, _vp, _vp, _vp, _vp, _vp]),
    "mvrl_flow_reconstruct": (_int, [_int, _i64, _int, _int, _vp, _int, _vp, _int, _vp, _vp, _vp]),
    "mvrl_flow_scale": (_int, [_int, _i64, _vp, _vp, _int, _d, _d, _vp]),
    "mvrl_policy_create": (_int, [C.POINTER(_vp), _int, _int, _int]),
    "mvrl_policy_destroy": (_int, [_vp]),
    "mvrl_policy_set_weights": (_int, [_vp] + [_vp] * 9),
    "mvrl_policy_act": (_int, [_vp, _i64, _i64, _vp, _vp, _vp, _vp, _vp, C.c_uint64, C.c_uint64, C.c_uint32, _int, _vp]),
    "mvrl_policy_create_head": (_int, [C.POINTER(_vp), _int, _int, _int, _int]),
    "mvrl_policy_set_weights_squashed": (_int, [_vp] + [_vp] * 11),
    "mvrl_policy_act_ex": (_int, [_vp, _i64, _i64, _vp, _vp, _vp, _vp, _vp, _vp, C.c_uint64, C.c_uint64, C.c_uint32, _int, _vp]),
    "mvrl_policy_create_ex": (_int, [C.POINTER(_vp), _int, _int, _int, _int, _int]),
    "mvrl_policy_set_weights_squashed_device": (_int, [_vp] + [_vp] * 11 + [_vp]),
    "mvrl_critic_create": (_int, [C.POINTER(_vp), _int, _int, _int, _int, _int, _int]),
    "mvrl_critic_destroy": (_int, [_vp]),
    "mvrl_critic_set_weights_device": (_int, [_vp, C.POINTER(_vp), _vp]),
    "mvrl_critic_target": (_int, [_vp, _vp, _i64, _vp, _vp, _vp, _vp, C.c_float, _int, C.c_uint64, _vp, _vp, _vp, _vp, _vp, _vp]),
    "mvrl_critic_saved_bytes": (_i64, [_vp, _i64]),
    "mvrl_critic_grad_scratch": (_i64, [_vp, _i64]),
    "mvrl_critic_forward": (_int, [_vp, _i64, _vp, _vp, _vp, _vp, _vp]),
    "mvrl_critic_backward": (_int, [_vp, _i64, _vp, _vp, _vp, _vp, C.POINTER(_vp), _vp, _vp, _vp]),
    "mvrl_actor_saved_bytes": (_i64, [_vp, _i64]),
    "mvrl_actor_grad_scratch": (_i64, [_vp, _i64]),
    "mvrl_actor_forward": (_int, [_vp, _i64, _vp, _vp, _vp, _vp, _vp, C.c_uint64, _vp, _vp]),
    "mvrl_actor_backward": (_int, [_vp, _i64, _vp, _vp, _vp, _vp, C.POINTER(_vp), _vp, _vp]),
    "mvrl_quantile_huber_scratch": (_i64, [_i64]),
    "mvrl_quantile_huber_loss": (_int, [_i64, _int, _int, _i64, _vp, _vp, _int, _vp, _vp, _vp, _vp]),
}

POLICY_HEAD_FIXED_STD, POLICY_HEAD_SQUASHED = 0, 1
POLICY_PRECISION_BF16, POLICY_PRECISION_FP32 = 0, 1
CRITIC_SAC, CRITIC_TQC = 0, 1

_lib = None


def _make(verbose):
    res = subprocess.run(["make", "-j8", "-C", CSRC_DIR], capture_output=True, text=True)
    if verbose or res.returncode != 0:
        print(res.stdout)
        print(res.stderr)
    if res.returncode != 0:
        raise RuntimeError("building libmvrl.so failed (see output above)")


def default_consts_header():
    """Text of csrc/rov6_default_consts.h for the default vehicle as THIS host computes it (numpy pinv / inv), through
    the built library's own double -> float conversion (mvrl_rov6_dev_constants_f32); exact hex-float literals."""
    from .rov6 import Rov6Constants
    lib = C.CDLL(LIB_PATH)
    lib.mvrl_rov6_dev_constants_f32.restype = _int
    lib.mvrl_rov6_dev_constants_f32.argtypes = [C.POINTER(MvrlRov6Params), C.POINTER(C.c_float), _int]
    params = Rov6Constants().to_struct()
    buf = (C.c_float * 1024)()
    n = lib.mvrl_rov6_dev_constants_f32(C.byref(params), buf, 1024)
    if n <= 0:
        raise RuntimeError("mvrl_rov6_dev_constants_f32 failed")
    lits = [(float(buf[i]).hex() + "f") for i in range(n)]
    rows = ["    " + ", ".join(lits[i:i + 6]) + "," for i in range(0, n, 6)]
    return ("// GENERATED by marinevehiclereinforcementlearning_b200._lib.default_consts_header() (python tools/gen_default_consts.py) -\n"
            "// do not edit.  Rov6Dev<float> of the reference's default BlueROV2 Heavy (dynamicsModel_BlueROV2_Heavy_6DoF.py:83-218,\n"
            "// allocation by numpy pinv as resources.py:19-35), member by member in declaration order, as exact hex-float\n"
            "// literals; the trailing 1 is thrusters_on.  The fp32 step kernels instantiated with CONSTP read these instead of\n"
            "// the kernel argument; mvrl_rov6_create selects them only if the handle's constants match bit for bit.\n"
            "#pragma once\n#define MVRL_ROV6_DEFAULT_WORDS %d\n#define MVRL_ROV6_DEFAULT_INIT_F32 { \\\n%s \\\n    1 }\n" % (n, " \\\n".join(rows)))


def build(verbose=False):
    """Compile libmvrl.so in-tree with nvcc for sm_100a (csrc/Makefile).  The default vehicle's constants are compiled
    into the fp32 step kernels (csrc/rov6_default_consts.h, committed); if this host's numpy produces different bits
    than the committed header holds, the header is regenerated and the library rebuilt once."""
    _make(verbose)
    path = os.path.join(CSRC_DIR, "rov6_default_consts.h")
    text = default_consts_header()
    if not os.path.exists(path) or open(path).read() != text:
        with open(path, "w") as f:
            f.write(text)
        _make(verbose)
    return LIB_PATH


def load():
    """Load libmvrl.so and bind every prototype.  Raises if it is not built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            "libmvrl.so is not built (%s). Build it with `make -C %s` or "
            "`python -c 'import __graft_entry__ as g; g.build()'`. There is no CPU fallback." % (LIB_PATH, CSRC_DIR))
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in PROTOTYPES.items():
        if os.environ.get("MVRL_LIB") and not hasattr(lib, name):
            continue   # an experiment build of older sources (A/B runs); the in-tree library must export everything
        fn = getattr(lib, name)  # AttributeError here = header/library mismatch
        fn.restype = res
        fn.argtypes = args
    if lib.mvrl_version() != 100:
        raise RuntimeError("libmvrl.so version %d does not match the Python binding (100)" % lib.mvrl_version())
    _lib = lib
    return lib


def check(rc):
    if rc != 0:
        msg = load().mvrl_last_error().decode("utf-8", "replace")
        raise RuntimeError("libmvrl error %d: %s" % (rc, msg))


def require_cuda():
    """The product path needs a GPU; fail loudly otherwise."""
    import torch
    if not torch.cuda.is_available() or load().mvrl_device_count() == 0:
        raise RuntimeError("marinevehiclereinforcementlearning_b200 needs a CUDA device (B200, sm_100a); "
                           "there is no CPU fallback")


class Handle:
    """Owner of one opaque libmvrl handle: ``<prefix>_<create>(&h, *args)`` at construction, ``<prefix>_destroy(h)`` when
    the object is collected.  ``_h`` is the handle and ``lib`` the library; ``fn(name)`` is the entry ``<prefix>_<name>``."""

    def __init__(self, prefix, *args, create="create"):
        require_cuda()
        self.lib = load()
        self.prefix = prefix
        self._h = C.c_void_p()
        check(self.fn(create)(C.byref(self._h), *args))

    def fn(self, name):
        return getattr(self.lib, "%s_%s" % (self.prefix, name))

    def __del__(self):
        h = getattr(self, "_h", None)
        if h:
            try:
                self.fn("destroy")(h)
            except Exception:
                pass
            self._h = None


def ptr(t):
    """Device pointer of a torch tensor (or None)."""
    return None if t is None else C.c_void_p(t.data_ptr())


def current_stream(device):
    import torch
    return C.c_void_p(torch.cuda.current_stream(device).cuda_stream)


def torch_dtype_code(dtype):
    import torch
    if dtype == torch.float32:
        return F32
    if dtype == torch.float64:
        return F64
    raise ValueError("dtype must be torch.float32 or torch.float64, got %r" % (dtype,))


def measure_fma_peak(dtype_code, device=0, iters=4096):
    """K6: measured FMA-pipe throughput in TFLOP/s (roofline denominator)."""
    require_cuda()
    tf, ms = C.c_double(), C.c_double()
    check(load().mvrl_measure_fma_peak(dtype_code, device, iters, C.byref(tf), C.byref(ms)))
    return tf.value
