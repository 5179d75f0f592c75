"""CPU: the C ABI of the device replay buffer (mvrl_replay_add / mvrl_replay_sample), the argument checks of
vec_tools.ReplayBuffer that run before the library is reached, the refusal without a GPU, and the NumPy restatement of the
sampler that tests/test_replay_gpu.py compares the kernel against."""
import ctypes as C
import os
import re
import subprocess
import sys
import textwrap

import numpy as np
import pytest
import torch

from conftest import ROOT
from marinevehiclereinforcementlearning_b200 import _lib
from oracle import oracle_np as o

SAMPLE_STREAM = 9


def mulhi64(a, b):
    """floor(a * b / 2^64) for uint64 arrays a and b < 2^32, exactly (no uint64 overflow: see the bounds below)."""
    a, b = np.asarray(a, dtype=np.uint64), np.asarray(b, dtype=np.uint64)
    assert int(b.max(initial=0)) < 2 ** 32
    lo, hi = a & np.uint64(0xFFFFFFFF), a >> np.uint64(32)
    # hi * b <= (2^32 - 1)^2 and (lo * b) >> 32 < 2^32, so their sum stays below 2^64
    return (hi * b + ((lo * b) >> np.uint64(32))) >> np.uint64(32)


def replay_sample_indices(seed, call, batch, size, n_envs):
    """The sampler of mvrl_replay_sample: sample i takes Philox4x32-10 block (i, call_lo, call_hi, 9 * 65536) under key
    (seed_lo, seed_hi); slot = (x | y << 32) * size >> 64, env = (z | w << 32) * n_envs >> 64."""
    i = np.arange(batch, dtype=np.uint64)
    ctr = np.stack([i, np.full(batch, call & 0xFFFFFFFF, dtype=np.uint64), np.full(batch, (call >> 32) & 0xFFFFFFFF, dtype=np.uint64),
                    np.full(batch, SAMPLE_STREAM * 65536, dtype=np.uint64)], axis=1)
    w = o.philox4x32(ctr, (seed & 0xFFFFFFFF, (seed >> 32) & 0xFFFFFFFF)).astype(np.uint64)
    u0 = w[:, 0] | (w[:, 1] << np.uint64(32))
    u1 = w[:, 2] | (w[:, 3] << np.uint64(32))
    return mulhi64(u0, np.uint64(size)).astype(np.int64), mulhi64(u1, np.uint64(n_envs)).astype(np.int64)


def test_sampler_restatement_known_answers():
    # Philox4x32-10 known-answer vectors of Random123 (kat_vectors): the block function itself
    w = o.philox4x32(np.array([[0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344]], dtype=np.uint64), (0xa4093822, 0x299f31d0))
    assert [int(v) for v in w[0]] == [0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1]
    # the 64-bit multiply-high, by hand: 2^63 * s >> 64 = s // 2; (2^64 - 1) * s >> 64 = s - 1; 2^32 * s >> 64 = s >> 32 = 0
    assert mulhi64([2 ** 63], 37)[0] == 18 and mulhi64([2 ** 64 - 1], 37)[0] == 36 and mulhi64([2 ** 32], 37)[0] == 0
    assert mulhi64([2 ** 64 - 1], 2 ** 32 - 1)[0] == 2 ** 32 - 2
    # counter (0, 0, 0, 9 * 65536), key (0, 0): the words and the indices they give, against Python's exact integers
    w = o.philox4x32(np.array([[0, 0, 0, SAMPLE_STREAM * 65536]], dtype=np.uint64), (0, 0))[0].astype(object)
    slot, env = replay_sample_indices(0, 0, 1, 7, 300)
    assert slot[0] == ((int(w[0]) | int(w[1]) << 32) * 7) >> 64 and env[0] == ((int(w[2]) | int(w[3]) << 32) * 300) >> 64
    # the call counter's high word and a 64-bit seed enter the counter / key
    s1, e1 = replay_sample_indices(2 ** 63 + 5, 2 ** 32 + 3, 64, 1000, 1000)
    s2, e2 = replay_sample_indices(5, 3, 64, 1000, 1000)
    assert not np.array_equal(s1, s2) and not np.array_equal(e1, e2)
    assert s1.min() >= 0 and s1.max() < 1000 and e1.max() < 1000


def test_abi_declarations_and_argument_types():
    header = open(os.path.join(ROOT, "include", "mvrl.h")).read()
    for name in ("mvrl_replay_add", "mvrl_replay_sample"):
        assert re.search(r"MVRL_API int %s\(" % name, header), name
    assert "#define MVRL_REPLAY_MAX_DIM 16" in header and _lib.REPLAY_MAX_DIM == 16
    fields = re.search(r"typedef struct MvrlReplayStorage \{(.*?)\} MvrlReplayStorage;", header, re.S).group(1)
    names = re.findall(r"\*\s*(\w+);", fields)
    assert names == [f for f, _ in _lib.MvrlReplayStorage._fields_]
    assert C.sizeof(_lib.MvrlReplayStorage) == 8 * 8
    res, args = _lib.PROTOTYPES["mvrl_replay_add"]
    assert res is C.c_int and len(args) == 14 and args[6]._type_ is _lib.MvrlReplayStorage
    assert args[:6] == [C.c_int, C.c_int64, C.c_int64, C.c_int, C.c_int, C.c_int64]
    res, args = _lib.PROTOTYPES["mvrl_replay_sample"]
    assert res is C.c_int and len(args) == 14 and args[5]._type_ is _lib.MvrlReplayStorage
    assert args[6] is C.c_int64 and args[7] is C.c_uint64


class _FakeEnv:
    """The attributes ReplayBuffer reads from an env, without any device buffer."""
    def __init__(self, n=4, obs=9, act=6, dtype=torch.float32):
        self.num_envs, self.lenObs, self.lenAction, self.dtype, self.ld = n, obs, act, dtype, 32
        self.device, self.auto_reset, self._terminal_obs = torch.device("cuda", 0), False, None


def test_python_argument_checks_before_the_library():
    from marinevehiclereinforcementlearning_b200 import ReplayBuffer
    with pytest.raises(ValueError, match="buffer_size"):
        ReplayBuffer(0, _FakeEnv())
    with pytest.raises(ValueError, match="obs_dim"):
        ReplayBuffer(100, _FakeEnv(obs=17))
    with pytest.raises(ValueError, match="obs_dim"):
        ReplayBuffer(100, _FakeEnv(act=0))
    with pytest.raises(ValueError, match="no environments"):
        ReplayBuffer(100, _FakeEnv(n=0))
    with pytest.raises(ValueError, match="dtype"):
        ReplayBuffer(100, _FakeEnv(dtype=torch.float16))


NO_GPU = textwrap.dedent("""
    import ctypes as C, sys
    sys.path.insert(0, %r)
    sys.path.insert(0, %r)
    import numpy as np, pytest, torch
    from marinevehiclereinforcementlearning_b200 import _lib, ReplayBuffer
    from test_replay_cpu import _FakeEnv
    assert not torch.cuda.is_available()
    with pytest.raises(RuntimeError):
        ReplayBuffer(100, _FakeEnv())
    lib = _lib.load()
    host = [np.zeros(64) for _ in range(8)]
    s = _lib.MvrlReplayStorage(*[a.ctypes.data for a in host])
    p = lambda a: C.c_void_p(a.ctypes.data)
    done = np.zeros(4, np.uint8)
    assert lib.mvrl_replay_add(0, 4, 32, 9, 6, 5, C.byref(s), p(host[0]), None, p(host[1]), p(host[2]), p(done), None, None) != 0
    assert lib.mvrl_replay_sample(0, 4, 9, 6, 5, C.byref(s), 8, 0, p(host[0]), p(host[1]), p(host[2]), p(host[3]), p(host[4]), None) != 0
    print("replay refuses without a gpu")
""")


def test_refuses_without_a_gpu():
    """Without a CUDA device the Python class raises RuntimeError and the C entries refuse (host pointers are not device
    memory); in a fresh interpreter that sees no device, so it runs on GPU machines too."""
    res = subprocess.run([sys.executable, "-c", NO_GPU % (ROOT, os.path.join(ROOT, "tests"))], env=dict(os.environ, CUDA_VISIBLE_DEVICES=""),
                         capture_output=True, text=True, timeout=600)
    assert res.returncode == 0 and "replay refuses without a gpu" in res.stdout, res.stdout[-2000:] + res.stderr[-2000:]
