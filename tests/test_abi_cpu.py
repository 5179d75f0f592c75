"""CPU: the C-ABI library loads, exports every symbol include/mvrl.h declares,
fills default constants natively, and refuses to compute without a GPU."""
import ctypes as C
import os
import re
import subprocess
import sys
import textwrap

import numpy as np
import pytest

from conftest import ROOT, load_golden
from marinevehiclereinforcementlearning_b200 import _lib


@pytest.fixture(scope="module")
def lib():
    if not os.path.exists(_lib.LIB_PATH):
        _lib.build()
    return _lib.load()


def test_exports_every_declared_symbol(lib):
    header = open(os.path.join(ROOT, "include", "mvrl.h")).read()
    declared = set(re.findall(r"MVRL_API\s+[\w\s\*]+?\b(mvrl_\w+)\s*\(", header))
    assert len(declared) >= 14
    assert declared == set(_lib.PROTOTYPES), "python binding and header disagree"
    for name in declared:
        assert hasattr(lib, name), name
    assert lib.mvrl_version() == 100


def test_struct_layout_matches_header(lib):
    # sizeof as the C compiler sees it: doubles then one int (padded to 8)
    n_doubles = 3 + 3 + 3 + 9 + 6 + 14 + 14 + 5 + 36 + 36 + 48 + 48 + 30
    assert C.sizeof(_lib.MvrlRov6Params) == n_doubles * 8 + 8
    assert C.sizeof(_lib.MvrlRov6Buffers) == 13 * 8


def test_native_default_params_match_reference(lib):
    g, r = load_golden("rov6"), load_golden("resources")
    p = _lib.MvrlRov6Params()
    assert lib.mvrl_rov6_default_params(C.byref(p)) == 0
    assert np.abs(np.array(p.A).reshape(6, 8) - r["A6"]).max() < 1e-15
    assert np.abs(np.array(p.Ainv).reshape(8, 6) - r["Ainv6"]).max() < 1e-14
    assert np.abs(np.array(p.M).reshape(6, 6) - g["M"]).max() == 0.0
    assert np.abs(np.array(p.Minv).reshape(6, 6) - g["Minv"]).max() < 1e-15
    assert p.thrust_coef == pytest.approx(float(g["rhoD4Kt"]), rel=1e-15)
    assert p.W - p.B == 0.0


def test_python_constants_match_reference():
    from marinevehiclereinforcementlearning_b200.rov6 import Rov6Constants
    g, r = load_golden("rov6"), load_golden("resources")
    c = Rov6Constants()
    q = c.to_struct()
    assert np.array_equal(c.A, r["A6"]) and np.abs(c.Ainv - r["Ainv6"]).max() < 1e-15
    assert np.array_equal(np.array(q.Minv).reshape(6, 6), g["Minv"])
    assert c.Kt_thruster == float(g["Kt_thruster"])
    v0 = c.fingerprint()
    c.m = 12.0
    assert c.fingerprint() != v0


def test_invalid_arguments_are_reported(lib):
    assert lib.mvrl_rov6_default_params(None) == -1
    assert b"null" in lib.mvrl_last_error()
    p = _lib.MvrlRov6Params()
    lib.mvrl_rov6_default_params(C.byref(p))
    cfg = _lib.MvrlRov6Config(dtype=7, action_mode=0, n_sub=8, max_steps=250, dt=0.2)
    h = C.c_void_p()
    assert lib.mvrl_rov6_create(C.byref(h), C.byref(p), C.byref(cfg)) == -1
    cfg.dtype = 0
    cfg.n_sub = 0
    assert lib.mvrl_rov6_create(C.byref(h), C.byref(p), C.byref(cfg)) == -1


NO_CPU_FALLBACK = textwrap.dedent("""
    import ctypes as C, sys
    sys.path.insert(0, %r)
    import pytest, torch
    from marinevehiclereinforcementlearning_b200 import _lib
    assert not torch.cuda.is_available()
    lib = _lib.load()
    p = _lib.MvrlRov6Params()
    lib.mvrl_rov6_default_params(C.byref(p))
    cfg = _lib.MvrlRov6Config(dtype=0, action_mode=0, n_sub=8, max_steps=250, dt=0.2)
    h = C.c_void_p()
    assert lib.mvrl_rov6_create(C.byref(h), C.byref(p), C.byref(cfg)) == -3  # MVRL_ENODEV
    from marinevehiclereinforcementlearning_b200 import BlueROV2Heavy6DoFVecEnv, resources
    with pytest.raises(RuntimeError):
        BlueROV2Heavy6DoFVecEnv(4)
    with pytest.raises(RuntimeError):
        resources.angleError(0.1, 0.2)
    print("no cpu fallback ok")
""")


def test_no_cpu_fallback(lib):
    """Without a CUDA device every compute entry point refuses; checked in a fresh interpreter that sees no device
    (CUDA_VISIBLE_DEVICES=""), so it runs on GPU machines too."""
    res = subprocess.run([sys.executable, "-c", NO_CPU_FALLBACK % ROOT], env=dict(os.environ, CUDA_VISIBLE_DEVICES=""),
                         capture_output=True, text=True, timeout=600)
    assert res.returncode == 0 and "no cpu fallback ok" in res.stdout, res.stdout[-2000:] + res.stderr[-2000:]


def test_product_does_not_import_oracle():
    pkg = os.path.join(ROOT, "marinevehiclereinforcementlearning_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                src = open(os.path.join(dirpath, f)).read()
                assert not re.search(r"oracle", src, re.I), os.path.join(dirpath, f)


def test_host_chunk_plan(lib):
    """Host logic of mvrl_rov6_step_host's piece schedule (no GPU needed)."""
    assert lib.mvrl_host_chunk_count(0, 0) == 0
    assert lib.mvrl_host_chunk_count(1, 0) == 1 and lib.mvrl_host_chunk_count(257, 0) == 1 and lib.mvrl_host_chunk_count(257, 8) == 2
    assert lib.mvrl_host_chunk_count(4096, 0) == 1 and lib.mvrl_host_chunk_count(1 << 18, 0) == 4   # default: no piece under 64 Ki envs
    assert lib.mvrl_host_chunk_count(1 << 20, 0) == 8
    assert lib.mvrl_host_chunk_count(1 << 20, 4) == 4 and lib.mvrl_host_chunk_count(1 << 20, -3) == 3
    assert lib.mvrl_host_chunk_count(1000, 64) == 4          # pieces are multiples of the 256-env transpose tile
    assert lib.mvrl_host_chunk_count(1 << 20, 1000) == 64    # capped


def test_committed_default_constants_header_is_what_this_host_generates():
    """csrc/rov6_default_consts.h (the default vehicle's fp32 constants compiled into the CONSTP step kernels) must equal
    what the library's own double -> float conversion gives for Rov6Constants() here; build() regenerates it otherwise."""
    from marinevehiclereinforcementlearning_b200 import _lib
    path = os.path.join(_lib.CSRC_DIR, "rov6_default_consts.h")
    assert open(path).read() == _lib.default_consts_header()
