"""CPU: the fp32 precision of the fused rollout actor - its C ABI declarations, the Python argument check, and the entry
point's argument checks on an interpreter that sees no CUDA device."""
import os
import re
import subprocess
import sys
import textwrap

import pytest

from conftest import ROOT
from marinevehiclereinforcementlearning_b200 import _lib


def test_abi_declares_the_precisions():
    header = open(os.path.join(ROOT, "include", "mvrl.h")).read()
    assert re.search(r"MVRL_API\s+int\s+mvrl_policy_create_ex\s*\(", header)
    assert len(_lib.PROTOTYPES["mvrl_policy_create_ex"][1]) == len(_lib.PROTOTYPES["mvrl_policy_create_head"][1]) + 1
    assert re.search(r"#define MVRL_POLICY_PRECISION_BF16 0\b", header) and re.search(r"#define MVRL_POLICY_PRECISION_FP32 1\b", header)
    assert (_lib.POLICY_PRECISION_BF16, _lib.POLICY_PRECISION_FP32) == (0, 1)


# the library path points nowhere: a ValueError (not the RuntimeError of a missing library) shows that the precision is
# checked before the library or CUDA is touched
BAD_PRECISION = textwrap.dedent("""
    import sys
    sys.path.insert(0, %r)
    import pytest
    from marinevehiclereinforcementlearning_b200 import MlpGaussianPolicy, SquashedGaussianPolicy
    for cls in (MlpGaussianPolicy, SquashedGaussianPolicy):
        for bad in ("fp16", "FP32", "tf32", None, 1):
            with pytest.raises(ValueError, match="precision"):
                cls(9, 6, precision=bad)
    print("precision check ok")
""")


def test_unknown_precision_raises_value_error_before_the_library():
    res = subprocess.run([sys.executable, "-c", BAD_PRECISION % ROOT],
                         env=dict(os.environ, CUDA_VISIBLE_DEVICES="", MVRL_LIB=os.path.join(ROOT, "no-such-libmvrl.so")),
                         capture_output=True, text=True, timeout=600)
    assert res.returncode == 0 and "precision check ok" in res.stdout, res.stdout[-2000:] + res.stderr[-2000:]


NO_DEVICE = textwrap.dedent("""
    import ctypes as C, os, sys
    sys.path.insert(0, %r)
    import torch
    from marinevehiclereinforcementlearning_b200 import _lib
    assert not torch.cuda.is_available()
    lib = _lib.load()
    h = C.c_void_p()
    for bad in (2, -1):
        assert lib.mvrl_policy_create_ex(C.byref(h), 0, 9, 6, 1, bad) == -1 and b"precision" in lib.mvrl_last_error()
    for head in (0, 1):
        assert lib.mvrl_policy_create_ex(C.byref(h), 0, 9, 6, head, 1) == -3                       # MVRL_ENODEV
        assert lib.mvrl_policy_create_ex(C.byref(h), 0, 9, 6, head, 0) == -3
    assert lib.mvrl_policy_create_ex(C.byref(h), 0, 9, 6, 2, 1) == -1 and b"head" in lib.mvrl_last_error()
    os.environ["MVRL_POLICY_MMA_SYNC"] = "1"
    assert lib.mvrl_policy_create_ex(C.byref(h), 0, 9, 6, 1, 1) == -1 and b"MVRL_POLICY_MMA_SYNC" in lib.mvrl_last_error()
    assert lib.mvrl_policy_create_ex(C.byref(h), 0, 9, 6, 1, 0) == -3
    print("fp32 precision no device ok")
""")


def test_entry_point_without_a_device():
    """In a fresh interpreter that sees no device: an unknown precision is MVRL_EINVAL naming the precision, fp32 with
    MVRL_POLICY_MMA_SYNC=1 is MVRL_EINVAL naming the variable, a valid handle MVRL_ENODEV."""
    res = subprocess.run([sys.executable, "-c", NO_DEVICE % ROOT], env=dict(os.environ, CUDA_VISIBLE_DEVICES=""),
                         capture_output=True, text=True, timeout=600)
    assert res.returncode == 0 and "fp32 precision no device ok" in res.stdout, res.stdout[-2000:] + res.stderr[-2000:]
