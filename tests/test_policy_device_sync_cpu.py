"""CPU: the ABI of the squashed head's stream-ordered weight sync (mvrl_policy_set_weights_squashed_device)."""
import ctypes as C
import os
import re

import pytest

from conftest import ROOT
from marinevehiclereinforcementlearning_b200 import _lib

NAME = "mvrl_policy_set_weights_squashed_device"


@pytest.fixture(scope="module")
def lib():
    if not os.path.exists(_lib.LIB_PATH):
        _lib.build()
    return _lib.load()


def test_prototype_matches_header():
    header = open(os.path.join(ROOT, "include", "mvrl.h")).read()
    m = re.search(r"MVRL_API\s+int\s+%s\s*\(([^;]*)\);" % NAME, header)
    assert m, NAME
    args = [a.strip() for a in m.group(1).split(",")]
    assert len(args) == 13 and args[0].startswith("MvrlPolicy*") and args[-1].startswith("mvrl_stream_t")
    res, argtypes = _lib.PROTOTYPES[NAME]
    assert res is C.c_int and len(argtypes) == 13
    # the same weights, in the same order, as the host entry; then the stream
    assert len(_lib.PROTOTYPES["mvrl_policy_set_weights_squashed"][1]) == 12


def test_null_handle_is_rejected_with_a_message(lib):
    w = (C.c_float * 16)()
    p = C.cast(w, C.c_void_p)
    assert getattr(lib, NAME)(None, *([p] * 10), None, None) == -1
    assert b"null" in lib.mvrl_last_error()
    assert getattr(lib, NAME)(None, *([p] * 10), p, None) == -1
    assert NAME.encode() in lib.mvrl_last_error()
