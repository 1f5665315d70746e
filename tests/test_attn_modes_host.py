"""CPU: the attention CNN's compute modes on the host side -- attn_model_struct.compute_mode accepts 'bf16x3' (the
default) and 'fp16' only, and attn_plan_create_mode is declared in the header, typed in the ctypes table and rejects
unknown modes before any CUDA call."""
import ctypes
import os
import re

import pytest

import monkey_pose_b200 as mp
from monkey_pose_b200 import _lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_compute_mode_default_and_values():
    am = mp.attn_model_struct()
    assert am.compute_mode == "bf16x3"
    am.compute_mode = "fp16"
    assert am.compute_mode == "fp16"
    am.compute_mode = "bf16x3"
    assert am.compute_mode == "bf16x3"


@pytest.mark.parametrize("mode", ["bf16", "fp32", "FP16", "tf32", None, 3])
def test_unknown_compute_mode_raises_value_error(mode):
    am = mp.attn_model_struct()
    with pytest.raises(ValueError):
        am.compute_mode = mode
    assert am.compute_mode == "bf16x3"


def test_attn_plan_create_mode_is_declared_and_typed():
    src = re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", "hgru_b200.h")).read(), flags=re.S)
    decl = re.search(r"HGRU_API\s+int\s+attn_plan_create_mode\s*\(([^)]*)\)", src)
    assert decl, "attn_plan_create_mode missing from the header"
    assert len([a for a in decl.group(1).split(",") if a.strip()]) == 8
    res, args = _lib.SIGNATURES["attn_plan_create_mode"]
    assert res is ctypes.c_int and len(args) == 8
    assert args[6] is ctypes.c_int                                  # mode
    assert args[:6] == _lib.SIGNATURES["attn_plan_create"][1][:6]   # the same shape arguments as attn_plan_create


def test_attn_plan_create_mode_rejects_unknown_modes_without_a_device():
    lib = _lib.load()
    w = (ctypes.c_int * 5)(64, 128, 256, 512, 1024)
    h = ctypes.c_void_p()
    for mode in (_lib.MODE_FP32, _lib.MODE_BF16, 7, -1):
        assert lib.attn_plan_create_mode(2, 424, 512, w, 1024, 3, mode, ctypes.byref(h)) == 2, mode   # UNSUPPORTED
        assert b"mode" in lib.hgru_last_error()
        assert not h.value
    assert lib.attn_plan_create_mode(2, 424, 512, w, 1024, 3, _lib.MODE_FP16, None) == 1              # null out
    assert lib.attn_plan_create_mode(0, 424, 512, w, 1024, 3, _lib.MODE_FP16, ctypes.byref(h)) == 1   # empty batch
