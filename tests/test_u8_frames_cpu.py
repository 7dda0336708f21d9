"""CPU suite of uint8 frames (ABI v7): the dtype constant, every refusal before any CUDA call, the host workspace of a uint8
frame bank, and the Python-level refusals that need no device."""
import ctypes
import math
import os
import re

import pytest
import torch

from conftest import ROOT

F32, BF16, U8 = 0, 1, 3
OCC, MOB = 1, 2


def _fake(n):
    """Host addresses that stand in for device pointers: validation fails before anything dereferences them."""
    return ctypes.c_void_p(0x10000 * n)


def test_u8_constant_matches_the_header(tcl):
    text = open(os.path.join(ROOT, "include", "tcl_b200.h")).read()
    assert int(re.search(r"#define TCLB200_U8 (\d+)", text).group(1)) == tcl._cabi.U8 == U8
    assert not re.search(r"#define TCLB200_\w+ 2\s", text.split("/* frame dtype */")[1].split("/* mask tests")[0])


def _u8_args(tcl, **kw):
    a = tcl._cabi.TclArgs()
    a.bf, a.ff, a.prev, a.cur = _fake(1), _fake(2), _fake(3), _fake(4)
    a.pair_sums, a.scratch, a.scratch_bytes = _fake(5), _fake(6), 1 << 30
    a.B, a.C, a.H, a.W = 2, 3, 16, 16
    a.dtype, a.flags = U8, OCC | MOB
    a.u8_scale[:] = (1 / 255,) * 3
    for k, v in kw.items():
        setattr(a, k, v)
    return a


@pytest.mark.parametrize("change,code,words", [
    (dict(warp_out=_fake(7)), 3, b"warp_out"),
    (dict(blend_out=_fake(7)), 3, b"blend_out"),
    (dict(pair_sums=None), 1, b"reduction"),
    (dict(cur=None), 1, b"reduction"),
    (dict(C=1), 1, b"C == 3"),
    (dict(C=4), 1, b"C == 3"),
])
def test_fused_forward_refusals_without_gpu(tcl, change, code, words):
    lib = tcl._cabi.lib()
    a = _u8_args(tcl, **change)
    assert lib.tclb200_tcl_forward(ctypes.byref(a), None) == code
    assert words in lib.tclb200_last_error()


@pytest.mark.parametrize("field,index,value", [("u8_scale", 0, math.nan), ("u8_scale", 2, math.inf), ("u8_offset", 1, -math.inf),
                                               ("u8_offset", 0, math.nan)])
def test_non_finite_normalisation_is_refused(tcl, field, index, value):
    lib = tcl._cabi.lib()
    a = _u8_args(tcl)
    getattr(a, field)[index] = value
    assert lib.tclb200_tcl_forward(ctypes.byref(a), None) == 1
    assert b"finite" in lib.tclb200_last_error()


def test_dtype_2_stays_unassigned(tcl):
    lib = tcl._cabi.lib()
    a = _u8_args(tcl, dtype=2)
    assert lib.tclb200_tcl_forward(ctypes.byref(a), None) == 1
    assert b"dtype" in lib.tclb200_last_error()


def test_warp_and_backward_entries_refuse_u8(tcl):
    lib = tcl._cabi.lib()
    x, f, out = _fake(1), _fake(2), _fake(3)
    assert lib.tclb200_warp(x, f, out, 2, 3, 8, 8, U8, 0, None) == 1
    assert b"uint8" in lib.tclb200_last_error()
    assert lib.tclb200_warp_backward_dt(_fake(1), x, f, _fake(4), _fake(5), 2, 3, 8, 8, U8, 0, None, 0, None) == 1
    assert b"uint8" in lib.tclb200_last_error()
    assert lib.tclb200_tcl_backward_dt(f, _fake(6), x, _fake(7), _fake(8), 1.0, _fake(9), _fake(10), 2, 3, 8, 8, U8, 0, 0,
                                       None, 0, None) == 1
    assert b"uint8" in lib.tclb200_last_error()


def test_host_workspace_of_a_u8_bank_is_smaller(tcl):
    lib = tcl._cabi.lib()
    f32 = lib.tclb200_host_workspace_bytes(4, 5, 3, 64, 64, F32, 0, 0)
    bf16 = lib.tclb200_host_workspace_bytes(4, 5, 3, 64, 64, BF16, 0, 0)
    u8 = lib.tclb200_host_workspace_bytes(4, 5, 3, 64, 64, U8, 0, 0)
    assert u8 < bf16 < f32
    assert bf16 - u8 >= 5 * 3 * 64 * 64 - 256 * 2       # one byte per value instead of two (frame bank, 256-byte rounding)


def test_host_entry_refusals_without_gpu(tcl):
    import numpy as np
    lib = tcl._cabi.lib()
    bf = np.zeros((1, 2, 8, 8), np.float32); fr = np.zeros((2, 3, 8, 8), np.uint8)
    pi = np.array([0], np.int32); ci = np.array([1], np.int32); out = np.zeros(1, np.float32)
    a = tcl._cabi.HostArgs()
    a.P, a.F, a.C, a.H, a.W, a.dtype = 1, 2, 3, 8, 8, U8
    a.bf, a.frames, a.prev_index, a.cur_index, a.pair_vals = (bf.ctypes.data, fr.ctypes.data, pi.ctypes.data, ci.ctypes.data,
                                                              out.ctypes.data)
    a.u8_scale[:] = (1 / 255,) * 3
    a.u8_offset[1] = math.nan
    assert lib.tclb200_tcl_forward_host(ctypes.byref(a), None) == 1
    assert b"finite" in lib.tclb200_last_error()
    a.u8_offset[1] = 0.0
    a.C = 1
    assert lib.tclb200_tcl_forward_host(ctypes.byref(a), None) == 1
    assert b"C == 3" in lib.tclb200_last_error()
    a.C = 3
    assert lib.tclb200_tcl_forward_host(ctypes.byref(a), None) == 1           # valid so far: the workspace is missing
    assert b"workspace" in lib.tclb200_last_error()


def test_python_normalisation_arguments(tcl):
    ops = tcl.ops
    assert ops._u8_norm(U8, None, None, 3) == ((ops.U8_SCALE,) * 3, (0.0,) * 3)
    assert ops.U8_SCALE == float(torch.tensor(1 / 255, dtype=torch.float32))
    s, o = ops._u8_norm(U8, 2 / 255, -1.0, 3)
    assert s == (float(torch.tensor(2 / 255, dtype=torch.float32)),) * 3 and o == (-1.0,) * 3
    s, o = ops._u8_norm(U8, 1.0, [-124.0, -117.5, -104.25], 3)
    assert s == (1.0,) * 3 and o == (-124.0, -117.5, -104.25)
    for bad in (dict(u8_scale=[1.0, 2.0]), dict(u8_offset=math.nan), dict(u8_scale=math.inf)):
        with pytest.raises(RuntimeError):
            ops._u8_norm(U8, bad.get("u8_scale"), bad.get("u8_offset"), 3)
    with pytest.raises(RuntimeError, match="3 channels"):
        ops._u8_norm(U8, None, None, 1)
    with pytest.raises(RuntimeError, match="uint8 frames only"):       # not silently ignored for float frames
        ops._u8_norm(F32, 1 / 255, None, 3)
    with pytest.raises(RuntimeError, match="uint8 frames only"):
        ops._u8_norm(BF16, None, 0.0, 3)


def test_non_evaluation_entries_still_refuse_u8_and_half(tcl):
    with pytest.raises(RuntimeError, match="float32 or bfloat16"):
        tcl.ops._frame_dtype(torch.zeros(1, 3, 4, 4, dtype=torch.uint8))
    with pytest.raises(RuntimeError, match="float32 or bfloat16"):
        tcl.ops._eval_frame_dtype(torch.zeros(1, 3, 4, 4).half())
    assert tcl.ops._eval_frame_dtype(torch.zeros(1, 3, 4, 4, dtype=torch.uint8)) == U8
