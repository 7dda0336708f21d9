"""CPU suite of channels-last host data in the host-buffer entry (ABI v8): which host tensors count as channels-last, that
they reach the C ABI without a copy, the workspace each layout bit adds, and the refusals before any CUDA call."""
import ctypes
import itertools
import os
import re

import numpy as np
import pytest
import torch

from conftest import ROOT

F32, BF16, U8 = 0, 1, 3
CL_FRAMES, CL_FF, CL_BF = 1, 2, 4


def _cl(n, h, w, c, dtype=torch.float32):
    """An (N,C,H,W) view of interleaved (N,H,W,C) memory, as `.permute(0, 3, 1, 2)` of a decoder's array gives it."""
    return torch.zeros(n, h, w, c, dtype=dtype).permute(0, 3, 1, 2)


def test_cl_constants_match_the_header(tcl):
    text = open(os.path.join(ROOT, "include", "tcl_b200.h")).read()
    for name, v in (("FRAMES", CL_FRAMES), ("FF", CL_FF), ("BF", CL_BF)):
        assert int(re.search(rf"#define TCLB200_CL_{name} (\d+)", text).group(1)) == getattr(tcl._cabi, f"CL_{name}") == v


@pytest.mark.parametrize("t", [
    _cl(2, 5, 7, 3), _cl(3, 4, 6, 2), _cl(2, 5, 7, 3, torch.uint8), _cl(2, 5, 7, 3, torch.bfloat16), _cl(1, 9, 1, 4),
])
def test_channels_last_views_are_detected(tcl, t):
    assert tcl.ops._is_channels_last(t)


@pytest.mark.parametrize("t", [
    torch.zeros(2, 3, 5, 7),                                  # planar
    _cl(2, 5, 7, 1),                                          # C == 1: both layouts are the same memory
    _cl(2, 1, 1, 3),                                          # H*W == 1: likewise
    torch.zeros(2, 5, 7, 3)[:, :, :6].permute(0, 3, 1, 2),    # a crop of interleaved memory: rows are not dense
    torch.zeros(2, 3, 5, 7).transpose(2, 3),                  # other strides
    torch.zeros(2, 4, 5, 7)[:, ::2],
    torch.zeros(5, 7, 3),                                     # not 4-D
])
def test_other_tensors_are_planar(tcl, t):
    assert not tcl.ops._is_channels_last(t)


def test_host_tensor_keeps_channels_last_storage_and_copies_everything_else(tcl):
    ht = tcl.ops._host_tensor
    fr = _cl(4, 6, 8, 3, torch.uint8)
    assert ht(fr, "frames", channels_last_ok=True) is fr                     # handed over as is: same storage, no copy
    planar = ht(fr, "frames")                                               # (the other callers: planar, as before)
    assert planar.is_contiguous() and planar.data_ptr() != fr.data_ptr() and torch.equal(planar, fr)
    fl = _cl(3, 6, 8, 2)
    assert ht(fl, "bf", torch.float32, channels_last_ok=True) is fl
    conv = ht(_cl(3, 6, 8, 2, torch.float64), "bf", torch.float32, channels_last_ok=True)   # a dtype conversion keeps the layout
    assert conv.dtype == torch.float32 and tcl.ops._is_channels_last(conv)
    odd = torch.zeros(2, 3, 5, 7).transpose(2, 3)
    got = ht(odd, "frames", channels_last_ok=True)
    assert got.is_contiguous() and torch.equal(got, odd)


SHAPES = [(1, 2, 3, 8, 8), (5, 6, 3, 37, 53), (64, 65, 3, 436, 1024), (40, 12, 4, 64, 96), (7, 3, 1, 17, 16)]


@pytest.mark.parametrize("P,F,C,H,W", SHAPES)
def test_zero_bits_give_the_planar_workspace(tcl, P, F, C, H, W):
    lib = tcl._cabi.lib()
    for dt, chunk, mask in itertools.product((F32, BF16, U8), (0, 1, 3, 8, 200), (0, 1)):
        assert lib.tclb200_host_workspace_bytes_cl(P, F, C, H, W, dt, chunk, mask, 0) == \
            lib.tclb200_host_workspace_bytes(P, F, C, H, W, dt, chunk, mask)


def _up256(v):
    return (v + 255) // 256 * 256


def _chunk(P, H, W, chunk_pairs):
    c = chunk_pairs if chunk_pairs > 0 else max(1, min(128, (256 << 20) // (H * W * 8)))
    return min(c, P)


@pytest.mark.parametrize("P,F,C,H,W", SHAPES)
def test_each_bit_adds_its_staging_or_planar_buffer(tcl, P, F, C, H, W):
    lib = tcl._cabi.lib()
    for dt, chunk_pairs, mask in itertools.product((F32, BF16, U8), (0, 1, 3, 200), (0, 1)):
        base = lib.tclb200_host_workspace_bytes(P, F, C, H, W, dt, chunk_pairs, mask)
        chunk = _chunk(P, H, W, chunk_pairs)
        frame_bytes = C * H * W * {F32: 4, BF16: 2, U8: 1}[dt]
        stage = 3 * _up256(min(F, 2 * chunk) * frame_bytes)          # one staging area per ring slot
        planar = _up256(chunk * 2 * H * W * 4)                        # one planar chunk buffer per flow field
        add = {CL_FRAMES: stage, CL_FF: planar, CL_BF: planar}
        for bits in range(8):
            want = base + sum(v for b, v in add.items() if bits & b)
            assert lib.tclb200_host_workspace_bytes_cl(P, F, C, H, W, dt, chunk_pairs, mask, bits) == want, (dt, chunk_pairs, mask, bits)


def test_workspace_of_unknown_bits_is_zero(tcl):
    lib = tcl._cabi.lib()
    for bits in (8, 9, 16, -1, 1 << 30):
        assert lib.tclb200_host_workspace_bytes_cl(4, 5, 3, 16, 16, F32, 0, 0, bits) == 0


def _host_args(tcl, arrays, **kw):
    bf, ff, fr, pi, ci, out = arrays
    a = tcl._cabi.HostArgs()
    a.P, a.F, a.C, a.H, a.W, a.dtype = 2, 3, 3, 8, 8, F32
    a.bf, a.ff, a.frames, a.prev_index, a.cur_index, a.pair_vals = (bf.ctypes.data, ff.ctypes.data, fr.ctypes.data, pi.ctypes.data,
                                                                    ci.ctypes.data, out.ctypes.data)
    for k, v in kw.items():
        setattr(a, k, v)
    return a


@pytest.fixture
def arrays():
    return (np.zeros((2, 8, 8, 2), np.float32), np.zeros((2, 8, 8, 2), np.float32), np.zeros((3, 8, 8, 3), np.float32),
            np.array([0, 1], np.int32), np.array([1, 2], np.int32), np.zeros(2, np.float32))


@pytest.mark.parametrize("bits", [8, 1 << 5, -1, CL_FRAMES | 16])
def test_unknown_bits_are_refused_before_any_cuda_call(tcl, arrays, bits):
    lib = tcl._cabi.lib()
    a = _host_args(tcl, arrays, channels_last=bits)
    assert lib.tclb200_tcl_forward_host(ctypes.byref(a), None) == 1
    assert b"unknown bits" in lib.tclb200_last_error()
    a.P = 0                                                    # even for a call that would have nothing to do
    assert lib.tclb200_tcl_forward_host(ctypes.byref(a), None) == 1


@pytest.mark.parametrize("bits", [CL_FRAMES, CL_FF, CL_BF, CL_FRAMES | CL_FF | CL_BF])
@pytest.mark.parametrize("dt", [F32, BF16, U8])
def test_a_workspace_sized_without_the_bits_is_refused(tcl, arrays, bits, dt):
    """Sized for planar data (or one byte short of the channels-last size), the workspace is too small: INVALID, and no CUDA
    call has been made (none could succeed here)."""
    lib = tcl._cabi.lib()
    P, F, C, H, W = 2, 3, 3, 8, 8
    planar = lib.tclb200_host_workspace_bytes(P, F, C, H, W, dt, 0, 0)
    need = lib.tclb200_host_workspace_bytes_cl(P, F, C, H, W, dt, 0, 0, bits)
    assert need > planar
    for have in (planar, need - 1):
        a = _host_args(tcl, arrays, channels_last=bits, dtype=dt, workspace=0x10000 * 256, workspace_bytes=have)
        a.u8_scale[:] = (1 / 255,) * 3
        assert lib.tclb200_tcl_forward_host(ctypes.byref(a), None) == 1
        assert b"tclb200_host_workspace_bytes_cl" in lib.tclb200_last_error()


def test_layout_refusals_before_any_cuda_call(tcl, arrays):
    lib = tcl._cabi.lib()
    a = _host_args(tcl, arrays, channels_last=CL_FF, ff=None)              # a layout for a flow that is not there
    assert lib.tclb200_tcl_forward_host(ctypes.byref(a), None) == 1
    assert b"CL_FF without ff" in lib.tclb200_last_error()
    a = _host_args(tcl, arrays, channels_last=CL_FRAMES, C=65)              # the de-interleave's channel limit
    assert lib.tclb200_tcl_forward_host(ctypes.byref(a), None) == 3
    assert b"64 channels" in lib.tclb200_last_error()
    a = _host_args(tcl, arrays, channels_last=CL_FRAMES | CL_BF, dtype=U8, C=1)   # the uint8 rules still apply
    a.u8_scale[:] = (1 / 255,) * 3
    assert lib.tclb200_tcl_forward_host(ctypes.byref(a), None) == 1
    assert b"C == 3" in lib.tclb200_last_error()
