"""CPU suite of the kept-pixel sums (ABI v9): the new entry points and struct fields, their sizing, and the refusals that
happen before any CUDA call."""
import ctypes
import os
import re

import numpy as np
import pytest

from conftest import ROOT


def test_new_symbols_are_declared_exported_and_mirrored(tcl):
    text = open(os.path.join(ROOT, "include", "tcl_b200.h")).read()
    handle = ctypes.CDLL(tcl._cabi.LIB_PATH)
    for s in ("tclb200_scratch_bytes_kept", "tclb200_host_workspace_bytes_kept"):
        assert re.search(rf"\b{s}\s*\(", text), s
        assert hasattr(handle, s), s
        assert s in tcl._cabi.exported_symbols(), s
    assert tcl._cabi.ABI_VERSION == 9 and tcl._cabi.lib().tclb200_abi_version() == 9
    for name in ("warping_error_per_pair", "fused_forward", "temporal_error_host"):
        assert callable(getattr(tcl, name))


def test_kept_fields_close_the_structs():
    """pair_kept / total_kept are appended: the offsets of every older field stay where callers of v8 had them."""
    import tcl_b200
    ta, ha = tcl_b200._cabi.TclArgs, tcl_b200._cabi.HostArgs
    assert [f[0] for f in ta._fields_][-2:] == ["pair_kept", "total_kept"]
    assert [f[0] for f in ha._fields_][-1:] == ["pair_kept"]
    assert ta.pair_kept.offset > ta.u8_offset.offset and ha.pair_kept.offset > ha.channels_last.offset


@pytest.mark.parametrize("B,H,W", [(1, 8, 8), (3, 37, 53), (16, 256, 256), (2, 436, 1024)])
def test_kept_scratch_adds_one_partial_per_generic_tile(tcl, B, H, W):
    lib = tcl._cabi.lib()
    base, kept = lib.tclb200_scratch_bytes(B, H, W), lib.tclb200_scratch_bytes_kept(B, H, W)
    tiles = -(-W // 32) * -(-H // 8)
    assert kept - base == -(-(B * tiles * 8) // 256) * 256
    assert lib.tclb200_scratch_bytes_kept(0, H, W) == 0 and lib.tclb200_scratch_bytes_kept(B, 0, W) == 0


@pytest.mark.parametrize("cl", [0, 1, 7])
@pytest.mark.parametrize("P,F,chunk", [(4, 5, 0), (9, 10, 4), (300, 301, 0)])
def test_host_workspace_with_kept_sums(tcl, P, F, chunk, cl):
    lib = tcl._cabi.lib()
    C, H, W = 3, 64, 96
    for dt in (0, 1, 3):
        for with_mask in (0, 1):
            plain = lib.tclb200_host_workspace_bytes_cl(P, F, C, H, W, dt, chunk, with_mask, cl)
            kept = lib.tclb200_host_workspace_bytes_kept(P, F, C, H, W, dt, chunk, with_mask, cl)
            c = min(chunk if chunk > 0 else P, P)   # (the default chunk of a 64 x 96 flow is 128 pairs, capped at P)
            c = min(c, 128)
            extra_scratch = lib.tclb200_scratch_bytes_kept(c, H, W) - lib.tclb200_scratch_bytes(c, H, W)
            assert kept == plain + extra_scratch + -(-(8 * P) // 256) * 256
    # the entries without kept sums keep their values
    assert lib.tclb200_host_workspace_bytes(P, F, C, H, W, 0, chunk, 0) == lib.tclb200_host_workspace_bytes_cl(P, F, C, H, W, 0, chunk, 0, 0)
    assert lib.tclb200_host_workspace_bytes_kept(0, F, C, H, W, 0, chunk, 0, cl) == 0
    assert lib.tclb200_host_workspace_bytes_kept(P, F, C, H, W, 0, chunk, 0, 8) == 0   # unknown layout bit


def _args(tcl):
    """A valid reducing call on fake device pointers: everything the checks before the first CUDA call look at."""
    a = tcl._cabi.TclArgs()
    fake = ctypes.c_void_p(1 << 20)
    a.bf = a.ff = a.prev = a.cur = fake
    a.B, a.C, a.H, a.W = 2, 3, 16, 64
    a.flags = tcl._cabi.OCC | tcl._cabi.MOB
    a.pair_sums = fake
    a.pair_kept = fake
    a.scratch = fake
    a.scratch_bytes = tcl._cabi.lib().tclb200_scratch_bytes_kept(2, 16, 64)
    return a


def test_kept_sums_without_a_reduction_are_refused(tcl):
    lib = tcl._cabi.lib()
    a = _args(tcl)
    a.pair_sums = None
    assert lib.tclb200_tcl_forward(ctypes.byref(a), None) == 1
    assert b"pair_kept / total_kept need a reduction" in lib.tclb200_last_error()
    a = _args(tcl)
    a.pair_kept, a.total_kept = None, ctypes.c_void_p(1 << 20)
    a.pair_sums, a.cur = None, None
    a.mask_out = ctypes.c_void_p(1 << 20)
    assert lib.tclb200_tcl_forward(ctypes.byref(a), None) == 1
    assert b"need a reduction" in lib.tclb200_last_error()


def test_kept_sums_with_a_scratch_sized_for_the_plain_call_are_refused(tcl):
    lib = tcl._cabi.lib()
    a = _args(tcl)
    a.scratch_bytes = lib.tclb200_scratch_bytes(2, 16, 64)
    assert lib.tclb200_tcl_forward(ctypes.byref(a), None) == 1
    assert b"tclb200_scratch_bytes_kept" in lib.tclb200_last_error()
    a.scratch = None
    assert lib.tclb200_tcl_forward(ctypes.byref(a), None) == 1
    assert b"tclb200_scratch_bytes_kept" in lib.tclb200_last_error()


def test_host_entry_refuses_a_workspace_without_room_for_kept_sums(tcl):
    lib = tcl._cabi.lib()
    P, F, C, H, W = 2, 3, 3, 8, 8
    bf = np.zeros((P, 2, H, W), np.float32); fr = np.zeros((F, C, H, W), np.float32)
    pi = np.array([0, 1], np.int32); ci = np.array([1, 2], np.int32)
    kept = np.zeros(P, np.float64)
    a = tcl._cabi.HostArgs()
    a.P, a.F, a.C, a.H, a.W = P, F, C, H, W
    a.bf, a.frames, a.prev_index, a.cur_index = bf.ctypes.data, fr.ctypes.data, pi.ctypes.data, ci.ctypes.data
    a.pair_kept = kept.ctypes.data            # (kept sums alone are something to return)
    a.workspace = ctypes.c_void_p(1 << 20)
    a.workspace_bytes = lib.tclb200_host_workspace_bytes_cl(P, F, C, H, W, 0, 0, 0, 0)
    assert lib.tclb200_tcl_forward_host(ctypes.byref(a), None) == 1
    assert b"tclb200_host_workspace_bytes_kept" in lib.tclb200_last_error()

