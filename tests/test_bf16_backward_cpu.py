"""CPU suite of the bf16 backward entries (ABI v6): exported, validated before any CUDA call, workspace sizing, and the
fp32 backward kernels' instructions unchanged by the frame-type template parameter."""
import ctypes
import os
import re
import shutil
import subprocess
import sys

import pytest

from conftest import ROOT

F32, BF16 = 0, 1
NEW = ("tclb200_backward_workspace_bytes", "tclb200_warp_backward_dt", "tclb200_tcl_backward_dt")


def test_new_entries_are_declared_and_exported(tcl):
    handle = ctypes.CDLL(tcl._cabi.LIB_PATH)
    for s in NEW:
        assert hasattr(handle, s)
        assert s in tcl._cabi.exported_symbols()


def test_workspace_bytes(tcl):
    lib = tcl._cabi.lib()
    assert lib.tclb200_backward_workspace_bytes(16, 3, 256, 256, F32) == 0
    assert lib.tclb200_backward_workspace_bytes(16, 3, 256, 256, BF16) >= 16 * 3 * 256 * 256 * 4
    assert lib.tclb200_backward_workspace_bytes(1, 5, 37, 53, BF16) >= 5 * 37 * 53 * 4
    assert lib.tclb200_backward_workspace_bytes(0, 3, 8, 8, BF16) == 0
    assert lib.tclb200_backward_workspace_bytes(1, 3, 8, 8, 7) == 0


def _fake(n):
    """Host addresses that stand in for device pointers: validation fails before anything dereferences them."""
    return ctypes.c_void_p(0x10000 * n)


def test_warp_backward_dt_validation_without_gpu(tcl):
    lib = tcl._cabi.lib()
    go, x, f, gx, gf = (_fake(i) for i in range(1, 6))
    call = lambda dt, gx_, ws, nbytes: lib.tclb200_warp_backward_dt(go, x, f, gx_, gf, 2, 3, 8, 8, dt, 0, ws, nbytes, None)
    assert lib.tclb200_warp_backward_dt(None, x, f, gx, gf, 2, 3, 8, 8, BF16, 0, None, 0, None) == 1
    assert b"required" in lib.tclb200_last_error()
    assert call(2, gx, None, 0) == 1                                      # fp16 frames: not implemented
    assert b"dtype" in lib.tclb200_last_error()
    assert call(BF16, gx, None, 0) == 1                                   # grad_x of bf16 frames without a workspace
    assert b"workspace" in lib.tclb200_last_error()
    need = lib.tclb200_backward_workspace_bytes(2, 3, 8, 8, BF16)
    assert call(BF16, gx, _fake(7), need - 4) == 1                        # too small
    assert b"workspace" in lib.tclb200_last_error() and str(need).encode() in lib.tclb200_last_error()
    assert call(BF16, gx, ctypes.c_void_p(0x70004), need) == 1            # misaligned
    assert b"aligned" in lib.tclb200_last_error()


def test_tcl_backward_dt_validation_without_gpu(tcl):
    lib = tcl._cabi.lib()
    bf, m, p, c, s, gp, gc = (_fake(i) for i in range(1, 8))

    def call(dt, gp_, ws, nbytes, loss=0):
        return lib.tclb200_tcl_backward_dt(bf, m, p, c, s, 1.0, gp_, gc, 2, 3, 8, 8, dt, 0, loss, ws, nbytes, None)
    assert lib.tclb200_tcl_backward_dt(bf, m, p, c, None, 1.0, gp, gc, 2, 3, 8, 8, BF16, 0, 0, None, 0, None) == 1
    assert b"grad_scale" in lib.tclb200_last_error()
    assert call(BF16, gp, None, 0, loss=5) == 1
    assert b"loss" in lib.tclb200_last_error()
    assert call(-1, gp, None, 0) == 1
    assert b"dtype" in lib.tclb200_last_error()
    assert call(BF16, gp, None, 0) == 1
    assert b"workspace" in lib.tclb200_last_error() and b"grad_prev" in lib.tclb200_last_error()
    # the existing fp32 entries validate exactly as before
    assert lib.tclb200_tcl_backward_scaled(bf, m, p, c, None, 1.0, gp, gc, 2, 3, 8, 8, 0, 0, None) == 1
    assert b"grad_scale" in lib.tclb200_last_error()
    assert lib.tclb200_warp_backward(None, p, bf, gp, None, 2, 3, 8, 8, 0, None) == 1
    assert b"required" in lib.tclb200_last_error()


# SHA-256 of the instruction text (tools/sass_diff.py --digest) of every fp32 backward kernel as CUDA 12.9's ptxas compiles
# it.  They are the digests of the kernels before the frame type became a template parameter: the fp32 instantiations must
# stay instruction for instruction what they were.
FP32_BACKWARD_SASS_CUDA_12_9 = {
    "void tcl::warp_backward_kernel<false, 0>(tcl::BwdParams)": "57f8107b6b28bfb373d885961ff6ef489f9b192d597559d7b61f81136b85131e",
    "void tcl::warp_backward_kernel<false, 2>(tcl::BwdParams)": "35f96dc2b53e5abf927faf595e720293fe99d0d6d49c2eeebab7d4da7fb587d7",
    "void tcl::warp_backward_kernel<false, 3>(tcl::BwdParams)": "ad53e73bbd4dfc3f986906172acde71ca03edda9c9fa6aa874f53f0e4ad119aa",
    "void tcl::warp_backward_kernel<true, 0>(tcl::BwdParams)": "0218e30879b1fcbdce969478832a726031c66e6b77a840d5ba5c8eece927061c",
    "void tcl::warp_backward_kernel<true, 3>(tcl::BwdParams)": "36e9042d07ced714247a28a743757eddd32163aef68bd71d4311be44004ffac0",
}


def test_fp32_backward_sass_is_unchanged(tcl):
    if shutil.which("cuobjdump") is None or shutil.which("nvcc") is None or shutil.which("c++filt") is None:
        pytest.skip("cuobjdump / nvcc / c++filt not available")
    release = re.search(r"release (\d+\.\d+)", subprocess.run(["nvcc", "--version"], capture_output=True, text=True).stdout)
    if not release or release.group(1) != "12.9":
        pytest.skip("the pinned digests are those of CUDA 12.9's ptxas")
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    try:
        import sass_diff
    finally:
        sys.path.pop(0)
    got = {sass_diff.fp32_key(k): sass_diff.digest(v)
           for k, v in sass_diff.kernels(tcl._cabi.build(), "warp_backward_kernel").items() if "__nv_bfloat16" not in k}
    assert got == FP32_BACKWARD_SASS_CUDA_12_9
