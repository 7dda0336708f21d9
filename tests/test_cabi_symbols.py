"""CPU suite: the C-ABI shared library builds, loads and exports every symbol include/*.h declares.
No compute is attempted here (no GPU); argument validation that happens before any CUDA call is."""
import ctypes
import glob
import os
import re

import pytest

from conftest import ROOT


def declared_symbols():
    names = set()
    for h in glob.glob(os.path.join(ROOT, "include", "*.h")):
        text = re.sub(r"/\*.*?\*/", "", open(h).read(), flags=re.S)
        names |= set(re.findall(r"\b(tclb200_[a-z0-9_]+)\s*\(", text))
    return sorted(names)


def test_header_declares_the_expected_entry_points():
    syms = declared_symbols()
    for s in ("tclb200_abi_version", "tclb200_last_error", "tclb200_scratch_bytes", "tclb200_gradient", "tclb200_warp",
              "tclb200_warp_backward", "tclb200_fbcheck", "tclb200_tcl_forward", "tclb200_tcl_backward"):
        assert s in syms


def test_library_exports_every_declared_symbol(tcl):
    handle = ctypes.CDLL(tcl._cabi.LIB_PATH)
    for s in declared_symbols():
        assert hasattr(handle, s), f"{s} declared in include/ but not exported"
    assert set(tcl._cabi.exported_symbols()) <= set(declared_symbols())
    assert tcl._cabi.lib().tclb200_abi_version() == tcl._cabi.ABI_VERSION


def test_header_version_matches_wrappers(tcl):
    text = open(os.path.join(ROOT, "include", "tcl_b200.h")).read()
    assert int(re.search(r"#define TCLB200_ABI_VERSION (\d+)", text).group(1)) == tcl._cabi.ABI_VERSION
    for name in ("F32", "BF16", "OCC", "MOB", "VALIDITY", "L2", "L1", "FIN_MEAN", "FIN_RMSE"):
        assert int(re.search(rf"#define TCLB200_{name} (\d+)", text).group(1)) == getattr(tcl._cabi, name)


@pytest.mark.parametrize("struct,mirror", [("tclb200_tcl_args", "TclArgs"), ("tclb200_host_args", "HostArgs")])
def test_struct_layout_matches_header(tcl, struct, mirror):
    text = open(os.path.join(ROOT, "include", "tcl_b200.h")).read()
    body = re.search(r"typedef struct %s \{(.*?)\} %s;" % (struct, struct), text, re.S).group(1)
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    fields = []
    for decl in body.split(";"):
        decl = decl.strip()
        if not decl:
            continue
        names = decl.split(",")
        first = re.findall(r"[A-Za-z_][A-Za-z0-9_]*", names[0])[-1]
        fields.append(first)
        fields += [n.strip().lstrip("*").strip() for n in names[1:]]
    assert fields == [f[0] for f in getattr(tcl._cabi, mirror)._fields_]


def test_argument_validation_without_gpu(tcl):
    lib = tcl._cabi.lib()
    assert lib.tclb200_scratch_bytes(0, 10, 10) == 0
    assert lib.tclb200_scratch_bytes(16, 256, 256) > 0
    assert lib.tclb200_tcl_forward(None, None) == 1                      # TCLB200_ERR_INVALID
    assert b"NULL" in lib.tclb200_last_error()
    assert lib.tclb200_gradient(None, None, 1, 4, 4, None) == 1
    assert lib.tclb200_warp(None, None, None, 1, 3, 4, 4, 0, 0, None) == 1
    assert lib.tclb200_fbcheck(None, None, None, 1, 4, 4, 3, None, None) == 1
    a = tcl._cabi.TclArgs()
    a.B, a.C, a.H, a.W = 1, 3, 0, 4
    assert lib.tclb200_tcl_forward(ctypes.byref(a), None) == 1
    a.H = 4
    assert lib.tclb200_tcl_forward(ctypes.byref(a), None) == 1           # bf missing
    assert b"bf" in lib.tclb200_last_error()


def test_host_entry_validation_without_gpu(tcl):
    import numpy as np
    lib = tcl._cabi.lib()
    assert lib.tclb200_host_workspace_bytes(0, 2, 3, 8, 8, 0, 0, 0) == 0
    small = lib.tclb200_host_workspace_bytes(4, 5, 3, 64, 64, 0, 0, 0)
    # frame bank + 3 ring slots of two flows each, at least
    assert small >= 5 * 3 * 64 * 64 * 4 + 3 * 2 * 4 * 2 * 64 * 64 * 4
    assert lib.tclb200_host_workspace_bytes(4, 5, 3, 64, 64, 0, 0, 1) > small          # + dataset-mask ring
    assert lib.tclb200_host_workspace_bytes(4, 5, 3, 64, 64, 1, 0, 0) < small          # bf16 frame bank
    assert lib.tclb200_tcl_forward_host(None, None) == 1
    a = tcl._cabi.HostArgs()
    a.P, a.F, a.C, a.H, a.W = 1, 2, 3, 8, 8
    assert lib.tclb200_tcl_forward_host(ctypes.byref(a), None) == 1           # bf / frames / indices missing
    assert b"required" in lib.tclb200_last_error()
    bf = np.zeros((1, 2, 8, 8), np.float32); fr = np.zeros((2, 3, 8, 8), np.float32)
    pi = np.array([0], np.int32); ci = np.array([2], np.int32); out = np.zeros(1, np.float32)
    a.bf, a.frames, a.prev_index, a.cur_index, a.pair_vals = (bf.ctypes.data, fr.ctypes.data, pi.ctypes.data, ci.ctypes.data,
                                                              out.ctypes.data)
    assert lib.tclb200_tcl_forward_host(ctypes.byref(a), None) == 1           # cur_index outside [0, F)
    assert b"outside" in lib.tclb200_last_error()
    ci[0] = 1
    assert lib.tclb200_tcl_forward_host(ctypes.byref(a), None) == 1           # no workspace
    assert b"workspace" in lib.tclb200_last_error()


def test_build_info_names_the_tile_configuration_and_tuning_builds_are_refused(tcl, monkeypatch):
    info = tcl._cabi.lib().tclb200_build_info().decode()
    assert tcl._cabi._is_product_build(info), info
    for key in ("abi=%d" % tcl._cabi.ABI_VERSION, "th=", "bh=", "bw=", "ns=", "nb=", "cwarps=", "hot_only=0", "diag=0", "trace=0"):
        assert key in info
    assert not tcl._cabi._is_product_build(info.replace("hot_only=0", "hot_only=1"))
    assert not tcl._cabi._is_product_build(info.replace("diag=0", "diag=1"))
    assert not tcl._cabi._is_product_build(info.replace("abi=%d" % tcl._cabi.ABI_VERSION, "abi=4"))
    a = tcl._cabi.HostArgs()      # a clip without pairs is not an error (and needs no GPU)
    a.P, a.F = 0, 1
    assert tcl._cabi.lib().tclb200_tcl_forward_host(ctypes.byref(a), None) == 0


def test_missing_library_fails_loudly(tcl, monkeypatch):
    monkeypatch.setattr(tcl._cabi, "_lib", None)
    monkeypatch.setattr(tcl._cabi, "LIB_PATH", os.path.join(ROOT, "does", "not", "exist.so"))
    with pytest.raises(tcl._cabi.TclB200Error):
        tcl._cabi.lib()


def test_product_package_never_touches_the_oracle():
    pkg = os.path.join(ROOT, "gan-based-video-style-transfer_b200")
    for path in glob.glob(os.path.join(pkg, "**", "*"), recursive=True):
        if os.path.isfile(path) and path.endswith((".py", ".cu", ".cuh", ".h", ".cpp")):
            src = open(path).read()
            assert "import oracle" not in src and "from oracle" not in src and "tcl_oracle" not in src, path
            if path.endswith(".py"):
                assert "grid_sample(" not in src, f"{path}: the product path must not fall back to F.grid_sample"


def test_packed_products_are_not_contracted_in_the_shipped_library():
    """ptxas 12.9 fuses mul.rn.f32x2 + add.rn.f32x2 into one FFMA2 (one rounding where the reference has two).  The hot kernel
    therefore multiplies its coordinate products as scalars; in its SASS every `... * W - 1` FFMA2 (flowtools.py:28-29 + the
    sampler's unnormalise) must be matched by a separate packed `- 1` add -- a contracted product would show up as extra FFMA2s
    with a -1 addend and no FADD2."""
    import shutil
    import subprocess
    import tcl_b200
    if shutil.which("cuobjdump") is None:
        pytest.skip("cuobjdump not available")
    lib = tcl_b200._cabi.build()
    names = subprocess.run(["cuobjdump", "-elf", lib], capture_output=True, text=True).stdout
    hot = sorted({w for line in names.splitlines() for w in line.split()
                  if w.startswith("_ZN3tcl23fused_forward_ws_kernelIfLi2ELb1ELi3ELi1E") and "Li8ELb1E" in w and not w.startswith(".")})
    assert hot, "hot kernel not found in the library"
    sass = subprocess.run(["cuobjdump", "-sass", "-fun", hot[0], lib], capture_output=True, text=True).stdout
    fma_m1 = sum(1 for l in sass.splitlines() if "FFMA2" in l and ", -1 ;" in l)
    add_m1 = sum(1 for l in sass.splitlines() if "FADD2" in l and ", -1 ;" in l)
    assert fma_m1 > 0 and fma_m1 == add_m1, (fma_m1, add_m1)
