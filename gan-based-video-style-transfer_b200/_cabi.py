"""ctypes binding of ``csrc/libtcl_b200.so`` (the C ABI declared in ``include/tcl_b200.h``).

There is deliberately no fallback of any kind: if the shared library is missing, cannot be
loaded, or reports a different ABI version, importing the compute wrappers raises.  Tensors are
handed over as raw device pointers (``Tensor.data_ptr()``) plus the current CUDA stream handle.
"""
import ctypes
import os
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(_HERE, "csrc")
LIB_PATH = os.environ.get("TCL_B200_LIB") or os.path.join(CSRC, "libtcl_b200.so")  # env override: tuning sweeps only
HEADER = os.path.join(os.path.dirname(_HERE), "include", "tcl_b200.h")
ABI_VERSION = 9

# enums mirrored from include/tcl_b200.h
F32, BF16, U8 = 0, 1, 3
OCC, MOB, VALIDITY = 1, 2, 4
L2, L1 = 0, 1
FIN_MEAN, FIN_RMSE = 0, 1
CL_FRAMES, CL_FF, CL_BF = 1, 2, 4

NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
              "-Xcompiler", "-fPIC", "-shared"]
SOURCES = ["tcl_kernels.cu", "tcl_host.cu", "tcl_cv2.cu", "tcl_agg.cu", "tcl_chain.cu"]
HEADERS = ["tcl_math.cuh", "tcl_common.cuh"]


class TclArgs(ctypes.Structure):
    """``tclb200_tcl_args`` (include/tcl_b200.h)."""
    _fields_ = [
        ("ff", ctypes.c_void_p), ("bf", ctypes.c_void_p), ("mask_in", ctypes.c_void_p),
        ("prev", ctypes.c_void_p), ("cur", ctypes.c_void_p),
        ("warp_out", ctypes.c_void_p), ("mask_out", ctypes.c_void_p), ("blend_out", ctypes.c_void_p),
        ("pair_sums", ctypes.c_void_p), ("total_sums", ctypes.c_void_p),
        ("pair_vals", ctypes.c_void_p), ("total_val", ctypes.c_void_p),
        ("near_threshold", ctypes.c_void_p),
        ("scratch", ctypes.c_void_p), ("scratch_bytes", ctypes.c_size_t),
        ("B", ctypes.c_int), ("C", ctypes.c_int), ("H", ctypes.c_int), ("W", ctypes.c_int),
        ("dtype", ctypes.c_int), ("flags", ctypes.c_int), ("loss", ctypes.c_int), ("finalize", ctypes.c_int),
        ("prev_index", ctypes.c_void_p), ("cur_index", ctypes.c_void_p),
        ("n_prev_frames", ctypes.c_int), ("n_cur_frames", ctypes.c_int),
        ("ff_plane_stride", ctypes.c_size_t), ("ff_batch_stride", ctypes.c_size_t),
        ("bf_plane_stride", ctypes.c_size_t), ("bf_batch_stride", ctypes.c_size_t),
        ("bf_index", ctypes.c_void_p), ("ff_index", ctypes.c_void_p),
        ("n_bf_fields", ctypes.c_int), ("n_ff_fields", ctypes.c_int), ("pair_group", ctypes.c_int),
        ("row_begin", ctypes.c_int), ("row_end", ctypes.c_int),
        ("u8_scale", ctypes.c_float * 3), ("u8_offset", ctypes.c_float * 3),
        ("pair_kept", ctypes.c_void_p), ("total_kept", ctypes.c_void_p),
    ]


class HostArgs(ctypes.Structure):
    """``tclb200_host_args`` (include/tcl_b200.h): every pointer is a HOST pointer except ``workspace``."""
    _fields_ = [
        ("ff", ctypes.c_void_p), ("bf", ctypes.c_void_p), ("mask_in", ctypes.c_void_p), ("frames", ctypes.c_void_p),
        ("prev_index", ctypes.c_void_p), ("cur_index", ctypes.c_void_p),
        ("pair_vals", ctypes.c_void_p), ("pair_sums", ctypes.c_void_p),
        ("workspace", ctypes.c_void_p), ("workspace_bytes", ctypes.c_size_t),
        ("P", ctypes.c_int), ("F", ctypes.c_int), ("C", ctypes.c_int), ("H", ctypes.c_int), ("W", ctypes.c_int),
        ("dtype", ctypes.c_int), ("flags", ctypes.c_int), ("loss", ctypes.c_int), ("finalize", ctypes.c_int),
        ("chunk_pairs", ctypes.c_int), ("frame_slots", ctypes.c_int),
        ("u8_scale", ctypes.c_float * 3), ("u8_offset", ctypes.c_float * 3),
        ("channels_last", ctypes.c_int),
        ("pair_kept", ctypes.c_void_p),
    ]


def _is_product_build(info):
    """True for a library compiled with the default configuration (no TCL_HOT_ONLY / TCL_DIAG / TCL_TRACE tuning macros)."""
    return all(tok in info.split() for tok in ("hot_only=0", "diag=0", "trace=0", f"abi={ABI_VERSION}"))


def _existing_lib_is_product_build():
    try:
        h = ctypes.CDLL(LIB_PATH)
        h.tclb200_build_info.restype = ctypes.c_char_p
        return _is_product_build(h.tclb200_build_info().decode())
    except Exception:
        return False


def build(force=False, verbose=False):
    """nvcc the kernels for sm_100a, in-tree (cross-compiles without a GPU): one object per source (stale ones only,
    compiled in parallel), then one link into ``libtcl_b200.so``."""
    deps_common = [os.path.join(CSRC, h) for h in HEADERS] + [HEADER]
    all_inputs = [os.path.join(CSRC, src) for src in SOURCES] + deps_common
    if (not force and os.path.exists(LIB_PATH)
            and all(os.path.getmtime(LIB_PATH) >= os.path.getmtime(d) for d in all_inputs)
            and (os.environ.get("TCL_B200_LIB") or _existing_lib_is_product_build())):
        return LIB_PATH   # up to date (also when the intermediate objects did not travel with the library)
    if os.path.exists(LIB_PATH) and not os.environ.get("TCL_B200_LIB") and not _existing_lib_is_product_build():
        force = True      # a library with another ABI or built with tuning macros: mtimes cannot tell, its build info can
    compile_flags = [f for f in NVCC_FLAGS if f != "-shared"]
    objs, jobs = [], []
    for src in SOURCES:
        path = os.path.join(CSRC, src)
        obj = os.path.join(CSRC, os.path.splitext(src)[0] + ".o")
        objs.append(obj)
        stale = (force or not os.path.exists(obj)
                 or any(os.path.getmtime(obj) < os.path.getmtime(d) for d in [path] + deps_common))
        if stale:
            cmd = ["nvcc"] + compile_flags + (["-Xptxas", "-v"] if verbose else []) + ["-c", "-o", obj, path]
            jobs.append((cmd, subprocess.Popen(cmd, cwd=CSRC)))
    for cmd, proc in jobs:
        if proc.wait() != 0:
            raise subprocess.CalledProcessError(proc.returncode, cmd)
    if jobs or not os.path.exists(LIB_PATH) or any(os.path.getmtime(LIB_PATH) < os.path.getmtime(o) for o in objs):
        subprocess.run(["nvcc", "-gencode", "arch=compute_100a,code=sm_100a", "-shared", "-o", LIB_PATH] + objs,
                       check=True, cwd=CSRC)
    return LIB_PATH


_c = ctypes
_vp, _i = ctypes.c_void_p, ctypes.c_int
_PROTOTYPES = {
    "tclb200_abi_version": (_c.c_int, []),
    "tclb200_last_error": (_c.c_char_p, []),
    "tclb200_build_info": (_c.c_char_p, []),
    "tclb200_scratch_bytes": (_c.c_size_t, [_i, _i, _i]),
    "tclb200_scratch_bytes_kept": (_c.c_size_t, [_i, _i, _i]),
    "tclb200_gradient": (_c.c_int, [_vp, _vp, _i, _i, _i, _vp]),
    "tclb200_gradient_strided": (_c.c_int, [_vp, _c.c_size_t, _vp, _i, _i, _i, _vp]),
    "tclb200_warp": (_c.c_int, [_vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _vp]),
    "tclb200_warp_backward": (_c.c_int, [_vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _vp]),
    "tclb200_fbcheck": (_c.c_int, [_vp, _vp, _vp, _i, _i, _i, _i, _vp, _vp]),
    "tclb200_tcl_forward": (_c.c_int, [_c.POINTER(TclArgs), _vp]),
    "tclb200_host_workspace_bytes": (_c.c_size_t, [_i, _i, _i, _i, _i, _i, _i, _i]),
    "tclb200_host_workspace_bytes_cl": (_c.c_size_t, [_i, _i, _i, _i, _i, _i, _i, _i, _i]),
    "tclb200_host_workspace_bytes_kept": (_c.c_size_t, [_i, _i, _i, _i, _i, _i, _i, _i, _i]),
    "tclb200_tcl_forward_host": (_c.c_int, [_c.POINTER(HostArgs), _vp]),
    "tclb200_tcl_backward": (_c.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _vp]),
    "tclb200_tcl_backward_scaled": (_c.c_int, [_vp, _vp, _vp, _vp, _vp, _c.c_float, _vp, _vp, _i, _i, _i, _i, _i, _i, _vp]),
    "tclb200_backward_workspace_bytes": (_c.c_size_t, [_i, _i, _i, _i, _i]),
    "tclb200_warp_backward_dt": (_c.c_int, [_vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _vp, _c.c_size_t, _vp]),
    "tclb200_tcl_backward_dt": (_c.c_int, [_vp, _vp, _vp, _vp, _vp, _c.c_float, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _vp,
                                           _c.c_size_t, _vp]),
    "tclb200_hwc_split": (_c.c_int, [_vp, _i, _i, _i, _i, _i, _vp, _vp, _vp, _vp]),
    "tclb200_occlusion_u8_to_mask": (_c.c_int, [_vp, _vp, _c.c_size_t, _vp]),
    "tclb200_upsample_flow": (_c.c_int, [_vp, _vp, _vp, _i, _i, _i, _vp]),
    "tclb200_cv2_remap": (_c.c_int, [_vp, _vp, _vp, _i, _i, _i, _i, _vp]),
    "tclb200_cv2_fb_check": (_c.c_int, [_vp, _vp, _vp, _i, _i, _i, _i, _i, _vp, _vp]),
    "tclb200_reconet_scratch_bytes": (_c.c_size_t, [_i, _i, _i]),
    "tclb200_reconet_loss": (_c.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _c.c_size_t, _i, _i, _i, _vp]),
    "tclb200_ruder_input": (_c.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _vp]),
    "tclb200_pack_sequence_sums": (_c.c_int, [_vp, _vp, _vp, _i, _i, _c.c_double, _vp, _vp]),
    "tclb200_unpack_sequence_means": (_c.c_int, [_vp, _i, _vp, _vp]),
    "tclb200_debug_force_generic": (None, [_i]),
    "tclb200_debug_tile_stats": (_c.c_int, [_vp, _i]),
    "tclb200_debug_launch_count": (_c.c_ulonglong, [_i]),
}

_lib = None


class TclB200Error(RuntimeError):
    pass


def lib():
    """Load (once) and return the C-ABI library; raises if it is not there."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise TclB200Error(
            f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(nvcc, sm_100a). There is no CPU or PyTorch fallback for this path.")
    handle = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in _PROTOTYPES.items():
        fn = getattr(handle, name)  # AttributeError here = the library does not export the header's symbol
        fn.restype, fn.argtypes = res, args
    got = handle.tclb200_abi_version()
    if got != ABI_VERSION:
        raise TclB200Error(f"ABI mismatch: library reports {got}, wrappers expect {ABI_VERSION}")
    info = handle.tclb200_build_info().decode()
    if not os.environ.get("TCL_B200_LIB") and not _is_product_build(info):
        raise TclB200Error(f"{LIB_PATH} was built with tuning macros ({info}); rebuild it with _cabi.build(force=True) "
                           "(tuning builds are loaded by name through TCL_B200_LIB only)")
    _lib = handle
    return _lib


def exported_symbols():
    return list(_PROTOTYPES)


def check(status):
    if status != 0:
        msg = lib().tclb200_last_error().decode("utf-8", "replace")
        raise TclB200Error(f"tcl_b200 call failed (status {status}): {msg}")
