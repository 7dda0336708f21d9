"""Host-side mirror of the reference's flow-tools interface over the C-ABI CUDA library.

Every function keeps the name, argument meaning and result convention of the reference function
it replaces (upstream paths relative to the repository root):

* ``gradient(x)``                         utils/flowtools.py:12-16
* ``warp(x, f)``                          utils/flowtools.py:18-32 (+ the inline copies, SURVEY.md section 8 a2)
* ``fbcCheckTorch(ff, bf, device)``       utils/flowtools.py:34-58
* ``fbcCheckTorch_mob(ff, bf, device)``   methods/optimization-based/flowtools.py:34-58 (occlusion test off)
* ``fs_warp(x, flo)``                     methods/learning-based/fs_lib.py:5-39
* ``temporal_error(...)``                 utils/sintel_eval.py:104-110 minus RAFT and the generator (fused)
* ``temporal_loss(...)``                  StarGANv2AdvCon/core/solver.py:427-446, fs_ruder.py:97, MoGAN ...:280-281
* ``temporal_rmse_per_sample(...)``       utils/metrics/eval.py:137-138
* ``warp_blend(...)``                     methods/optimization-based/obst_eval.py:500
* ``generateMask(simg, prev, flow)``      ConGAN/models/cycle_gan_model.py:136-137 with the warp fused in
* ``temporal_error_host(...)``            the evaluation loop of utils/sintel_eval.py:206-222 with HOST tensors in and out

PyTorch is used for device memory, streams and autograd plumbing only; all arithmetic runs in
``csrc/tcl_kernels.cu``.  There is no CPU path: CPU tensors raise, like the reference's hard-coded
``.cuda()`` (flowtools.py:25) does on a box without a GPU.
"""
import ctypes

import torch

from . import _cabi
from ._cabi import BF16, F32, FIN_MEAN, FIN_RMSE, L1, L2, MOB, OCC, VALIDITY, HostArgs, TclArgs, check

_scratch_cache = {}


def _stream_handle():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _ptr(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else None


def _require_cuda(*tensors):
    for t in tensors:
        if t is not None and not t.is_cuda:
            raise RuntimeError("tcl_b200: expected CUDA tensors; this path has no CPU implementation "
                               "(the reference moves its grid with .cuda(), utils/flowtools.py:25)")


def _flow(f, name="flow"):
    if f.dim() != 4 or f.shape[1] != 2:
        raise RuntimeError(f"tcl_b200: {name} must be (B,2,H,W), got {tuple(f.shape)}")
    if f.dtype != torch.float32:
        f = f.float()
    return f.contiguous()


def _flow_view(f, name="flow"):
    """-> (tensor whose data_ptr is handed over, plane stride, pair stride) in elements; 0 strides = dense.

    A row-dense view of a larger tensor -- what ``InputPadder.unpad`` (utils/raft/raft/utils/utils.py:21-24) or
    ``flow_up[:,:,:H,:]`` (ConGAN/sintel_eval.py:61) make of RAFT's padded output when only rows were padded -- is read
    in place through its strides; anything else is made contiguous like before."""
    if f.dim() != 4 or f.shape[1] != 2:
        raise RuntimeError(f"tcl_b200: {name} must be (B,2,H,W), got {tuple(f.shape)}")
    B, _, H, W = f.shape
    if (f.dtype == torch.float32 and not f.is_contiguous() and H * W > 0 and f.stride(3) == 1 and f.stride(2) == W
            and f.stride(1) >= H * W and (B == 1 or f.stride(0) >= 2 * H * W)):
        return f, f.stride(1), (f.stride(0) if B > 1 else 2 * f.stride(1))
    return _flow(f, name), 0, 0


def _frame_dtype(t):
    if t.dtype == torch.float32:
        return F32
    if t.dtype == torch.bfloat16:
        return BF16
    raise RuntimeError(f"tcl_b200: frames must be float32 or bfloat16, got {t.dtype}")


def _scratch(B, H, W, device):
    """Zero-filled ticket/partials scratch, cached per (device, stream); kernels leave it zeroed."""
    need = _cabi.lib().tclb200_scratch_bytes(B, H, W)
    key = (device.index, torch.cuda.current_stream(device).cuda_stream)
    buf = _scratch_cache.get(key)
    if buf is None or buf.numel() < need:
        buf = torch.zeros(max(need, 1 << 16), dtype=torch.uint8, device=device)
        _scratch_cache[key] = buf
    return buf


# ------------------------------------------------------------------------------------------------
# reference-named functions
# ------------------------------------------------------------------------------------------------
def gradient(x):
    """Zero-padded central differences of (B,H,W) -> (2,B,H,W) = stack([dx, dy])."""
    _require_cuda(x)
    if x.dim() != 3:
        raise RuntimeError(f"tcl_b200: gradient expects (B,H,W), got {tuple(x.shape)}")
    x = x.float()
    B, H, W = x.shape
    # one channel of a (B,2,H,W) flow (the reference's gradient(bf[:,0,:,:]), flowtools.py:47): planes are contiguous, only
    # the batch stride differs -- handed to the kernel as is; anything else is made contiguous first
    if not (x.stride(2) == 1 and x.stride(1) == W and (B == 1 or x.stride(0) >= H * W)):
        x = x.contiguous()
    out = torch.empty((2, B, H, W), dtype=torch.float32, device=x.device)
    with torch.cuda.device(x.device):
        check(_cabi.lib().tclb200_gradient_strided(_ptr(x), x.stride(0) if B > 1 else H * W, _ptr(out), B, H, W, _stream_handle()))
    return out


def _warp_forward(x, f, flags, f_plane=0, f_batch=0):
    B, C, H, W = x.shape
    out = torch.empty_like(x)
    with torch.cuda.device(x.device):
        if not (f_plane or f_batch):
            check(_cabi.lib().tclb200_warp(_ptr(x), _ptr(f), _ptr(out), B, C, H, W, _frame_dtype(x), flags,
                                           _stream_handle()))
        else:   # a strided flow view: the same launch through the struct entry, which carries the strides
            a = TclArgs()
            a.bf, a.prev, a.warp_out = _ptr(f), _ptr(x), _ptr(out)
            a.B, a.C, a.H, a.W, a.dtype, a.flags = B, C, H, W, _frame_dtype(x), flags & VALIDITY
            a.bf_plane_stride, a.bf_batch_stride = f_plane, f_batch
            check(_cabi.lib().tclb200_tcl_forward(ctypes.byref(a), _stream_handle()))
    return out


class _WarpFn(torch.autograd.Function):
    """warp with the gradients F.grid_sample + the grid normalisation give the reference."""

    @staticmethod
    def forward(ctx, x, f, flags):
        ctx.flags = flags
        ctx.save_for_backward(x, f)
        return _warp_forward(x, f, flags)

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, grad_out):
        x, f = ctx.saved_tensors
        gx, gf = _warp_backward_raw(grad_out, x, f, ctx.flags, ctx.needs_input_grad[0], ctx.needs_input_grad[1])
        return gx, gf, None


def _backward_workspace(B, C, H, W, dtype, device):
    """The fp32 accumulator a bf16 grad_x / grad_prev is scattered into, from torch's caching allocator: stream-ordered
    reuse makes it safe to drop as soon as the launches are enqueued, and inside a CUDA graph capture it comes from the
    graph's pool."""
    nbytes = _cabi.lib().tclb200_backward_workspace_bytes(B, C, H, W, dtype)
    return torch.empty(nbytes, dtype=torch.uint8, device=device), nbytes


def _warp_backward_raw(grad_out, x, f, flags, need_x=True, need_f=True):
    """Autograd of ``warp`` / ``fs_lib.warp`` on raw tensors (``tclb200_warp_backward``): (grad_x, grad_f).

    bf16 ``x``: ``grad_out`` is read in bf16 and ``grad_x`` comes back in bf16 (``tclb200_warp_backward_dt``): the fp32
    gradients of the upcast frame, rounded once."""
    B, C, H, W = x.shape
    gx = torch.empty_like(x) if need_x else None
    gf = torch.empty_like(f) if need_f else None
    if x.dtype == torch.float32:
        go = grad_out.float().contiguous()
        with torch.cuda.device(x.device):
            check(_cabi.lib().tclb200_warp_backward(_ptr(go), _ptr(x), _ptr(f), _ptr(gx), _ptr(gf), B, C, H, W, flags, _stream_handle()))
        return gx, gf
    dt = _frame_dtype(x)
    go = grad_out.to(x.dtype).contiguous()
    with torch.cuda.device(x.device):
        ws, nbytes = _backward_workspace(B, C, H, W, dt, x.device) if need_x else (None, 0)
        check(_cabi.lib().tclb200_warp_backward_dt(_ptr(go), _ptr(x), _ptr(f), _ptr(gx), _ptr(gf), B, C, H, W, dt, flags, _ptr(ws),
                                                   nbytes, _stream_handle()))
    return gx, gf


def _warp(x, f, flags):
    _require_cuda(x, f)
    if x.dim() != 4:
        raise RuntimeError(f"tcl_b200: warp expects x of shape (B,C,H,W), got {tuple(x.shape)}")
    if f.dim() != 4 or f.shape[1] != 2:
        raise RuntimeError(f"tcl_b200: f must be (B,2,H,W), got {tuple(f.shape)}")
    if f.shape[0] != x.shape[0] or f.shape[2:] != x.shape[2:]:
        raise RuntimeError(f"tcl_b200: x {tuple(x.shape)} and flow {tuple(f.shape)} do not match")
    _frame_dtype(x)
    x = x.contiguous()
    if torch.is_grad_enabled() and (x.requires_grad or f.requires_grad):
        return _WarpFn.apply(x, _flow(f, "f"), flags)
    f, f_plane, f_batch = _flow_view(f, "f")
    return _warp_forward(x, f, flags, f_plane, f_batch)


def warp(x, f):
    """Bilinear zero-padded backward warp of ``x`` (B,C,H,W) by pixel flow ``f`` (B,2,H,W).

    Keeps the reference's sampling convention exactly (normalise by size-1, sample with
    align_corners=False), so zero flow is NOT the identity -- see SURVEY.md section 7 hard part 3.
    """
    return _warp(x, f, 0)


def fs_warp(x, flo):
    """fs_lib.warp: ``warp`` times the binarised (>= 0.9999) warp of an all-ones image."""
    return _warp(x, flo, VALIDITY)


def _fbcheck(ff, bf, flags, device, return_near=False):
    _require_cuda(bf)
    bf, bf_plane, bf_batch = _flow_view(bf, "bf")
    ff_plane = ff_batch = 0
    if flags & OCC:
        _require_cuda(ff)
        ff, ff_plane, ff_batch = _flow_view(ff, "ff")
        if ff.shape != bf.shape:
            raise RuntimeError(f"tcl_b200: ff {tuple(ff.shape)} and bf {tuple(bf.shape)} do not match")
    else:
        ff = None
    B, _, H, W = bf.shape
    mask = torch.empty((B, 1, H, W), dtype=torch.float32, device=bf.device)
    near = torch.zeros(1, dtype=torch.int64, device=bf.device) if return_near else None
    with torch.cuda.device(bf.device):
        if not (bf_plane or ff_plane):
            check(_cabi.lib().tclb200_fbcheck(_ptr(ff), _ptr(bf), _ptr(mask), B, H, W, flags, _ptr(near),
                                              _stream_handle()))
        else:   # strided flow views: the same launch through the struct entry, which carries the strides
            a = TclArgs()
            a.ff, a.bf, a.mask_out, a.near_threshold = _ptr(ff if ff is not None else bf), _ptr(bf), _ptr(mask), _ptr(near)
            a.B, a.H, a.W, a.flags = B, H, W, flags
            a.bf_plane_stride, a.bf_batch_stride = bf_plane, bf_batch
            a.ff_plane_stride, a.ff_batch_stride = (ff_plane, ff_batch) if ff is not None else (bf_plane, bf_batch)
            check(_cabi.lib().tclb200_tcl_forward(ctypes.byref(a), _stream_handle()))
    if device is not None and torch.device(device) != mask.device and torch.device(device).type != "cuda":
        mask = mask.to(device)
    return (mask, near) if return_near else mask


def fbcCheckTorch(ff, bf, device="cuda"):
    """Forward-backward consistency + motion-boundary mask (B,1,H,W) fp32 in {0,1}, no grad."""
    return _fbcheck(ff, bf, OCC | MOB, device)


def fbcCheckTorch_mob(ff, bf, device="cuda"):
    """The optimisation-based variant: motion-boundary test only (``ff`` is ignored)."""
    return _fbcheck(ff, bf, MOB, device)


def fbcheck_with_near_count(ff, bf, flags=OCC | MOB):
    """``fbcCheckTorch`` plus the count of pixels whose test margin is within 1e-6 of the threshold."""
    return _fbcheck(ff, bf, flags, None, return_near=True)


def upsample_flow(flow, mask):
    """RAFT's convex upsampling (utils/raft/raft/raft.py:72-83): flow (N,2,H,W), mask (N,576,H,W) -> (N,2,8H,8W).

    Drop-in for ``RAFT.upsample_flow`` (bind it with ``raft_model.upsample_flow = tcl_b200.upsample_flow``); one fused
    pass instead of softmax + unfold + mul + sum + permute.  No autograd (the reference uses it under ``no_grad``,
    utils/sintel_eval.py:55-58)."""
    _require_cuda(flow, mask)
    if flow.dim() != 4 or flow.shape[1] != 2:
        raise RuntimeError(f"tcl_b200: flow must be (N,2,H,W), got {tuple(flow.shape)}")
    N, _, H, W = flow.shape
    if mask.dim() != 4 or mask.shape != (N, 576, H, W):
        raise RuntimeError(f"tcl_b200: mask must be (N,576,H,W) = {(N, 576, H, W)}, got {tuple(mask.shape)}")
    flow, mask = flow.float().contiguous(), mask.float().contiguous()
    out = torch.empty((N, 2, 8 * H, 8 * W), dtype=torch.float32, device=flow.device)
    with torch.cuda.device(flow.device):
        check(_cabi.lib().tclb200_upsample_flow(_ptr(flow), _ptr(mask), _ptr(out), N, H, W, _stream_handle()))
    return out


# ------------------------------------------------------------------------------------------------
# fused path
# ------------------------------------------------------------------------------------------------
class FusedResult:
    """Device-resident results of one fused launch (nothing is synchronised)."""
    __slots__ = ("pair_vals", "total_val", "pair_sums", "total_sums", "warp", "mask", "blend", "near_threshold")

    def __init__(self):
        for s in self.__slots__:
            setattr(self, s, None)


def _index(idx, B, n_frames, name, validate=True):
    if idx is None:
        return None
    if idx.dim() != 1 or idx.numel() != B:
        raise RuntimeError(f"tcl_b200: {name} must hold one frame index per pair ({B}), got {tuple(idx.shape)}")
    if validate and idx.numel() and (int(idx.min()) < 0 or int(idx.max()) >= n_frames):   # (a device sync: skip with validate=False)
        raise RuntimeError(f"tcl_b200: {name} outside [0, {n_frames})")
    return idx.to(dtype=torch.int32).contiguous()


def fused_forward(bf, prev, cur, ff=None, mask=None, loss=L2, finalize=FIN_RMSE, flags=OCC | MOB,
                  want_warp=False, want_mask=False, want_blend=False, want_near=False, want_sums=True,
                  prev_index=None, cur_index=None, validate_index=True, bf_index=None, ff_index=None, pair_group=0, rows=None):
    """One launch: warp ``prev`` by ``bf``, build or read the mask, reduce the masked error against ``cur``.

    ``ff`` given -> the mask is computed (fbcCheckTorch semantics, tests per ``flags``);
    else ``mask`` given -> dataset mask (B,1,H,W); else no mask.  Returns a ``FusedResult``.

    Clip mode: with ``prev_index`` / ``cur_index`` (int tensors, one entry per pair) ``prev`` / ``cur`` are banks of
    frames (F,C,H,W) and pair b reads frame ``prev_index[b]`` / ``cur_index[b]`` -- a video stored once serves as
    ``cur`` of pair t and ``prev`` of pair t+1 (see ``temporal_error_clip``).

    Window mode: with ``bf_index`` / ``ff_index`` the flows are banks of fields as well and pair b reads field
    ``bf_index[b]`` / ``ff_index[b]`` (a field is the ``bf`` of one evaluation and the ``ff`` of the opposite one);
    ``pair_group`` interleaves the tiles of that many consecutive pairs (see ``temporal_error_window``).

    Band mode: ``rows=(r0, r1)`` evaluates target rows [r0, r1) of every pair only (inputs stay whole frames); the result
    carries ``pair_sums`` / ``total_sums`` but no means (see ``sharding.evaluate_banded``).
    """
    _require_cuda(bf, prev, cur, ff, mask, bf_index, ff_index)
    bf, bf_plane, bf_batch = _flow_view(bf, "bf")
    _, _, H, W = bf.shape
    B = bf.shape[0] if bf_index is None else int(bf_index.numel())
    ff, ff_plane, ff_batch = _flow_view(ff, "ff") if ff is not None else (None, 0, 0)
    bf_index = _index(bf_index, B, bf.shape[0], "bf_index", validate_index)
    ff_index = _index(ff_index, B, ff.shape[0], "ff_index", validate_index) if ff is not None else None
    if ff is not None and ff_index is None and ff.shape[0] != B:
        raise RuntimeError(f"tcl_b200: ff holds {ff.shape[0]} fields for {B} pairs (pass ff_index for a bank of fields)")
    if prev.dim() != 4 or (prev_index is None and prev.shape[0] != B) or prev.shape[2:] != bf.shape[2:]:
        raise RuntimeError(f"tcl_b200: prev {tuple(prev.shape)} does not match flow {tuple(bf.shape)}")
    if cur.dim() != 4 or cur.shape[1:] != prev.shape[1:] or cur.dtype != prev.dtype or (cur_index is None and cur.shape[0] != B):
        raise RuntimeError("tcl_b200: prev and cur must have the same frame shape and dtype")
    _require_cuda(prev_index, cur_index)
    prev_index = _index(prev_index, B, prev.shape[0], "prev_index", validate_index)
    cur_index = _index(cur_index, B, cur.shape[0], "cur_index", validate_index)
    if (want_warp or want_blend) and (prev_index is not None or cur_index is not None):
        out_like = torch.empty((B,) + tuple(prev.shape[1:]), dtype=prev.dtype, device=prev.device)
    else:
        out_like = None
    dt = _frame_dtype(prev)
    prev, cur = prev.contiguous(), cur.contiguous()
    C = prev.shape[1]
    dev = bf.device
    if mask is not None and ff is None:
        if mask.shape != (B, 1, H, W):
            raise RuntimeError(f"tcl_b200: mask must be (B,1,H,W), got {tuple(mask.shape)}")
        mask = mask.float().contiguous()
    else:
        mask = None
    res = FusedResult()
    if rows is not None:
        r0, r1 = int(rows[0]), int(rows[1])
        if not (0 <= r0 < r1 <= H):
            raise RuntimeError(f"tcl_b200: rows must satisfy 0 <= r0 < r1 <= H = {H}, got {rows}")
    if want_sums:
        f64 = torch.empty(B + 2, dtype=torch.float64, device=dev)
        res.pair_sums, res.total_sums = f64[:B], f64[B:]
        if rows is None:
            f32 = torch.empty(B + 1, dtype=torch.float32, device=dev)
            res.pair_vals, res.total_val = f32[:B], f32[B]
    if want_warp:
        res.warp = torch.empty_like(prev) if out_like is None else torch.empty_like(out_like)
    if want_mask:
        res.mask = torch.empty((B, 1, H, W), dtype=torch.float32, device=dev)
    if want_blend:
        res.blend = torch.empty_like(prev) if out_like is None else torch.empty_like(out_like)
    if want_near:
        res.near_threshold = torch.zeros(1, dtype=torch.int64, device=dev)
    with torch.cuda.device(dev):
        scratch = _scratch(B, H, W, dev) if want_sums else None
        a = TclArgs()
        a.ff, a.bf, a.mask_in, a.prev, a.cur = _ptr(ff), _ptr(bf), _ptr(mask), _ptr(prev), _ptr(cur)
        a.warp_out, a.mask_out, a.blend_out = _ptr(res.warp), _ptr(res.mask), _ptr(res.blend)
        if want_sums:
            a.pair_sums, a.total_sums = _ptr(res.pair_sums), _ptr(res.total_sums)
            a.pair_vals, a.total_val = _ptr(res.pair_vals), _ptr(res.total_val)
            a.scratch, a.scratch_bytes = _ptr(scratch), scratch.numel()
        a.near_threshold = _ptr(res.near_threshold)
        a.B, a.C, a.H, a.W = B, C, H, W
        a.dtype, a.flags, a.loss, a.finalize = dt, flags, loss, finalize
        a.prev_index, a.cur_index = _ptr(prev_index), _ptr(cur_index)
        a.n_prev_frames, a.n_cur_frames = prev.shape[0], cur.shape[0]
        a.ff_plane_stride, a.ff_batch_stride, a.bf_plane_stride, a.bf_batch_stride = ff_plane, ff_batch, bf_plane, bf_batch
        a.bf_index, a.ff_index = _ptr(bf_index), _ptr(ff_index)
        a.n_bf_fields, a.n_ff_fields = bf.shape[0], (ff.shape[0] if ff is not None else 0)
        a.pair_group = int(pair_group)
        if rows is not None:
            a.row_begin, a.row_end = r0, r1
        check(_cabi.lib().tclb200_tcl_forward(ctypes.byref(a), _stream_handle()))
    return res


def temporal_error(ff, bf, prev, cur):
    """``computeTCL`` minus RAFT and the generator: sqrt(mean((mask*(cur - warp(prev,bf)))**2)), 0-dim tensor."""
    return fused_forward(bf, prev, cur, ff=ff, finalize=FIN_RMSE).total_val


def temporal_error_per_pair(ff, bf, prev, cur):
    """Per-pair RMSE (B,) with the mask computed from (ff,bf) -- the batched form of ``computeTCL``."""
    return fused_forward(bf, prev, cur, ff=ff, finalize=FIN_RMSE).pair_vals


def temporal_error_clip(frames, ff, bf):
    """Per-pair RMSE (T-1,) over a clip of T stylised frames stored ONCE: pair i warps ``frames[i]`` by ``bf[i]`` and
    compares with ``frames[i+1]`` under the mask of (``ff[i]``, ``bf[i]``) -- the evaluation loop of
    utils/sintel_eval.py:206-222 for a deterministic generator.  Every frame is read from HBM once (28 instead of
    40 B/px): its second use comes out of L2."""
    T = frames.shape[0]
    if bf.shape[0] != T - 1:
        raise RuntimeError(f"tcl_b200: a clip of {T} frames has {T - 1} consecutive pairs, got {bf.shape[0]} flows")
    idx = torch.arange(T, dtype=torch.int32, device=frames.device)
    return fused_forward(bf, frames, frames, ff=ff, finalize=FIN_RMSE, prev_index=idx[:-1], cur_index=idx[1:],
                         validate_index=False).pair_vals


def window_evaluations(n_frames, window=4):
    """Index arrays of every directed evaluation of a clip's temporal windows (BASELINE config 4; the long-term pairs of
    utils/sintel_eval.py:84-86,216-222 generalised to both directions): for every target frame t and every source
    s = t-1 .. t-(window-1), "warp s into t" and "warp t into s".

    Flow bank layout the indices refer to: for j enumerating (t, d = t-s) with t ascending, d = 1 .. window-1, field 2j is
    flow(t -> s) (sampled on t's grid: the ``bf`` of warping s into t) and field 2j+1 is flow(s -> t).  Returns a dict of
    int32 CPU tensors ``prev_index, cur_index, bf_index, ff_index`` (one entry per evaluation), ``target`` / ``source`` /
    ``field_t`` / ``field_s`` (frames of field pair j) and ``group`` = 2 * (window-1), the evaluations per complete window;
    complete windows come first, so that ``pair_group=group`` keeps every target frame's evaluations together."""
    fields, full, part = [], [], []
    for t in range(1, n_frames):
        evs = []
        for d in range(1, window):
            s_ = t - d
            if s_ < 0:
                break
            j = len(fields)
            fields.append((t, s_))
            evs.append((s_, t, 2 * j, 2 * j + 1))       # warp s into t: prev = s, cur = t, bf = flow(t -> s), ff = flow(s -> t)
            evs.append((t, s_, 2 * j + 1, 2 * j))       # warp t into s
        (full if len(evs) == 2 * (window - 1) else part).extend(evs)
    evs = full + part
    col = lambda k: torch.tensor([e[k] for e in evs], dtype=torch.int32)
    return {"prev_index": col(0), "cur_index": col(1), "bf_index": col(2), "ff_index": col(3),
            "field_t": torch.tensor([f[0] for f in fields], dtype=torch.int32), "field_s": torch.tensor([f[1] for f in fields], dtype=torch.int32),
            "group": 2 * (window - 1), "n_complete": len(full)}


def temporal_error_window(frames, flow_bank, window=4, index=None, finalize=FIN_RMSE):
    """Temporal error of every directed evaluation of a clip's temporal windows in ONE launch, everything stored once:
    ``frames`` (T,C,H,W) fp32/bf16, ``flow_bank`` (2*J,2,H,W) in the layout of ``window_evaluations`` (``index`` = its
    result, computed when omitted).  Each frame is the ``cur`` of up to window-1 evaluations and the ``prev`` of as many,
    each flow field the ``bf`` of one and the ``ff`` of the opposite one; the tiles of a target frame's evaluations are
    interleaved (``pair_group``), so the re-reads are L2 hits: 4 frames + 6 fields per complete window of 6 evaluations
    instead of 12 frames + 12 fields.  Returns the per-evaluation values (E,) in the order of ``index``."""
    _require_cuda(frames, flow_bank)
    if index is None:
        index = window_evaluations(frames.shape[0], window)
    dev = frames.device
    to = lambda k: index[k].to(dev)
    res = fused_forward(flow_bank, frames, frames, ff=flow_bank, finalize=finalize, prev_index=to("prev_index"), cur_index=to("cur_index"),
                        bf_index=to("bf_index"), ff_index=to("ff_index"), pair_group=index["group"])
    return res.pair_vals


_host_ws_cache = {}


def free_workspaces():
    """Drop the cached device buffers (per-stream reduction scratch, the host entry's frame bank / flow ring).  They are
    re-allocated on demand; call this to hand the memory back to the caching allocator, e.g. after a one-off evaluation of a
    long clip.  The caches are plain dicts: like the reference's loops, the wrappers assume one Python thread per device."""
    _scratch_cache.clear()
    _host_ws_cache.clear()
    _loss_plans.clear()


def _host_tensor(t, name, dtype=None):
    if t is None:
        return None
    if t.is_cuda:
        raise RuntimeError(f"tcl_b200: {name} must be a host (CPU) tensor for the host-buffer entry")
    if dtype is not None and t.dtype != dtype:
        t = t.to(dtype)
    return t.contiguous()


def temporal_error_host(frames, ff, bf, prev_index=None, cur_index=None, mask=None, loss=L2, finalize=FIN_RMSE,
                        flags=OCC | MOB, chunk_pairs=0, device=None, sync=True, return_sums=False, max_device_frames=None):
    """The evaluation loop of utils/sintel_eval.py:206-222 (and solver.py:336-347) on HOST tensors.

    ``frames`` (F,C,H,W) fp32/bf16: the stylised frames of one or more clips, each stored once; ``ff`` / ``bf``
    (P,2,H,W) fp32; pair p warps ``frames[prev_index[p]]`` by ``bf[p]`` and compares with ``frames[cur_index[p]]``
    under the mask of (``ff[p]``, ``bf[p]``) -- or under ``mask[p]`` (P,1,H,W) when ``ff`` is None
    (utils/metrics/eval.py:137-138).  Default indices: the consecutive pairs of ONE clip (P = F-1).
    All tensors are CPU tensors (pinned memory runs at PCIe speed); the result is a pinned CPU tensor (P,) of per-pair
    values per ``finalize``.  One C-ABI call (``tclb200_tcl_forward_host``) pipelines H2D copies and fused launches
    on ``device`` (default: the current CUDA device); there is no CPU arithmetic anywhere.
    ``return_sums=True`` returns ``(values, sums)`` with the per-pair float64 sums S_p as well (for pooled statistics).
    ``max_device_frames``: device frame slots.  None = the whole frame bank stays resident when it takes at most a
    quarter of the free device memory, else a ring of as many frames as that quarter holds (long or 4K clips: a slot is
    reused once every chunk that reads its frame has completed; at least four chunks' worth of frames must fit).
    A clip without pairs (P == 0) returns empty results.
    """
    if not torch.cuda.is_available():
        raise RuntimeError("tcl_b200: temporal_error_host needs a CUDA device; this path has no CPU implementation")
    frames = _host_tensor(frames, "frames")
    dt = _frame_dtype(frames)
    bf = _host_tensor(bf, "bf", torch.float32)
    ff = _host_tensor(ff, "ff", torch.float32)
    mask = _host_tensor(mask, "mask", torch.float32) if ff is None else None
    if frames.dim() != 4 or bf.dim() != 4 or bf.shape[1] != 2 or bf.shape[2:] != frames.shape[2:]:
        raise RuntimeError(f"tcl_b200: frames {tuple(frames.shape)} / bf {tuple(bf.shape)} must be (F,C,H,W) / (P,2,H,W)")
    F_, C, H, W = frames.shape
    P = bf.shape[0]
    if ff is not None and ff.shape != bf.shape:
        raise RuntimeError(f"tcl_b200: ff {tuple(ff.shape)} and bf {tuple(bf.shape)} do not match")
    if mask is not None and tuple(mask.shape) != (P, 1, H, W):
        raise RuntimeError(f"tcl_b200: mask must be (P,1,H,W), got {tuple(mask.shape)}")
    if prev_index is None and cur_index is None:
        if P != F_ - 1:
            raise RuntimeError(f"tcl_b200: a clip of {F_} frames has {F_ - 1} consecutive pairs, got {P} flows")
        idx = torch.arange(F_, dtype=torch.int32)
        prev_index, cur_index = idx[:-1], idx[1:]
    prev_index = _host_tensor(prev_index, "prev_index", torch.int32)
    cur_index = _host_tensor(cur_index, "cur_index", torch.int32)
    if prev_index.numel() != P or cur_index.numel() != P:
        raise RuntimeError(f"tcl_b200: prev_index / cur_index must hold one frame index per pair ({P})")
    dev = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
    lib = _cabi.lib()
    if P == 0:
        out = torch.empty(0, dtype=torch.float32, pin_memory=True)
        return (out, torch.empty(0, dtype=torch.float64, pin_memory=True)) if return_sums else out
    slots = F_
    ws = _host_ws_cache.get(dev.index)
    with_mask = 1 if mask is not None else 0
    if max_device_frames is not None:
        slots = max(1, min(F_, int(max_device_frames)))
    elif ws is None or ws.numel() < lib.tclb200_host_workspace_bytes(P, F_, C, H, W, dt, chunk_pairs, with_mask):
        # only when a workspace has to be allocated: cudaMemGetInfo costs 1.5 ms at the median and 20-90 ms in one call of ten
        # (measured, tools/e2e_stall_probe.py) -- per step it was the whole difference between a 6 ms step and a 12 ms one
        frame_bytes = C * H * W * frames.element_size()
        free_b = torch.cuda.mem_get_info(dev)[0] + (ws.numel() if ws is not None else 0)
        if F_ * frame_bytes > free_b // 4:
            slots = max(1, min(F_, (free_b // 4) // frame_bytes))
    need = lib.tclb200_host_workspace_bytes(P, slots, C, H, W, dt, chunk_pairs, with_mask)
    if ws is None or ws.numel() < need:
        _host_ws_cache.pop(dev.index, None)
        ws = torch.empty(need, dtype=torch.uint8, device=dev)
        _host_ws_cache[dev.index] = ws
    out = torch.empty(P, dtype=torch.float32, pin_memory=True)
    sums = torch.empty(P, dtype=torch.float64, pin_memory=True) if return_sums else None
    a = HostArgs()
    a.ff, a.bf, a.mask_in, a.frames = _ptr(ff), _ptr(bf), _ptr(mask), _ptr(frames)
    a.prev_index, a.cur_index = _ptr(prev_index), _ptr(cur_index)
    a.pair_vals, a.pair_sums = _ptr(out), _ptr(sums)
    a.workspace, a.workspace_bytes = _ptr(ws), ws.numel()
    a.P, a.F, a.C, a.H, a.W = P, F_, C, H, W
    a.dtype, a.flags, a.loss, a.finalize, a.chunk_pairs = dt, flags, loss, finalize, chunk_pairs
    a.frame_slots = 0 if slots >= F_ else slots
    with torch.cuda.device(dev):
        stream = torch.cuda.current_stream()
        check(lib.tclb200_tcl_forward_host(ctypes.byref(a), ctypes.c_void_p(stream.cuda_stream)))
        if sync:
            stream.synchronize()
        else:   # the caller synchronises the stream; keep the host inputs alive until then
            out._tcl_keepalive = (frames, ff, bf, mask, prev_index, cur_index)
    return (out, sums) if return_sums else out


def temporal_rmse_per_sample(mask, cur, prev, flow):
    """FC2 metric: ((mask*(cur - warp(prev,flow)))**2).mean(dim=(1,2,3))**0.5 -> (N,)."""
    return fused_forward(flow, prev, cur, mask=mask, finalize=FIN_RMSE).pair_vals


def warp_blend(mask, prev, flow, img):
    """mask*warp(prev,flow) + (1-mask)*img in one pass (obst_eval.py:500)."""
    return fused_forward(flow, prev, img, mask=mask, want_blend=True, want_sums=False).blend


# The training loss is a ~30 us job called every iteration (solver.py:427-446, twice per step): its wrapper avoids every
# avoidable Python / dispatcher cost -- one argument struct per (device, stream) filled in place, the scratch looked up once,
# a single 4-byte result tensor, no device-context switch when the tensors' device is already current, one scalar op in backward.
_loss_plans = {}


class _LossPlan:
    __slots__ = ("args", "scratch", "scratch_bytes", "stream", "lib", "fwd", "bwd")

    def __init__(self, device, stream_handle):
        self.args = TclArgs()
        self.stream = ctypes.c_void_p(stream_handle)
        self.lib = _cabi.lib()
        self.fwd, self.bwd = self.lib.tclb200_tcl_forward, self.lib.tclb200_tcl_backward_scaled
        self.scratch, self.scratch_bytes = None, 0


def _loss_plan(device, B, H, W):
    handle = torch.cuda.current_stream(device).cuda_stream
    key = (device.index, handle)
    plan = _loss_plans.get(key)
    if plan is None:
        plan = _loss_plans[key] = _LossPlan(device, handle)
    need = plan.lib.tclb200_scratch_bytes(B, H, W)
    if plan.scratch is None or plan.scratch_bytes < need:
        plan.scratch = _scratch(B, H, W, device)
        plan.scratch_bytes = plan.scratch.numel()
        plan.args.scratch, plan.args.scratch_bytes = plan.scratch.data_ptr(), plan.scratch_bytes
    return plan


def _loss_forward(prev, cur, flow, mask, loss, flags):
    """mean masked error of the training loss: one launch pair, total only (no per-pair outputs)."""
    B, C, H, W = prev.shape
    dev = prev.device
    out = torch.empty((), dtype=torch.float32, device=dev)
    switch = torch.cuda.current_device() != dev.index
    if switch:
        ctx = torch.cuda.device(dev)
        ctx.__enter__()
    try:
        plan = _loss_plan(dev, B, H, W)
        a = plan.args
        a.bf, a.mask_in, a.prev, a.cur, a.total_val = flow.data_ptr(), mask.data_ptr(), prev.data_ptr(), cur.data_ptr(), out.data_ptr()
        a.B, a.C, a.H, a.W = B, C, H, W
        a.dtype, a.flags, a.loss, a.finalize = (F32 if prev.dtype == torch.float32 else BF16), flags, loss, FIN_MEAN
        rc = plan.fwd(ctypes.byref(a), plan.stream)
        if rc != 0:
            check(rc)
    finally:
        if switch:
            ctx.__exit__(None, None, None)
    return out


class _TemporalLossFn(torch.autograd.Function):
    """Gradients to ``prev`` and ``cur`` only (what the reference's trainers use: the flow and the mask come from the data
    set or from a frozen flow network under no_grad).  ``temporal_loss`` routes flows / masks that require grad through the
    differentiable ``warp`` instead (never a silently missing gradient); double backward is not defined (once_differentiable)."""

    @staticmethod
    def forward(ctx, prev, cur, flow, mask, loss, flags):
        ctx.save_for_backward(prev, cur, flow, mask)
        ctx.loss, ctx.flags = loss, flags
        return _loss_forward(prev, cur, flow, mask, loss, flags)

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, grad_out):
        prev, cur, flow, mask = ctx.saved_tensors
        if prev.dtype != torch.float32:
            return _loss_backward_bf16(ctx, grad_out, prev, cur, flow, mask)
        B, C, H, W = prev.shape
        need_prev, need_cur = ctx.needs_input_grad[0], ctx.needs_input_grad[1]
        gp = torch.empty_like(prev) if need_prev else None
        gc = torch.empty_like(cur) if need_cur else None
        # the upstream gradient as it is; the kernel multiplies it by 1/N (one rounded fp32 product, like `grad_out * (1.0 / N)`)
        scale = grad_out if (grad_out.dtype == torch.float32 and grad_out.is_cuda) else grad_out.to(device=prev.device, dtype=torch.float32)
        dev = prev.device
        switch = torch.cuda.current_device() != dev.index
        if switch:
            dctx = torch.cuda.device(dev)
            dctx.__enter__()
        try:
            plan = _loss_plan(dev, B, H, W)
            rc = plan.bwd(flow.data_ptr(), mask.data_ptr(), prev.data_ptr(), cur.data_ptr(), scale.data_ptr(), 1.0 / float(B * C * H * W),
                          gp.data_ptr() if gp is not None else None, gc.data_ptr() if gc is not None else None,
                          B, C, H, W, ctx.flags, ctx.loss, plan.stream)
            if rc != 0:
                check(rc)
        finally:
            if switch:
                dctx.__exit__(None, None, None)
        return gp, gc, None, None, None, None


def _loss_backward_bf16(ctx, grad_out, prev, cur, flow, mask):
    """``_TemporalLossFn.backward`` for bf16 frames (``tclb200_tcl_backward_dt``): the fp32 gradients of the upcast frames,
    each rounded once to bf16 -- what autograd gives the reference expression under ``torch.autocast(..., torch.bfloat16)``."""
    B, C, H, W = prev.shape
    dt = _frame_dtype(prev)
    need_prev, need_cur = ctx.needs_input_grad[0], ctx.needs_input_grad[1]
    gp = torch.empty_like(prev) if need_prev else None
    gc = torch.empty_like(cur) if need_cur else None
    scale = grad_out if (grad_out.dtype == torch.float32 and grad_out.is_cuda) else grad_out.to(device=prev.device, dtype=torch.float32)
    with torch.cuda.device(prev.device):
        ws, nbytes = _backward_workspace(B, C, H, W, dt, prev.device) if need_prev else (None, 0)
        check(_cabi.lib().tclb200_tcl_backward_dt(_ptr(flow), _ptr(mask), _ptr(prev), _ptr(cur), _ptr(scale), 1.0 / float(B * C * H * W),
                                                  _ptr(gp), _ptr(gc), B, C, H, W, dt, ctx.flags, ctx.loss, _ptr(ws), nbytes,
                                                  _stream_handle()))
    return gp, gc, None, None, None, None


def temporal_loss(mask, cur, prev, flow, loss="l2", validity=False):
    """Training temporal loss, differentiable w.r.t. ``cur`` and ``prev`` in one fused launch each way; a ``flow`` or ``mask``
    that requires grad gets its gradient too (composed from the differentiable ``warp``, like the reference expression).

    ``loss='l2'``: ((mask*(cur - warp(prev,flow)))**2).mean()      (solver.py:444, fs_ruder.py:97)
    ``loss='l1'``: (mask*abs(warp(prev,flow) - cur)).mean()         (MoGAN cycle_gan_model.py:280-281)
    ``validity`` selects fs_lib.warp for the learning-based trainers.

    bf16 frames: the loss is evaluated in fp32 on the upcast frames and returned as an fp32 scalar; the frames' gradients
    are the fp32 ones rounded to bf16 -- the reference expression under ``torch.autocast("cuda", torch.bfloat16)``, where
    ``grid_sampler`` runs in fp32 and ``mask*(cur - w)`` promotes to fp32.
    """
    if not (cur.is_cuda and prev.is_cuda and flow.is_cuda and (mask is None or mask.is_cuda)):
        _require_cuda(mask, cur, prev, flow)
    code = L2 if loss == "l2" else {"l1": L1}[loss]
    if flow.dim() != 4 or flow.shape[1] != 2:
        raise RuntimeError(f"tcl_b200: flow must be (B,2,H,W), got {tuple(flow.shape)}")
    B, _, H, W = flow.shape
    if flow.dtype != torch.float32 or not flow.is_contiguous():
        flow = flow.float().contiguous()
    if not prev.is_contiguous():
        prev = prev.contiguous()
    if not cur.is_contiguous():
        cur = cur.contiguous()
    if prev.dim() != 4 or prev.shape[0] != B or prev.shape[2] != H or prev.shape[3] != W or cur.shape != prev.shape or cur.dtype != prev.dtype:
        raise RuntimeError(f"tcl_b200: prev {tuple(prev.shape)} / cur {tuple(cur.shape)} must be (B,C,H,W) frames matching the flow {tuple(flow.shape)}")
    _frame_dtype(prev)
    if mask is None:
        mask = torch.ones((B, 1, H, W), dtype=torch.float32, device=flow.device)
    elif mask.dtype != torch.float32 or not mask.is_contiguous():
        mask = mask.float().contiguous()
    if mask.shape != (B, 1, H, W):
        raise RuntimeError(f"tcl_b200: mask must be (B,1,H,W), got {tuple(mask.shape)}")
    flags = VALIDITY if validity else 0
    if torch.is_grad_enabled():
        if flow.requires_grad or mask.requires_grad:
            # a learnable flow (MoGAN's motion network: warp(fake_B, netM_A(bf)), cycle_gan_model.py:177-178,280) or a soft mask that
            # is being trained: the fused backward has no gradient for them, so the loss is composed like the reference expression
            # from the differentiable warp (gradients to the frame and the flow, tclb200_warp_backward) and autograd's elementwise ops.
            # bf16 frames are upcast first, like autocast does for grid_sampler: the warp and the tail run in fp32 and the value is
            # an fp32 scalar as on the fused path; autograd rounds the frames' gradients back to bf16
            if prev.dtype != torch.float32:
                prev, cur = prev.float(), cur.float()
            w = _warp(prev, flow, flags)
            return ((mask * (cur - w)) ** 2).mean() if code == L2 else (mask * torch.abs(w - cur)).mean()
        if prev.requires_grad or cur.requires_grad:
            return _TemporalLossFn.apply(prev, cur, flow, mask, code, flags)
    return _loss_forward(prev, cur, flow, mask, code, flags)


def generateMask(simg, prev, flow):
    """ConGAN's scalar soft mask ``exp(-50 * |simg - warp(prev, flow)|.mean())`` (ConGAN/models/cycle_gan_model.py:136-137,
    where ``wimg`` is ``warp(...)`` of the previous frame): the warp and the mean absolute difference are one fused
    launch; differentiable like the reference expression.  ``loss_TCL_A`` (``:298``) is then
    ``generateMask(...) * temporal_loss(None, fuse_B, prev_B, flow, loss='l1') * lambda_TCL``."""
    return torch.exp(-50.0 * temporal_loss(None, simg, prev, flow, loss="l1"))
