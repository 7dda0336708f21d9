"""The path's entries as ``torch.library`` custom operators (namespace ``tcl_b200``), so that TorchDynamo, FakeTensor / export
tracing and CUDA-graph capture under ``torch.compile`` see them as single operators instead of opaque ctypes calls.

One operator per family of C entries; flags are integer arguments.  Each CUDA implementation calls the internal function
the eager route calls (``ops._warp_forward``, ``ops._loss_forward``, ``ops.fused_forward``, ...), so the argument
marshalling of every C entry exists once.  The fake implementations derive outputs from input shapes alone (no CUDA
runtime, no ctypes, no ``data_ptr()``), symbolic sizes included.  Every output is a fresh tensor: where a gradient is not
asked for, a backward operator returns an empty placeholder in its place.

The public functions validate their arguments and then call these operators when the call is being traced
(``ops._traced``); eager calls keep the direct route.  Validation is not repeated here: call the public functions, or
pass these operators what the public functions would.
"""
from typing import List, Optional, Tuple

import torch
from torch import Tensor

from . import chains, ops
from ._cabi import VALIDITY


def _op(name):
    return torch.library.custom_op(f"tcl_b200::{name}", mutates_args=(), device_types="cuda")


def _or_empty(grad, like):
    return grad if grad is not None else like.new_empty(0)


def _new(t, shape, dtype=torch.float32):
    return t.new_empty(shape, dtype=dtype)


# ------------------------------------------------------------------------------------------------
# gradient (tclb200_gradient_strided), no autograd
# ------------------------------------------------------------------------------------------------
@_op("gradient")
def gradient(x: Tensor) -> Tensor:
    return ops._gradient_launch(x)


@gradient.register_fake
def _(x):
    return _new(x, (2,) + tuple(x.shape))


# ------------------------------------------------------------------------------------------------
# warp / fs_lib.warp (tclb200_warp, the struct entry for strided flows; tclb200_warp_backward[_dt])
# ------------------------------------------------------------------------------------------------
@_op("warp")
def warp(x: Tensor, f: Tensor, flags: int) -> Tensor:
    f, f_plane, f_batch = ops._flow_view(f, "f")
    return ops._warp_forward(x.contiguous(), f, flags, f_plane, f_batch)


@warp.register_fake
def _(x, f, flags):
    return _new(x, x.shape, x.dtype)


@_op("warp_backward")
def warp_backward(grad_out: Tensor, x: Tensor, f: Tensor, flags: int, need_x: bool, need_f: bool) -> Tuple[Tensor, Tensor]:
    gx, gf = ops._warp_backward_raw(grad_out, x.contiguous(), ops._flow(f, "f"), flags, need_x, need_f)
    return _or_empty(gx, x), _or_empty(gf, f)


@warp_backward.register_fake
def _(grad_out, x, f, flags, need_x, need_f):
    return _new(x, x.shape if need_x else (0,), x.dtype), _new(f, f.shape if need_f else (0,), f.dtype)


def _warp_setup(ctx, inputs, output):
    x, f, ctx.flags = inputs
    ctx.save_for_backward(x, f)


def _warp_grad(ctx, grad):
    x, f = ctx.saved_tensors
    need_x, need_f = ctx.needs_input_grad[0], ctx.needs_input_grad[1]
    gx, gf = warp_backward(grad, x, f, ctx.flags, need_x, need_f)
    return (gx if need_x else None), (gf if need_f else None), None


warp.register_autograd(_warp_grad, setup_context=_warp_setup)


# ------------------------------------------------------------------------------------------------
# fbcCheckTorch and its variants (tclb200_fbcheck, the struct entry for strided flows), no autograd
# ------------------------------------------------------------------------------------------------
@_op("fbcheck")
def fbcheck(ff: Optional[Tensor], bf: Tensor, flags: int, want_near: bool) -> List[Tensor]:
    """-> [mask] or, with ``want_near``, [mask, near-threshold count]."""
    bf, bf_plane, bf_batch = ops._flow_view(bf, "bf")
    ff, ff_plane, ff_batch = ops._flow_view(ff, "ff") if ff is not None else (None, 0, 0)
    mask, near = ops._fbcheck_launch(ff, bf, flags, want_near, ff_plane, ff_batch, bf_plane, bf_batch)
    return [mask, near] if want_near else [mask]


@fbcheck.register_fake
def _(ff, bf, flags, want_near):
    B, _, H, W = bf.shape
    mask = _new(bf, (B, 1, H, W))
    return [mask, _new(bf, (1,), torch.int64)] if want_near else [mask]


# ------------------------------------------------------------------------------------------------
# RAFT's convex upsampling (tclb200_upsample_flow), no autograd
# ------------------------------------------------------------------------------------------------
@_op("upsample_flow")
def upsample_flow(flow: Tensor, mask: Tensor) -> Tensor:
    return ops._upsample_flow_launch(flow, mask)


@upsample_flow.register_fake
def _(flow, mask):
    N, _, H, W = flow.shape
    return _new(flow, (N, 2, 8 * H, 8 * W))


# ------------------------------------------------------------------------------------------------
# training loss (tclb200_tcl_forward through the loss plan; tclb200_tcl_backward_scaled / _dt)
# ------------------------------------------------------------------------------------------------
@_op("temporal_loss")
def temporal_loss(prev: Tensor, cur: Tensor, flow: Tensor, mask: Tensor, loss: int, flags: int) -> Tensor:
    """The 0-dim fp32 mean of ``ops.temporal_loss``; ``mask`` (B,1,H,W) fp32 is required (all ones for none)."""
    return ops._loss_forward(prev.contiguous(), cur.contiguous(), flow.contiguous(), mask.contiguous(), loss, flags)


@temporal_loss.register_fake
def _(prev, cur, flow, mask, loss, flags):
    return _new(prev, ())


@_op("temporal_loss_backward")
def temporal_loss_backward(grad_out: Tensor, prev: Tensor, cur: Tensor, flow: Tensor, mask: Tensor, loss: int, flags: int,
                           need_prev: bool, need_cur: bool) -> Tuple[Tensor, Tensor]:
    prev, cur = prev.contiguous(), cur.contiguous()
    gp, gc = ops._loss_backward(grad_out, prev, cur, flow.contiguous(), mask.contiguous(), loss, flags, need_prev, need_cur)
    return _or_empty(gp, prev), _or_empty(gc, cur)


@temporal_loss_backward.register_fake
def _(grad_out, prev, cur, flow, mask, loss, flags, need_prev, need_cur):
    return _new(prev, prev.shape if need_prev else (0,), prev.dtype), _new(cur, cur.shape if need_cur else (0,), cur.dtype)


def _loss_setup(ctx, inputs, output):
    prev, cur, flow, mask, ctx.loss, ctx.flags = inputs
    ctx.save_for_backward(prev, cur, flow, mask)


def _loss_grad(ctx, grad):
    prev, cur, flow, mask = ctx.saved_tensors
    need_prev, need_cur = ctx.needs_input_grad[0], ctx.needs_input_grad[1]
    gp, gc = temporal_loss_backward(grad, prev, cur, flow, mask, ctx.loss, ctx.flags, need_prev, need_cur)
    return (gp if need_prev else None), (gc if need_cur else None), None, None, None, None


temporal_loss.register_autograd(_loss_grad, setup_context=_loss_setup)


# ------------------------------------------------------------------------------------------------
# evaluation helpers (tclb200_tcl_forward without index arrays or bands), no autograd
# ------------------------------------------------------------------------------------------------
@_op("fused_eval")
def fused_eval(bf: Tensor, prev: Tensor, cur: Tensor, ff: Optional[Tensor], mask: Optional[Tensor], loss: int, finalize: int,
               what: int, u8_scale: Optional[List[float]], u8_offset: Optional[List[float]]) -> List[Tensor]:
    """One fused evaluation launch -> the outputs ``what`` selects (``ops.EVAL_TOTAL`` / ``EVAL_PAIRS`` / ``EVAL_KEPT`` /
    ``EVAL_BLEND``, see ``ops._evaluate``)."""
    return ops._evaluate_launch(what, bf, prev, cur, ff, mask, loss, finalize, u8_scale, u8_offset)


@fused_eval.register_fake
def _(bf, prev, cur, ff, mask, loss, finalize, what, u8_scale, u8_offset):
    # the same views of one result buffer per dtype that fused_forward allocates
    B = bf.shape[0]
    if what == ops.EVAL_TOTAL:
        return [_new(bf, (B + 1,))[B]]
    if what == ops.EVAL_PAIRS:
        return [_new(bf, (B + 1,))[:B]]
    if what == ops.EVAL_KEPT:
        return [_new(bf, (B + 2,), torch.float64)[:B], _new(bf, (B + 1,), torch.float64)[:B]]
    return [_new(prev, prev.shape, prev.dtype)]


# ------------------------------------------------------------------------------------------------
# chains (tclb200_reconet_loss + tclb200_tcl_backward; tclb200_ruder_input + the warp backward)
# ------------------------------------------------------------------------------------------------
@_op("reconet_loss")
def reconet_loss(styled2: Tensor, styled1: Tensor, img2: Tensor, img1: Tensor, flow: Tensor,
                 mask: Optional[Tensor]) -> Tuple[Tensor, Tensor]:
    """-> (the 0-dim loss, the luminance term its backward reads)."""
    c = lambda t: t.contiguous() if t is not None else None
    return chains._reconet_forward(c(styled2), c(styled1), c(img2), c(img1), c(flow), c(mask))


@reconet_loss.register_fake
def _(styled2, styled1, img2, img1, flow, mask):
    B, _, H, W = flow.shape
    return _new(flow, ()), _new(flow, (B, 1, H, W))


@_op("reconet_loss_backward")
def reconet_loss_backward(grad_out: Tensor, styled1: Tensor, styled2: Tensor, flow: Tensor, mask: Optional[Tensor], lum: Tensor,
                          need2: bool, need1: bool) -> Tuple[Tensor, Tensor]:
    styled1, styled2 = styled1.contiguous(), styled2.contiguous()
    g2, g1 = chains._reconet_backward(grad_out, styled1, styled2, flow.contiguous(), mask.contiguous() if mask is not None else None,
                                      lum.contiguous(), need2, need1)
    return _or_empty(g2, styled2), _or_empty(g1, styled1)


@reconet_loss_backward.register_fake
def _(grad_out, styled1, styled2, flow, mask, lum, need2, need1):
    return _new(styled2, styled2.shape if need2 else (0,)), _new(styled1, styled1.shape if need1 else (0,))


def _reconet_setup(ctx, inputs, output):
    styled2, styled1, _, _, flow, mask = inputs
    ctx.save_for_backward(styled1, styled2, flow, mask, output[1])


def _reconet_grad(ctx, grad_loss, grad_lum):
    styled1, styled2, flow, mask, lum = ctx.saved_tensors
    need2, need1 = ctx.needs_input_grad[0], ctx.needs_input_grad[1]
    g2, g1 = reconet_loss_backward(grad_loss, styled1, styled2, flow, mask, lum, need2, need1)
    return (g2 if need2 else None), (g1 if need1 else None), None, None, None, None


reconet_loss.register_autograd(_reconet_grad, setup_context=_reconet_setup)


@_op("ruder_input")
def ruder_input(styled_prev: Tensor, img: Tensor, mask: Optional[Tensor], flow: Tensor) -> Tuple[Tensor, Tensor]:
    """-> (the 7-channel network input, the warped frame)."""
    return chains._ruder_forward(styled_prev.contiguous(), img.contiguous(), mask.contiguous() if mask is not None else None,
                                 flow.contiguous())


@ruder_input.register_fake
def _(styled_prev, img, mask, flow):
    B, _, H, W = flow.shape
    return _new(flow, (B, 7, H, W)), _new(flow, (B, 3, H, W))


def _ruder_setup(ctx, inputs, output):
    styled_prev, _, _, flow = inputs
    ctx.save_for_backward(styled_prev, flow)


def _ruder_grad(ctx, g_cat, g_warped):
    styled_prev, flow = ctx.saved_tensors
    if not ctx.needs_input_grad[0]:
        return None, None, None, None
    # the warped frame reaches the outputs twice: channels 4..6 of the network input and `warped` itself
    g = g_cat[:, 4:7]
    g = (g + g_warped) if g_warped is not None else g
    gx, _ = warp_backward(g.contiguous(), styled_prev, flow, VALIDITY, True, False)
    return gx, None, None, None


ruder_input.register_autograd(_ruder_grad, setup_context=_ruder_setup)
