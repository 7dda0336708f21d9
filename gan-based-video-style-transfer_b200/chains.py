"""Warp chains of the learning-based trainers (SURVEY.md section 8f, rank 2) as fused helpers.

* ``reconet_output_temporal_loss`` -- ReCoNet's output-level temporal loss, methods/learning-based/fs_reconet.py:63-69
  (``o_temporal_loss`` without its ``gamma_o`` weight)
* ``ruder_network_input``          -- one step of Ruder's recurrent chain, methods/learning-based/fs_ruder.py:50-75:
  ``torch.cat((img, mask, warp(styled_prev, flow)), 1)`` plus the warped frame for the loss of ``:97``
* ``long_term_blend_step``         -- one step of the optimisation-based method's cumulative long-term initialisation,
  methods/optimization-based/obst_eval.py:512-518 (disabled upstream: the lines sit inside a string literal)

Both use ``fs_lib.warp`` (methods/learning-based/fs_lib.py:5-39: bilinear taps times the binarised warp of an all-ones
image) as the reference trainers do (``from fs_lib import warp``).  CUDA fp32 tensors only; no CPU implementation.
"""
import ctypes

import torch

from . import _cabi
from ._cabi import check
from .ops import L2, VALIDITY, _cache_pool, _flow, _ptr, _require_cuda, _stream_handle, _traced, _warp_backward_raw

_scratch = {}


def _frames3(t, name):
    if t.dim() != 4 or t.shape[1] != 3:
        raise RuntimeError(f"tcl_b200: {name} must be (B,3,H,W), got {tuple(t.shape)}")
    return t.float().contiguous()


def _mask1(mask, B, H, W):
    if mask is None:
        return None
    if tuple(mask.shape) != (B, 1, H, W):
        raise RuntimeError(f"tcl_b200: mask must be (B,1,H,W) = {(B, 1, H, W)}, got {tuple(mask.shape)}")
    return mask.float().contiguous()


class _ReconetLossFn(torch.autograd.Function):
    """Gradients to the two stylised frames (the images, the flow and the mask are data in fs_reconet.py)."""

    @staticmethod
    def forward(ctx, styled2, styled1, img2, img1, flow, mask):
        loss, lum = _reconet_forward(styled2, styled1, img2, img1, flow, mask)
        ctx.save_for_backward(styled1, styled2, flow, mask, lum)
        return loss

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, grad_out):
        styled1, styled2, flow, mask, lum = ctx.saved_tensors
        g2, g1 = _reconet_backward(grad_out, styled1, styled2, flow, mask, lum, ctx.needs_input_grad[0], ctx.needs_input_grad[1])
        return g2, g1, None, None, None, None


def _reconet_forward(styled2, styled1, img2, img1, flow, mask):
    """-> (loss, lum): the 0-dim loss and the luminance term its backward reads."""
    B, _, H, W = flow.shape
    lib = _cabi.lib()
    need = lib.tclb200_reconet_scratch_bytes(B, H, W)
    key = (flow.device.index, torch.cuda.current_stream().cuda_stream)
    buf = _scratch.get(key)
    if buf is None or buf.numel() < need:
        with _cache_pool(flow.device):
            buf = torch.empty(need, dtype=torch.uint8, device=flow.device)
        _scratch[key] = buf
    lum = torch.empty((B, 1, H, W), dtype=torch.float32, device=flow.device)
    loss = torch.empty((), dtype=torch.float32, device=flow.device)
    with torch.cuda.device(flow.device):
        check(lib.tclb200_reconet_loss(_ptr(flow), _ptr(mask), _ptr(styled1), _ptr(styled2), _ptr(img1), _ptr(img2), _ptr(lum), _ptr(loss),
                                       None, _ptr(buf), buf.numel(), B, H, W, _stream_handle()))
    return loss, lum


def _reconet_backward(grad_out, styled1, styled2, flow, mask, lum, need2, need1):
    """(grad_styled2, grad_styled1), None where not needed."""
    B, C, H, W = styled1.shape
    g2 = torch.empty_like(styled2) if need2 else None
    g1 = torch.empty_like(styled1) if need1 else None
    # d loss / d (styled2 - warp(styled1)) = 2/N * mask^2 * ((styled2 - lum) - warp(styled1)): the fused training-loss
    # backward with `cur` = styled2 - lum (the luminance term carries no gradient: the images are data)
    cur = styled2 - lum
    scale = (grad_out.float() / float(B * C * H * W)).reshape(1).contiguous()
    with torch.cuda.device(styled1.device):
        check(_cabi.lib().tclb200_tcl_backward(_ptr(flow), _ptr(mask), _ptr(styled1), _ptr(cur), _ptr(scale), _ptr(g1), _ptr(g2),
                                               B, C, H, W, VALIDITY, L2, _stream_handle()))
    return g2, g1


def reconet_output_temporal_loss(mask, styled2, styled1, img2, img1, flow):
    """``((mask * ((styled2 - warp(styled1, flow)) - lum(img2 - warp(img1, flow))))**2).mean()`` in one fused pass
    (fs_reconet.py:63-69; ``lum = 0.2126 r + 0.7152 g + 0.0722 b``); differentiable w.r.t. ``styled2`` and ``styled1``."""
    _require_cuda(mask, styled2, styled1, img2, img1, flow)
    flow = _flow(flow)
    B, _, H, W = flow.shape
    s2, s1, i2, i1 = (_frames3(t, n) for t, n in ((styled2, "styled2"), (styled1, "styled1"), (img2, "img2"), (img1, "img1")))
    for t in (s2, s1, i2, i1):
        if tuple(t.shape) != (B, 3, H, W):
            raise RuntimeError(f"tcl_b200: frames must be {(B, 3, H, W)} like the flow, got {tuple(t.shape)}")
    m = _mask1(mask, B, H, W)
    if torch.is_grad_enabled() and (flow.requires_grad or (m is not None and m.requires_grad) or i1.requires_grad or i2.requires_grad):
        raise RuntimeError("tcl_b200: reconet_output_temporal_loss differentiates w.r.t. the stylised frames only")
    if _traced(s2, s1, i2, i1, flow, m):
        return torch.ops.tcl_b200.reconet_loss(s2, s1, i2, i1, flow, m)[0]
    return _ReconetLossFn.apply(s2, s1, i2, i1, flow, m)


class _RuderInputFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, styled_prev, img, mask, flow):
        cat, warped = _ruder_forward(styled_prev, img, mask, flow)
        ctx.save_for_backward(styled_prev, flow)
        ctx.mark_non_differentiable()
        return cat, warped

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, g_cat, g_warped):
        styled_prev, flow = ctx.saved_tensors
        if not ctx.needs_input_grad[0]:
            return None, None, None, None
        # the warped frame reaches the outputs twice: channels 4..6 of the network input and `warped` itself
        g = g_cat[:, 4:7]
        g = (g + g_warped) if g_warped is not None else g
        gx, _ = _warp_backward_raw(g.contiguous(), styled_prev, flow, VALIDITY, need_x=True, need_f=False)
        return gx, None, None, None


def _ruder_forward(styled_prev, img, mask, flow):
    B, _, H, W = flow.shape
    cat = torch.empty((B, 7, H, W), dtype=torch.float32, device=flow.device)
    warped = torch.empty((B, 3, H, W), dtype=torch.float32, device=flow.device)
    with torch.cuda.device(flow.device):
        check(_cabi.lib().tclb200_ruder_input(_ptr(img), _ptr(mask), _ptr(styled_prev), _ptr(flow), _ptr(cat), _ptr(warped), B, H, W,
                                              _stream_handle()))
    return cat, warped


def ruder_network_input(img, mask, styled_prev, flow):
    """One step of Ruder's chain (fs_ruder.py:50-75): returns ``(torch.cat((img, mask, warped), 1), warped)`` with
    ``warped = warp(styled_prev, flow)`` (fs_lib.warp), written in one pass.  ``warped`` is the ``loss_warped`` of the
    temporal term (``:97``).  Differentiable w.r.t. ``styled_prev`` (the chain back-propagates through the earlier steps)."""
    _require_cuda(img, mask, styled_prev, flow)
    flow = _flow(flow)
    B, _, H, W = flow.shape
    img, sp = _frames3(img, "img"), _frames3(styled_prev, "styled_prev")
    if tuple(img.shape) != (B, 3, H, W) or tuple(sp.shape) != (B, 3, H, W):
        raise RuntimeError(f"tcl_b200: img / styled_prev must be {(B, 3, H, W)} like the flow")
    m = _mask1(mask, B, H, W)
    if torch.is_grad_enabled() and (flow.requires_grad or img.requires_grad or (m is not None and m.requires_grad)):
        raise RuntimeError("tcl_b200: ruder_network_input differentiates w.r.t. styled_prev only (images, masks and flows are data)")
    if _traced(img, sp, m, flow):
        return tuple(torch.ops.tcl_b200.ruder_input(sp, img, m, flow))
    return _RuderInputFn.apply(sp, img, m, flow)


def long_term_blend_step(mask_last, ff_last, bf_last, styled_past, pre):
    """One step of the cumulative long-term initialisation of methods/optimization-based/obst_eval.py:515-516 (the block is
    disabled upstream -- it sits inside a string literal -- and kept here for whoever switches it back on):

        mask_last = torch.clamp(mask_last - fbcCheckTorch(ff_last, bf_last), 0.0, 1.0)
        pre       = mask_last * warp(styled_past, bf_last) + (1 - mask_last) * pre

    Two launches of the library (the consistency mask; warp + blend in one pass, ``obst_eval.py:500``'s form) around the one
    elementwise clamp; no gradients, like the reference's initialisation.  Returns ``(mask_last, pre)``.  ``fbcCheckTorch`` is the
    two-test mask of utils/flowtools.py:34-58 as imported by the evaluation scripts; pass ``ops.fbcCheckTorch_mob`` results through
    ``mask_last`` yourself for the motion-boundary-only copy."""
    from .ops import fbcCheckTorch, warp_blend
    _require_cuda(mask_last, ff_last, bf_last, styled_past, pre)
    B, _, H, W = bf_last.shape
    mask_last = _mask1(mask_last, B, H, W)
    with torch.no_grad():
        mask_last = torch.clamp(mask_last - fbcCheckTorch(ff_last, bf_last), 0.0, 1.0)
        return mask_last, warp_blend(mask_last, styled_past, bf_last, pre)
