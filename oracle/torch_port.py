"""TEST INFRASTRUCTURE ONLY -- ATen-op restatement of the reference's temporal-consistency path.

This module is part of the *oracle* (see oracle/README.md): only ``tests/``,
``__graft_entry__.smoke()`` and ``bench.py``'s cpu_baseline / ``--impl reference`` legs
may import it.  The product package never does.

It issues the SAME sequence of ATen ops as the reference functions it restates, so that

* on CPU it is bit-identical to the reference (checked in ``tests/test_oracle_pinning.py``
  against the reference's outputs stored in ``tests/golden/ref_cpu_*.npz``), and
* on a GPU it reproduces what the
  reference would compute on CUDA -- the arithmetic lives in ATen's ``grid_sampler_2d``,
  ``linalg_vector_norm``, ``constant_pad_nd`` and elementwise kernels, not in the
  reference's Python.

Reference lines followed (paths relative to the upstream repository root):

* ``central_diff``       -> ``utils/flowtools.py:12-16``  (``gradient``)
* ``backward_warp``      -> ``utils/flowtools.py:18-32``  (``warp``)
* ``fb_consistency``     -> ``utils/flowtools.py:34-58``  (``fbcCheckTorch``)
* ``fb_consistency_mob`` -> ``methods/optimization-based/flowtools.py:34-58`` (occlusion test disabled)
* ``validity_warp``      -> ``methods/learning-based/fs_lib.py:5-39`` (``warp`` x binarised ones-warp)
* ``tcl_rmse``           -> ``utils/sintel_eval.py:110``
* ``tcl_rmse_per_sample``-> ``utils/metrics/eval.py:138``
* ``tcl_l2``             -> ``methods/GAN-based/StarGANv2AdvCon/core/solver.py:444``
* ``tcl_l1``             -> ``methods/GAN-based/MoGAN/models/cycle_gan_model.py:280-281``
* ``blend``              -> ``methods/optimization-based/obst_eval.py:500``
* ``reconet_output_loss``-> ``methods/learning-based/fs_reconet.py:63-69``  (``o_temporal_loss`` / ``gamma_o``)
* ``ruder_input``        -> ``methods/learning-based/fs_ruder.py:47-50``    (``warp`` + ``torch.cat`` of one chain step)
"""
import torch
import torch.nn.functional as F


def _pixel_grid(B, H, W, device):
    # integer pixel coordinates as fp32, channel 0 = x, channel 1 = y
    xs = torch.arange(0, W).view(1, 1, 1, W).expand(B, 1, H, W)
    ys = torch.arange(0, H).view(1, 1, H, 1).expand(B, 1, H, W)
    return torch.cat((xs, ys), 1).float().to(device)


def _normalised_sampling_grid(f):
    """(B,2,H,W) pixel flow -> (B,H,W,2) grid in the reference's [-1,1] convention.

    The divisor is ``size-1`` (align_corners=True style) although sampling is later done
    with align_corners=False -- that quirk is the reference's (flowtools.py:28-32) and is kept.
    Op order: add, mul 2.0, div by python scalar, sub 1.0 (each a separate rounded ATen op).
    """
    B, _, H, W = f.shape
    v = _pixel_grid(B, H, W, f.device) + f
    gx = 2.0 * v[:, 0, :, :] / max(W - 1, 1) - 1.0
    gy = 2.0 * v[:, 1, :, :] / max(H - 1, 1) - 1.0
    return torch.stack((gx, gy), dim=3)


def central_diff(x):
    """Zero-padded central differences of a (B,H,W) plane stack -> (2,B,H,W) = [d/dx, d/dy]."""
    right = F.pad(x, (0, 1, 0, 0))[:, :, 1:]
    left = F.pad(x, (1, 0, 0, 0))[:, :, :-1]
    down = F.pad(x, (0, 0, 0, 1))[:, 1:, :]
    up = F.pad(x, (0, 0, 1, 0))[:, :-1, :]
    return torch.stack([(right - left) / 2, (down - up) / 2])


def backward_warp(x, f):
    """Bilinear, zero-padded backward warp of ``x`` (B,C,H,W) by pixel flow ``f`` (B,2,H,W)."""
    return F.grid_sample(x, _normalised_sampling_grid(f), mode="bilinear",
                         padding_mode="zeros", align_corners=False)


def _sqnorm(t, dim):
    # the reference squares a 2-norm (sqrt then square), it does not sum squares directly
    return torch.norm(t, dim=dim) ** 2


def fb_consistency(ff, bf, occlusion_test=True, return_margins=False):
    """Forward-backward consistency + motion-boundary mask, (B,1,H,W) fp32 in {0,1}.

    ``return_margins`` additionally returns (margin_occ, margin_mob): lhs - rhs of the two
    strict ``>`` tests in fp32, which define north_star's 1e-6 near-threshold exemption band.
    """
    B, _, H, W = bf.shape
    dev = bf.device
    keep = torch.ones((B, H, W), device=dev)
    zero = torch.zeros(1, device=dev)
    nb = _sqnorm(bf, 1)
    m_occ = None
    if occlusion_test:
        wf = backward_warp(ff, bf)
        nwb = _sqnorm(wf + bf, 1)
        nw = _sqnorm(wf, 1)
        thr = 0.01 * (nw + nb) + 0.5
        keep = torch.where(nwb > thr, zero, keep)
        m_occ = nwb - thr
    gu = central_diff(bf[:, 0, :, :])
    gv = central_diff(bf[:, 1, :, :])
    lhs = _sqnorm(gu, 0) + _sqnorm(gv, 0)
    rhs = 0.01 * nb + 0.002
    keep = torch.where(lhs > rhs, zero, keep)
    if return_margins:
        return keep.unsqueeze(1), m_occ, lhs - rhs
    return keep.unsqueeze(1)


def fb_consistency_mob(ff, bf):
    """Optimisation-based variant: motion-boundary test only (``ff`` unused)."""
    return fb_consistency(ff, bf, occlusion_test=False)


def validity_warp(x, flo):
    """fs_lib.warp: warp times the binarised warp of an all-ones image (>= 0.9999 -> 1)."""
    g = _normalised_sampling_grid(flo)
    out = F.grid_sample(x, g, mode="bilinear", padding_mode="zeros", align_corners=False)
    valid = F.grid_sample(torch.ones_like(x), g, mode="bilinear", padding_mode="zeros",
                          align_corners=False)
    valid = torch.where(valid < 0.9999, torch.zeros_like(valid), valid)
    valid = torch.where(valid > 0, torch.ones_like(valid), valid)
    return out * valid


def tcl_l2(mask, cur, warped):
    return ((mask * (cur - warped)) ** 2).mean()


def tcl_rmse(mask, cur, warped):
    return ((mask * (cur - warped)) ** 2).mean() ** 0.5


def tcl_rmse_per_sample(mask, cur, warped):
    return ((mask * (cur - warped)) ** 2).mean(dim=(1, 2, 3)) ** 0.5


def tcl_l1(mask, cur, warped):
    return (mask * torch.abs(warped - cur)).mean()


def blend(mask, warped, img):
    return mask * warped + (1 - mask) * img


def reconet_output_loss(mask, styled2, styled1, img2, img1, flow):
    """ReCoNet's output-level temporal loss without its weight (fs_reconet.py:63-69); ``warp`` there is fs_lib.warp."""
    output_term = styled2 - validity_warp(styled1, flow)
    input_term = img2 - validity_warp(img1, flow)
    input_term = (0.2126 * input_term[:, 0, :, :] + 0.7152 * input_term[:, 1, :, :] + 0.0722 * input_term[:, 2, :, :]).unsqueeze(1)
    return ((mask * (output_term - input_term)) ** 2).mean()


def ruder_input(img, mask, styled_prev, flow):
    """One step of Ruder's chain (fs_ruder.py:47-50): the network input and the warped frame."""
    warped = validity_warp(styled_prev, flow)
    return torch.cat((img, mask, warped), 1), warped


def long_term_step(mask_last, ff_last, bf_last, styled_past, pre):
    """One step of the cumulative long-term initialisation (obst_eval.py:515-516, disabled upstream)."""
    mask_last = torch.clamp(mask_last - fb_consistency(ff_last, bf_last), 0.0, 1.0)
    return mask_last, mask_last * backward_warp(styled_past, bf_last) + (1 - mask_last) * pre


def temporal_error(ff, bf, prev, cur):
    """computeTCL minus RAFT and the generator (utils/sintel_eval.py:104-110)."""
    m = fb_consistency(ff, bf)
    return tcl_rmse(m, cur, backward_warp(prev, bf))


def upsample_flow(flow, mask):
    """Convex 8x upsampling of a coarse flow as RAFT defines it (utils/raft/raft/raft.py:72-83): per fine pixel a
    softmax over 9 logits weights the zero-padded 3x3 coarse neighbourhood of 8*flow.  Written with explicit
    neighbour shifts instead of unfold; same arithmetic up to summation order."""
    n, _, hc, wc = flow.shape
    weights = torch.softmax(mask.reshape(n, 9, 64, hc, wc), dim=1)          # (n, neighbour, 8*8 sub-pixel, h, w)
    padded = F.pad(8.0 * flow, (1, 1, 1, 1))                                # zero border, like unfold(padding=1)
    fine = torch.zeros(n, 2, 64, hc, wc, dtype=flow.dtype, device=flow.device)
    for k in range(9):
        dy, dx = divmod(k, 3)
        neighbour = padded[:, :, dy:dy + hc, dx:dx + wc]                     # coarse flow at (h + dy - 1, w + dx - 1)
        fine = fine + weights[:, k].unsqueeze(1) * neighbour.unsqueeze(2)
    fine = fine.reshape(n, 2, 8, 8, hc, wc).permute(0, 1, 4, 2, 5, 3)       # (n, 2, h, i, w, j)
    return fine.reshape(n, 2, 8 * hc, 8 * wc)
