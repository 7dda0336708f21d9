"""CPU suite: pin the oracle (oracle/tcl_oracle.c + oracle/torch_port.py) to the reference.

Chain of evidence:
  1. torch_port == the reference functions' outputs stored in ref_cpu_*.npz, bit for bit, on CPU  (same ATen ops)
  2. C oracle (ATEN_CPU flavour) == golden vectors produced by the imported reference, bit for bit
  3. C oracle (ATEN_CUDA flavour) == vectors produced on a B200 by torch_port (ref_cuda_*.npz), bit for bit
The GPU suite then compares the CUDA kernels with the ATEN_CUDA flavour and with torch_port live.
"""
import warnings

import numpy as np
import pytest
import torch

from conftest import golden_files, load_npz
from oracle import torch_port as tp

warnings.filterwarnings("ignore", message="Default grid_sample")


def _synth_case(tcl, B=2, H=37, W=53, seed=5, kind="white", **kw):
    ff, bf = tcl.synth.make_flows(B, H, W, seed=seed, **kw)
    prev, cur = tcl.synth.make_frames(B, 3, H, W, seed=seed, kind=kind)
    return ff, bf, prev, cur


# ---------------------------------------------------------------- known-answer facts (SURVEY.md 8c)
def test_gradient_known_answer(oracle_mod):
    x = np.arange(12, dtype=np.float32).reshape(1, 3, 4)
    g = oracle_mod.central_diff(x)
    assert g[0, 0, 0].tolist() == [0.5, 1.0, 1.0, -1.0]
    assert g[1, 0, :, 0].tolist() == [2.0, 4.0, -2.0]
    assert np.array_equal(g, tp.central_diff(torch.from_numpy(x)).numpy())


def test_zero_flow_is_not_identity(oracle_mod):
    rng = np.random.default_rng(0)
    x = rng.standard_normal((1, 3, 16, 20)).astype(np.float32)
    f = np.zeros((1, 2, 16, 20), np.float32)
    for variant in (oracle_mod.ATEN_CPU, oracle_mod.ATEN_CUDA):
        assert np.abs(oracle_mod.warp(x, f, variant) - x).max() > 0.1  # the size-1 / align_corners quirk is kept


def test_white_noise_flow_masks_everything(oracle_mod):
    rng = np.random.default_rng(1)
    ff = rng.standard_normal((1, 2, 24, 24)).astype(np.float32) * 5
    bf = rng.standard_normal((1, 2, 24, 24)).astype(np.float32) * 5
    assert oracle_mod.fbcheck(ff, bf).sum() == 0


def test_border_is_masked_for_nonzero_flow(oracle_mod):
    yy, xx = np.meshgrid(np.arange(40, dtype=np.float32), np.arange(48, dtype=np.float32), indexing="ij")
    bf = np.stack([2.0 + 0.5 * np.sin(xx / 9), 1.5 + 0.5 * np.cos(yy / 7)])[None].astype(np.float32)
    m = oracle_mod.fbcheck(-bf, bf)[0, 0]
    assert m[0].sum() == 0 and m[-1].sum() == 0 and m[:, 0].sum() == 0 and m[:, -1].sum() == 0
    assert m[2:-2, 2:-2].mean() > 0.5
    assert set(np.unique(m)) <= {0.0, 1.0}


# ---------------------------------------------------------------- 1. torch_port == reference (CPU)
def _golden_tensors(path):
    return {k: torch.from_numpy(v) for k, v in load_npz(path).items() if v.dtype.kind == "f"}


@pytest.mark.parametrize("path", golden_files("ref_cpu_"))
def test_torch_port_bit_identical_to_reference(path):
    """ref_cpu_*.npz hold what the reference's own flowtools / fs_lib functions returned on CPU (tests/golden/make_golden.py)."""
    g = _golden_tensors(path)
    ff, bf, prev, cur = g["ff"], g["bf"], g["prev"], g["cur"]
    assert torch.equal(g["warp"], tp.backward_warp(prev, bf))
    assert torch.equal(g["mask"], tp.fb_consistency(ff, bf))
    assert torch.equal(g["grad_u"], tp.central_diff(bf[:, 0]))
    assert torch.equal(g["fs_warp"], tp.validity_warp(prev, bf))
    assert torch.equal(g["rmse"], tp.temporal_error(ff, bf, prev, cur))
    w = tp.backward_warp(prev, bf)
    assert torch.equal(g["rmse_per_sample"], tp.tcl_rmse_per_sample(g["mask"], cur, w))
    assert torch.equal(g["l2"], tp.tcl_l2(g["mask"], cur, w)) and torch.equal(g["l1"], tp.tcl_l1(g["mask"], cur, w))


def test_long_term_step_is_the_upstream_lines():
    """obst_eval.py:515-516 (inside a string literal upstream), composed from the reference's fbcCheckTorch and warp outputs."""
    g = _golden_tensors(golden_files("ref_cpu_smooth")[0])
    ff, bf, styled, pre = g["ff"], g["bf"], g["prev"], g["cur"]
    mask_last = (torch.rand(g["mask"].shape, generator=torch.Generator().manual_seed(1)) > 0.3).float()
    m = torch.clamp(mask_last - g["mask"], 0.0, 1.0)
    want = m * g["warp"] + (1 - m) * pre
    got_m, got = tp.long_term_step(mask_last, ff, bf, styled, pre)
    assert torch.equal(got_m, m) and torch.equal(got, want) and 0 < float(m.mean()) < 1


def test_reference_autograd_matches_port():
    """Gradients of the masked L2 loss through the reference's warp (stored by make_golden.py) == through torch_port."""
    paths = golden_files("ref_cpu_")
    assert paths
    for path in paths:
        g = _golden_tensors(path)
        p, f, c = (g[k].clone().requires_grad_(True) for k in ("prev", "bf", "cur"))
        ((g["mask"] * (c - tp.backward_warp(p, f))) ** 2).mean().backward()
        assert torch.equal(p.grad, g["grad_prev"]) and torch.equal(f.grad, g["grad_flow"]) and torch.equal(c.grad, g["grad_cur"])


# ---------------------------------------------------------------- 2. C oracle == golden (reference on CPU)
@pytest.mark.parametrize("path", golden_files("ref_cpu_"))
def test_c_oracle_matches_reference_golden_bitwise(oracle_mod, path):
    g = load_npz(path)
    v = oracle_mod.ATEN_CPU
    assert np.array_equal(oracle_mod.warp(g["prev"], g["bf"], v), g["warp"])
    assert np.array_equal(oracle_mod.fbcheck(g["ff"], g["bf"], variant=v), g["mask"])
    assert np.array_equal(oracle_mod.central_diff(g["bf"][:, 0]), g["grad_u"])
    assert np.array_equal(oracle_mod.validity_warp(g["prev"], g["bf"], v), g["fs_warp"])
    B, C, H, W = g["prev"].shape
    s2 = oracle_mod.masked_sums(g["mask"], g["cur"], g["warp"], 0)
    s1 = oracle_mod.masked_sums(g["mask"], g["cur"], g["warp"], 1)
    n = C * H * W
    assert np.allclose(np.sqrt(s2 / n), g["rmse_per_sample"], rtol=1e-5, atol=0)
    assert np.isclose(np.sqrt(s2.sum() / (B * n)), g["rmse"], rtol=1e-5, atol=0)
    assert np.isclose(s2.sum() / (B * n), g["l2"], rtol=1e-5, atol=0)
    assert np.isclose(s1.sum() / (B * n), g["l1"], rtol=1e-5, atol=0)
    fused = oracle_mod.temporal_error_sums(g["ff"], g["bf"], g["prev"], g["cur"], variant=v)
    assert np.allclose(fused, s2, rtol=1e-12)


@pytest.mark.parametrize("path", golden_files("ref_cpu_"))
def test_c_oracle_backward_matches_reference_autograd(oracle_mod, path):
    g = load_npz(path)
    B, C, H, W = g["prev"].shape
    n = B * C * H * W
    warped = oracle_mod.warp(g["prev"], g["bf"], oracle_mod.ATEN_CPU)
    m = g["mask"]
    grad_cur = 2.0 * m * m * (g["cur"] - warped) / n
    assert np.allclose(grad_cur, g["grad_cur"], rtol=1e-5, atol=1e-9)
    gx, gf = oracle_mod.warp_bwd(-grad_cur, g["prev"], g["bf"], oracle_mod.ATEN_CPU)
    assert np.allclose(gx, g["grad_prev"], rtol=1e-4, atol=1e-8)
    assert np.allclose(gf, g["grad_flow"], rtol=1e-3, atol=1e-7)


@pytest.mark.parametrize("shape,shift", [((2, 37, 53), 8.0), ((1, 96, 160), 20.0)])
def test_c_oracle_matches_port_bitwise(oracle_mod, tcl, shape, shift):
    """Shapes and displacements beyond the golden cases, against torch_port (bit-identical to the reference's outputs, 1. above)."""
    B, H, W = shape
    ff, bf, prev, cur = _synth_case(tcl, B, H, W, seed=21, max_shift=shift)
    v = oracle_mod.ATEN_CPU
    assert np.array_equal(oracle_mod.warp(prev.numpy(), bf.numpy(), v), tp.backward_warp(prev, bf).numpy())
    ref_mask, pmo, pmm = tp.fb_consistency(ff, bf, return_margins=True)
    mask, mo, mm = oracle_mod.fbcheck(ff.numpy(), bf.numpy(), variant=v, margins=True)
    assert np.array_equal(mask, ref_mask.numpy())
    # margins (the quantities the 1e-6 exemption band is defined on) are bit-identical too
    assert np.array_equal(mo, pmo.numpy()) and np.array_equal(mm, pmm.numpy())
    assert 0.2 < float(ref_mask.mean()) < 0.98
    assert np.array_equal(oracle_mod.validity_warp(prev.numpy(), bf.numpy(), v), tp.validity_warp(prev, bf).numpy())


def test_mob_only_variant(oracle_mod, tcl):
    ff, bf, _, _ = _synth_case(tcl, 1, 40, 56, seed=2, max_shift=5.0)
    m = oracle_mod.fbcheck(ff.numpy(), bf.numpy(), flags=oracle_mod.FLAG_MOB, variant=oracle_mod.ATEN_CPU)
    assert np.array_equal(m, tp.fb_consistency_mob(ff, bf).numpy())
    full = oracle_mod.fbcheck(ff.numpy(), bf.numpy(), variant=oracle_mod.ATEN_CPU)
    assert (m >= full).all() and m.sum() > full.sum()


# ---------------------------------------------------------------- 3. C oracle (CUDA flavour) == B200 torch vectors
@pytest.mark.parametrize("path", golden_files("ref_cuda_"))
def test_c_oracle_cuda_flavour_matches_b200_vectors(oracle_mod, path):
    g = load_npz(path)
    v = oracle_mod.ATEN_CUDA
    assert np.array_equal(oracle_mod.warp(g["prev"], g["bf"], v), g["warp"])
    mask, mo, mm = oracle_mod.fbcheck(g["ff"], g["bf"], variant=v, margins=True)
    assert np.array_equal(mask, g["mask"])
    assert np.array_equal(mo, g["margin_occ"]) and np.array_equal(mm, g["margin_mob"])
    assert np.array_equal(oracle_mod.validity_warp(g["prev"], g["bf"], v), g["fs_warp"])
    B, C, H, W = g["prev"].shape
    s2 = oracle_mod.masked_sums(g["mask"], g["cur"], g["warp"], 0)
    assert np.isclose(np.sqrt(s2.sum() / (B * C * H * W)), g["rmse"], rtol=1e-5, atol=0)


def test_cuda_and_cpu_flavours_differ_only_at_ulp_level(oracle_mod, tcl):
    ff, bf, prev, _ = _synth_case(tcl, 1, 64, 96, seed=9, max_shift=10.0, kind="white")
    a = oracle_mod.warp(prev.numpy(), bf.numpy(), oracle_mod.ATEN_CPU)
    b = oracle_mod.warp(prev.numpy(), bf.numpy(), oracle_mod.ATEN_CUDA)
    assert np.abs(a - b).max() < 1e-4
    ma = oracle_mod.fbcheck(ff.numpy(), bf.numpy(), variant=oracle_mod.ATEN_CPU)
    mb = oracle_mod.fbcheck(ff.numpy(), bf.numpy(), variant=oracle_mod.ATEN_CUDA)
    assert (ma != mb).mean() < 1e-3


def _raft_upsample_flow(flow, mask):
    """RAFT.upsample_flow as published with RAFT (core/raft.py; vendored upstream as utils/raft/raft/raft.py:72-83):
    softmax over the 9 logits, unfold of 8*flow, weighted sum, permute -- the formulation torch_port restates with shifts."""
    import torch.nn.functional as F
    N, _, H, W = flow.shape
    mask = torch.softmax(mask.view(N, 1, 9, 8, 8, H, W), dim=2)
    up_flow = F.unfold(8 * flow, [3, 3], padding=1).view(N, 2, 9, 1, 1, H, W)
    up_flow = torch.sum(mask * up_flow, dim=2).permute(0, 1, 4, 2, 5, 3)
    return up_flow.reshape(N, 2, 8 * H, 8 * W)


def test_upsample_restatement_matches_reference_raft():
    """oracle/torch_port.upsample_flow against RAFT's own unfold formulation of upsample_flow (CPU)."""
    g = torch.Generator().manual_seed(7)
    for (n, h, w) in [(1, 6, 7), (2, 9, 11), (1, 55, 128)]:
        flow = torch.randn(n, 2, h, w, generator=g) * 5
        mask = torch.randn(n, 576, h, w, generator=g) * 3
        want = _raft_upsample_flow(flow, mask)
        got = tp.upsample_flow(flow, mask)
        assert got.shape == want.shape
        assert torch.allclose(got, want, rtol=1e-6, atol=1e-6)
