"""NumPy / OpenCV flavour of the path (SURVEY.md section 8f rank 4): oracle pinning on CPU, kernel parity on the GPU.

CPU suite: ``oracle/cv2_port.py`` (a NumPy restatement of cv2.remap's fixed-point bilinear sampling and of the
generators' ``fb_check``) is pinned bit for bit against ``cv2.remap`` itself and against small golden vectors made by the
reference's own functions (tests/golden/make_golden_cv2.py).
GPU suite: ``tcl_b200.cv2compat`` (csrc/tcl_cv2.cu) against the oracle -- bit-exact for the remap (tolerance 0) and the
mask -- and against the golden vectors.
"""
import numpy as np
import pytest
import torch

from conftest import golden_files, load_npz
from oracle import cv2_port as cp


def flows(H, W, amp, seed):
    rng = np.random.default_rng(seed)
    yy, xx = np.mgrid[0:H, 0:W]
    bf = np.stack([amp * np.sin(xx / 17 + yy / 29), amp * np.cos(xx / 23 - yy / 13)], -1).astype(np.float32)
    bf += rng.normal(0, 0.02, (H, W, 2)).astype(np.float32)
    bf[H // 3:H // 2, W // 4:W // 2] += np.float32(3.0)          # a moving rectangle: interior motion boundary
    ff = -bf + rng.normal(0, 0.2, (H, W, 2)).astype(np.float32)
    img = rng.standard_normal((H, W, 3)).astype(np.float32)
    return ff, bf, img


CASES = [(64, 96, 0.5, 0), (37, 53, 4.0, 1), (128, 200, 30.0, 2), (2, 2, 1.0, 3), (5, 3, 0.7, 4)]


# ------------------------------------------------------------------ CPU: pin the oracle
@pytest.mark.parametrize("H,W,amp,seed", CASES)
def test_oracle_remap_equals_cv2_bitwise(H, W, amp, seed):
    cv2 = pytest.importorskip("cv2")
    ff, bf, img = flows(H, W, amp, seed)
    x, y = cp.sample_maps(bf)
    assert np.array_equal(cp.remap_linear(img, x, y), cv2.remap(img, x, y, cv2.INTER_LINEAR))
    assert np.array_equal(cp.remap_linear(ff, x, y), cv2.remap(ff, x, y, cv2.INTER_LINEAR))
    assert np.array_equal(cp.remap_linear(img[..., 0], x, y), cv2.remap(img[..., 0], x, y, cv2.INTER_LINEAR))


def test_oracle_remap_extreme_coordinates_equal_cv2():
    cv2 = pytest.importorskip("cv2")
    rng = np.random.default_rng(9)
    A = rng.standard_normal((16, 16)).astype(np.float32)
    x = np.tile(np.arange(16, dtype=np.float32), (16, 1))
    y = np.tile(np.arange(16, dtype=np.float32)[:, None], (1, 16))
    x[0, :10] = [1e10, -1e10, np.inf, -np.inf, np.nan, 15.49, 15.5, -0.5, -0.51, 14.984375]
    y[1, :6] = [np.nan, 1e30, -1.0, -0.015625, 15.984375, 16.0]
    assert np.array_equal(cp.remap_linear(A, x, y), cv2.remap(A, x, y, cv2.INTER_LINEAR))


@pytest.mark.parametrize("path", golden_files("ref_cv2_"))
def test_oracle_equals_golden(path):
    """ref_cv2_*.npz: outputs of the generators' warp_flow / warp_image (coco-generation.py:66-113) and of both fb_check
    variants (coco: occlusion test only; hollywood2-generation.py:63-111: both tests)."""
    g = load_npz(path)
    wf = cp.warp_flow(g["ff"], g["bf"])
    assert np.array_equal(wf, g["warped_flow"])
    assert np.array_equal(cp.warp_flow(g["img"], g["bf"]), g["warped_img"])
    assert np.array_equal(cp.fb_check(wf, g["bf"], motion_boundaries=False), g["mask_occ"])
    assert np.array_equal(cp.fb_check(wf, g["bf"], motion_boundaries=True), g["mask_both"])


def test_known_answers():
    # np.gradient is one-sided at the borders (not the zero padding of flowtools.gradient)
    f = np.arange(12, dtype=np.float32).reshape(3, 4) ** 2
    gy, gx = cp.gradient_np(f)
    assert np.array_equal(gy, np.gradient(f)[0]) and np.array_equal(gx, np.gradient(f)[1])
    # zero flow IS the identity here (the torch path's size-1 quirk does not exist in the cv2 flavour)
    img = np.random.default_rng(0).standard_normal((8, 9, 3)).astype(np.float32)
    assert np.array_equal(cp.warp_flow(img, np.zeros((8, 9, 2), np.float32)), img)
    # consistent constant flows keep everything; inconsistent ones nothing
    one = np.ones((8, 9, 2), np.float32)
    assert cp.fb_check(-one, one).min() == 1.0 and cp.fb_check(one * 3, one * 3).max() == 0.0


# ------------------------------------------------------------------ GPU: kernels vs the oracle
def _masks_equal_outside_band(got, want, m_occ, m_mob, use_mob):
    band = np.abs(m_occ) < 1e-6
    if use_mob:
        band |= np.abs(m_mob) < 1e-6
    ne = got != want
    assert not (ne & ~band).any(), f"{int((ne & ~band).sum())} mask mismatches outside the 1e-6 band"
    return int(ne.sum()), int(band.sum())


@pytest.mark.gpu
@pytest.mark.parametrize("H,W,amp,seed", CASES + [(436, 1024, 12.0, 7), (256, 256, 40.0, 8)])
def test_kernels_equal_oracle(tcl, H, W, amp, seed):
    d = torch.device("cuda:0")
    ff, bf, img = flows(H, W, amp, seed)
    cc = tcl.cv2compat
    # remap: tolerance 0 (every product and sum is rounded exactly like cv2 does)
    assert np.array_equal(cc.warp_image(img, bf), cp.warp_flow(img, bf))
    wf = cc.warp_flow(ff, bf)
    assert np.array_equal(wf, cp.warp_flow(ff, bf))
    assert np.array_equal(cc.warp_flow(img[..., 0], bf), cp.warp_flow(img[..., 0], bf))          # (H,W) single channel
    img5 = np.concatenate([img, img[..., :2]], -1)
    assert np.array_equal(cc.warp_flow(img5, bf), cp.warp_flow(img5, bf))                        # C = 5: runtime channel loop
    for mob in (False, True):
        want, m_occ, m_mob = cp.fb_check(wf, bf, motion_boundaries=mob, margins=True)
        got = cc.fb_check(wf, bf, motion_boundaries=mob)                                          # the reference's two-argument form
        assert got.dtype == np.float64
        _masks_equal_outside_band(got, want, m_occ, m_mob, mob)
        fused, near = cc.fb_check_flows(torch.from_numpy(ff).to(d), torch.from_numpy(bf).to(d), motion_boundaries=mob,
                                        return_near=True)                                         # one pass, on the device
        assert fused.is_cuda and fused.dtype == torch.float32
        n_ne, n_band = _masks_equal_outside_band(fused.cpu().numpy(), want, m_occ, m_mob, mob)
        assert int(near) == n_band, "near-threshold count must equal the oracle's band count"
        assert n_ne == 0, "observed: identical also inside the band"
    # batched device tensors stay on the device
    b2 = torch.from_numpy(np.stack([bf, -bf])).to(d)
    i2 = torch.from_numpy(np.stack([img, img[::-1].copy()])).to(d)
    out = cc.warp_image(i2, b2)
    assert out.is_cuda and out.shape == i2.shape
    assert np.array_equal(out[1].cpu().numpy(), cp.warp_flow(img[::-1].copy(), -bf))


@pytest.mark.gpu
def test_kernels_extreme_and_nonfinite_flows(tcl):
    rng = np.random.default_rng(3)
    H, W = 24, 40
    img = rng.standard_normal((H, W, 3)).astype(np.float32)
    fl = rng.uniform(-60, 60, (H, W, 2)).astype(np.float32)
    fl[0, :6, 0] = [np.nan, np.inf, -np.inf, 1e30, -1e30, 3e9]
    fl[1, :3, 1] = [np.nan, 1e12, -0.5]
    assert np.array_equal(tcl.cv2compat.warp_image(img, fl), cp.warp_flow(img, fl))


@pytest.mark.gpu
@pytest.mark.parametrize("path", golden_files("ref_cv2_"))
def test_kernels_equal_reference_golden(tcl, path):
    """vectors produced by the reference's own functions (cv2 + NumPy) in the build container"""
    g = load_npz(path)
    cc = tcl.cv2compat
    assert np.array_equal(cc.warp_flow(g["ff"], g["bf"]), g["warped_flow"])
    assert np.array_equal(cc.warp_image(g["img"], g["bf"]), g["warped_img"])
    assert np.array_equal(cc.fb_check(g["warped_flow"], g["bf"], motion_boundaries=False), g["mask_occ"])
    assert np.array_equal(cc.fb_check(g["warped_flow"], g["bf"], motion_boundaries=True), g["mask_both"])
    assert np.array_equal(cc.fb_check_flows(g["ff"], g["bf"], motion_boundaries=True), g["mask_both"])


@pytest.mark.gpu
def test_errors(tcl):
    cc = tcl.cv2compat
    with pytest.raises(AssertionError):
        cc.warp_flow(np.zeros((4, 5, 3), np.float32), np.zeros((4, 6, 2), np.float32))      # the reference's assert
    with pytest.raises(RuntimeError):
        cc.fb_check(np.zeros((1, 5, 2), np.float32), np.zeros((1, 5, 2), np.float32))       # np.gradient needs >= 2 rows
    with pytest.raises(RuntimeError):
        cc.warp_flow(torch.zeros(4, 5, 3), torch.zeros(4, 5, 2))                            # CPU tensors: no CPU path
