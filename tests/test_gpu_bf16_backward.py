"""GPU suite: autograd of warp, fs_lib.warp and the temporal losses for bf16 frames.

The oracle is what the reference computes under ``torch.autocast("cuda", torch.bfloat16)``: grid_sampler is on autocast's
fp32 list and ``mask*(cur - w)`` promotes to fp32, so the loss is the fp32 expression of ``oracle/torch_port`` on the upcast
frames, and autograd casts each frame's gradient back to bf16.  ``want32`` below is that fp32 gradient; a bf16 gradient
is accepted when ``|got - want32| <= 2^-8 |want32| + 1e-5 max|want32|`` elementwise (the bf16 rounding, plus the fp32
tolerance the fp32 backward tests use for the reordered scatter-add)."""
import pytest
import torch
import torch.nn.functional as F

from oracle import torch_port as tp

pytestmark = pytest.mark.gpu

BF16 = torch.bfloat16


def _tol(want32):
    return 2.0 ** -8 * want32.abs() + 1e-5 * float(want32.abs().max())


def assert_bf16_grad(got, want32):
    assert got.dtype == BF16
    err = (got.float() - want32).abs() - _tol(want32)
    assert float(err.max()) <= 0.0, f"{int((err > 0).sum())} of {err.numel()} elements outside the tolerance"


def assert_within_one_ulp(got, other):
    """Two bf16 roundings of nearly equal fp32 values (the scatter-add's atomics reorder): at most one bf16 ulp apart."""
    assert got.dtype == BF16 and other.dtype == BF16
    t = other.float()
    err = (got.float() - t).abs() - (2.0 ** -7 * t.abs() + 1e-5 * float(t.abs().max()))
    assert float(err.max()) <= 0.0, f"{int((err > 0).sum())} of {err.numel()} elements more than one ulp apart"


def _frames(tcl, B, C, H, W, seed, shift, kind="white"):
    d = torch.device("cuda:0")
    ff, bf = tcl.synth.make_flows(B, H, W, seed=seed, max_shift=shift, device=d)
    prev, cur = (t.to(d).to(BF16) for t in tcl.synth.make_frames(B, C, H, W, seed=seed, kind=kind))
    return ff, bf, prev, cur


def _soften(mask):
    H, W = mask.shape[2:]
    return F.interpolate(F.avg_pool2d(mask, 2), size=(H, W), mode="bilinear")


WARP_SHAPES = [(2, 3, 32, 48, 4.0), (16, 3, 256, 256, 24.0), (1, 3, 436, 1024, 32.0), (1, 5, 37, 53, 20.0), (2, 32, 64, 64, 6.0)]


@pytest.mark.parametrize("which", ["warp", "fs_warp"])
@pytest.mark.parametrize("B,C,H,W,shift", WARP_SHAPES)
def test_warp_backward_bf16(tcl, which, B, C, H, W, shift):
    _, bf, prev, _ = _frames(tcl, B, C, H, W, 81, shift)
    go = torch.randn(prev.shape, device=prev.device).to(BF16)
    ours, ref = (tcl.warp, tp.backward_warp) if which == "warp" else (tcl.fs_warp, tp.validity_warp)
    # oracle: the fp32 expression on the upcast frame and upstream gradient
    x32, f32 = prev.float().requires_grad_(True), bf.clone().requires_grad_(True)
    ref(x32, f32).backward(go.float())
    # ours on the bf16 frame
    x, f = prev.clone().requires_grad_(True), bf.clone().requires_grad_(True)
    out = ours(x, f)
    assert out.dtype == BF16
    out.backward(go)
    assert_bf16_grad(x.grad, x32.grad)
    # the flow gradient is computed per pixel without atomics: bit for bit the fp32 entry's on the upcast tensors
    fk = bf.clone().requires_grad_(True)
    ours(prev.float(), fk).backward(go.float())
    assert f.grad.dtype == torch.float32 and torch.equal(f.grad, fk.grad)
    # only one of the two gradients requested
    x1 = prev.clone().requires_grad_(True)
    ours(x1, bf).backward(go)
    assert_bf16_grad(x1.grad, x32.grad)
    f1 = bf.clone().requires_grad_(True)
    ours(prev, f1).backward(go)
    assert torch.equal(f1.grad, fk.grad)


@pytest.mark.parametrize("loss", ["l2", "l1"])
@pytest.mark.parametrize("validity", [False, True])
@pytest.mark.parametrize("soft", [False, True])
@pytest.mark.parametrize("B,H,W,shift", [(2, 32, 48, 4.0), (16, 256, 256, 24.0)])
def test_temporal_loss_backward_bf16(tcl, loss, validity, soft, B, H, W, shift):
    ff, bf, prev, cur = _frames(tcl, B, 3, H, W, 91, shift)
    mask = tcl.fbcCheckTorch(ff, bf)
    if soft:
        mask = _soften(mask)
    warp_ref = tp.validity_warp if validity else tp.backward_warp
    crit = tp.tcl_l2 if loss == "l2" else tp.tcl_l1
    p32, c32 = prev.float().requires_grad_(True), cur.float().requires_grad_(True)
    want = crit(mask, c32, warp_ref(p32, bf))
    (want * 100.0).backward()                                   # lambda_tcl = 100 (main.py:94)
    p, c = prev.clone().requires_grad_(True), cur.clone().requires_grad_(True)
    got = tcl.temporal_loss(mask, c, p, bf, loss=loss, validity=validity)
    assert got.dtype == torch.float32 and got.dim() == 0
    (got * 100.0).backward()
    assert abs(got.item() - want.item()) <= 1e-5 * abs(want.item())
    # grad_cur: the fp32 kernel's on the upcast frames, rounded once
    pk, ck = prev.float().requires_grad_(True), cur.float().requires_grad_(True)
    (tcl.temporal_loss(mask, ck, pk, bf, loss=loss, validity=validity) * 100.0).backward()
    assert c.grad.dtype == BF16 and torch.equal(c.grad, ck.grad.to(BF16))
    assert_bf16_grad(p.grad, p32.grad)
    # one frame only
    p1 = prev.clone().requires_grad_(True)
    (tcl.temporal_loss(mask, cur, p1, bf, loss=loss, validity=validity) * 100.0).backward()
    assert_bf16_grad(p1.grad, p32.grad)
    c1 = cur.clone().requires_grad_(True)
    (tcl.temporal_loss(mask, c1, prev, bf, loss=loss, validity=validity) * 100.0).backward()
    assert torch.equal(c1.grad, c.grad)


@pytest.mark.parametrize("loss", ["l2", "l1"])
def test_matches_the_reference_under_autocast(tcl, loss):
    """The reference expression itself under autocast with bf16 frames: grid_sampler runs in fp32 there, and its gradients
    are those of the explicit-upcast oracle.  Ours and autocast's are two independent roundings of nearly the same fp32
    value, so they may differ by one bf16 ulp (2^-7 relative)."""
    ff, bf, prev, cur = _frames(tcl, 4, 3, 128, 160, 95, 12.0)
    mask = tcl.fbcCheckTorch(ff, bf)
    crit = tp.tcl_l2 if loss == "l2" else tp.tcl_l1
    pa, ca = prev.clone().requires_grad_(True), cur.clone().requires_grad_(True)
    with torch.autocast("cuda", dtype=torch.bfloat16):
        w = tp.backward_warp(pa, bf)
        assert w.dtype == torch.float32, "autocast did not run grid_sampler in fp32"
        ref = crit(mask, ca, w)
    assert ref.dtype == torch.float32
    (ref * 100.0).backward()
    p32, c32 = prev.float().requires_grad_(True), cur.float().requires_grad_(True)
    (crit(mask, c32, tp.backward_warp(p32, bf)) * 100.0).backward()
    assert_bf16_grad(pa.grad, p32.grad)
    assert_bf16_grad(ca.grad, c32.grad)
    p, c = prev.clone().requires_grad_(True), cur.clone().requires_grad_(True)
    got = tcl.temporal_loss(mask, c, p, bf, loss=loss)
    (got * 100.0).backward()
    assert abs(got.item() - ref.item()) <= 1e-5 * abs(ref.item())
    assert_within_one_ulp(p.grad, pa.grad)
    assert_within_one_ulp(c.grad, ca.grad)


@pytest.mark.parametrize("loss", ["l2", "l1"])
@pytest.mark.parametrize("B,C,H,W,shift", [(2, 3, 64, 96, 8.0), (1, 5, 37, 53, 20.0)])
def test_learnable_flow_and_mask_bf16(tcl, loss, B, C, H, W, shift):
    """MoGAN's learnable flow / a trained soft mask with bf16 frames: the composed branch.  Its value is an fp32 scalar and
    all four gradients match the oracle."""
    ff, bf, prev, cur = _frames(tcl, B, C, H, W, 97, shift)
    mask = _soften(tcl.fbcCheckTorch(ff, bf))
    crit = tp.tcl_l2 if loss == "l2" else tp.tcl_l1
    p32, c32 = prev.float().requires_grad_(True), cur.float().requires_grad_(True)
    f32, m32 = bf.clone().requires_grad_(True), mask.clone().requires_grad_(True)
    want = crit(m32, c32, tp.backward_warp(p32, f32))
    (want * 100.0).backward()
    p, c = prev.clone().requires_grad_(True), cur.clone().requires_grad_(True)
    f, m = bf.clone().requires_grad_(True), mask.clone().requires_grad_(True)
    got = tcl.temporal_loss(m, c, p, f, loss=loss)
    assert got.dtype == torch.float32 and got.dim() == 0
    (got * 100.0).backward()
    assert abs(got.item() - want.item()) <= 1e-5 * abs(want.item())
    assert_bf16_grad(p.grad, p32.grad)
    assert_bf16_grad(c.grad, c32.grad)
    assert f.grad.dtype == torch.float32 and m.grad.dtype == torch.float32
    assert float((f.grad - f32.grad).abs().max()) <= 1e-4 * max(1.0, float(f32.grad.abs().max()))
    assert float((m.grad - m32.grad).abs().max()) <= 1e-5 * float(m32.grad.abs().max())


def test_generate_mask_bf16(tcl):
    """ConGAN's soft mask exp(-50 * |simg - warp(prev)|.mean()) (cycle_gan_model.py:136-137) on bf16 frames."""
    ff, bf, prev, cur = _frames(tcl, 4, 3, 64, 96, 61, 6.0)
    cur = (prev.float() + 0.01 * cur.float()).to(BF16)
    c32 = cur.float().requires_grad_(True)
    want = torch.exp(-50 * torch.abs(c32 - tp.backward_warp(prev.float(), bf)).mean())
    want.backward()
    c = cur.clone().requires_grad_(True)
    got = tcl.generateMask(c, prev, bf)
    assert got.dtype == torch.float32 and abs(got.item() - want.item()) <= 1e-5 * want.item()
    got.backward()
    assert_bf16_grad(c.grad, c32.grad)


def test_other_frame_dtypes_still_raise(tcl):
    _, bf, prev, cur = _frames(tcl, 1, 3, 16, 16, 5, 2.0)
    with pytest.raises(RuntimeError, match="float32 or bfloat16"):
        tcl.warp(prev.half().requires_grad_(True), bf)
    with pytest.raises(RuntimeError, match="float32 or bfloat16"):
        tcl.temporal_loss(None, cur.half().requires_grad_(True), prev.half(), bf)


@pytest.mark.parametrize("loss", ["l2", "l1"])
def test_cuda_graph_replay_equals_eager(tcl, loss):
    """bf16 forward + backward of the training loss captured in a CUDA graph: the workspace comes from the graph's pool and
    the replay on new inputs equals the eager call (grad_cur bit for bit; grad_prev within one bf16 ulp, the atomics reorder)."""
    B, H, W = 16, 256, 256
    ff, bf, prev, cur = _frames(tcl, B, 3, H, W, 111, 24.0)
    mask = tcl.fbcCheckTorch(ff, bf)
    p, c = prev.clone().requires_grad_(True), cur.clone().requires_grad_(True)

    def step():
        val = tcl.temporal_loss(mask, c, p, bf, loss=loss)
        return (val,) + torch.autograd.grad(val * 100.0, (p, c))
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(2):
            step()
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        g_val, g_gp, g_gc = step()
    _, bf2, prev2, cur2 = _frames(tcl, B, 3, H, W, 112, 24.0)
    with torch.no_grad():
        p.copy_(prev2)
        c.copy_(cur2)
        bf.copy_(bf2)
    graph.replay()
    torch.cuda.synchronize()
    e_val, e_gp, e_gc = step()
    assert torch.equal(g_val, e_val)
    assert torch.equal(g_gc, e_gc)
    assert_within_one_ulp(g_gp, e_gp)
