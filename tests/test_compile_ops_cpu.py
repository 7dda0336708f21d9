"""The torch.library operators of ``library.py`` without a GPU: registration and schemas, the public functions under
FakeTensorMode with fake CUDA tensors (output metadata, no CUDA initialisation), make_fx graphs (fake and symbolic), and
validation errors that read as in eager.

Without a device, the autograd engine refuses to run a backward over CUDA tensors (it checks the device's context), so
these tests call the backward nodes themselves (``grad_fn.apply``); tests/test_gpu_under_compile.py traces through
``torch.autograd.grad``."""
import pytest
import torch
from torch._subclasses.fake_tensor import FakeTensorMode
from torch.fx.experimental.proxy_tensor import make_fx

from torch._dynamo.source import ConstantSource
from torch.fx.experimental.symbolic_shapes import DimDynamic, ShapeEnv, StatelessSymbolicContext

import tcl_b200
from tcl_b200 import ops

SCHEMAS = {
    "gradient": "tcl_b200::gradient(Tensor x) -> Tensor",
    "warp": "tcl_b200::warp(Tensor x, Tensor f, SymInt flags) -> Tensor",
    "warp_backward": "tcl_b200::warp_backward(Tensor grad_out, Tensor x, Tensor f, SymInt flags, bool need_x, bool need_f) -> (Tensor, Tensor)",
    "fbcheck": "tcl_b200::fbcheck(Tensor? ff, Tensor bf, SymInt flags, bool want_near) -> Tensor[]",
    "upsample_flow": "tcl_b200::upsample_flow(Tensor flow, Tensor mask) -> Tensor",
    "temporal_loss": "tcl_b200::temporal_loss(Tensor prev, Tensor cur, Tensor flow, Tensor mask, SymInt loss, SymInt flags) -> Tensor",
    "temporal_loss_backward": "tcl_b200::temporal_loss_backward(Tensor grad_out, Tensor prev, Tensor cur, Tensor flow, Tensor mask, "
                              "SymInt loss, SymInt flags, bool need_prev, bool need_cur) -> (Tensor, Tensor)",
    "fused_eval": "tcl_b200::fused_eval(Tensor bf, Tensor prev, Tensor cur, Tensor? ff, Tensor? mask, SymInt loss, SymInt finalize, "
                  "SymInt what, float[]? u8_scale, float[]? u8_offset) -> Tensor[]",
    "reconet_loss": "tcl_b200::reconet_loss(Tensor styled2, Tensor styled1, Tensor img2, Tensor img1, Tensor flow, Tensor? mask) "
                    "-> (Tensor, Tensor)",
    "reconet_loss_backward": "tcl_b200::reconet_loss_backward(Tensor grad_out, Tensor styled1, Tensor styled2, Tensor flow, Tensor? mask, "
                             "Tensor lum, bool need2, bool need1) -> (Tensor, Tensor)",
    "ruder_input": "tcl_b200::ruder_input(Tensor styled_prev, Tensor img, Tensor? mask, Tensor flow) -> (Tensor, Tensor)",
}

B, C, H, W = 2, 3, 16, 24
CUDA = torch.device("cuda", 0)


def meta(t, shape, dtype, device=CUDA):
    assert tuple(t.shape) == tuple(shape) and t.dtype == dtype and t.device == device, (t.shape, t.dtype, t.device)


@pytest.fixture(autouse=True)
def no_cuda_init():
    yield
    assert not torch.cuda.is_initialized()


def test_operators_are_registered_with_their_schemas():
    for name, schema in SCHEMAS.items():
        assert str(getattr(torch.ops.tcl_b200, name).default._schema) == schema


def fake_inputs(mode, dtype=torch.float32, grad=False, n=B, h=H, w=W):
    with mode:
        prev = torch.rand(n, C, h, w, device=CUDA).to(dtype)
        cur = torch.rand(n, C, h, w, device=CUDA).to(dtype)
        ff = torch.randn(n, 2, h, w, device=CUDA)
        bf = torch.randn(n, 2, h, w, device=CUDA)
        mask = torch.rand(n, 1, h, w, device=CUDA)
        if grad:
            prev.requires_grad_(True)
            cur.requires_grad_(True)
    return prev, cur, ff, bf, mask


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("grad", [False, True])
def test_warp_fbcheck_gradient_upsample_under_fake_mode(dtype, grad):
    mode = FakeTensorMode()
    prev, cur, ff, bf, mask = fake_inputs(mode, dtype, grad)
    with mode:
        for fn in (tcl_b200.warp, tcl_b200.fs_warp):
            out = fn(prev, bf)
            meta(out, prev.shape, dtype)
            assert out.requires_grad == grad
        meta(tcl_b200.fbcCheckTorch(ff, bf), (B, 1, H, W), torch.float32)
        meta(tcl_b200.fbcCheckTorch_mob(ff, bf), (B, 1, H, W), torch.float32)
        m, near = tcl_b200.fbcheck_with_near_count(ff, bf)
        meta(m, (B, 1, H, W), torch.float32)
        meta(near, (1,), torch.int64)
        meta(tcl_b200.gradient(bf[:, 0]), (2, B, H, W), torch.float32)
        up = tcl_b200.upsample_flow(bf, torch.rand(B, 576, H, W, device=CUDA))
        meta(up, (B, 2, 8 * H, 8 * W), torch.float32)


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("loss", ["l2", "l1"])
@pytest.mark.parametrize("validity", [False, True])
@pytest.mark.parametrize("mask_kind", ["dataset", "none"])
@pytest.mark.parametrize("grad", [False, True])
def test_temporal_loss_under_fake_mode(dtype, loss, validity, mask_kind, grad):
    mode = FakeTensorMode()
    prev, cur, ff, bf, mask = fake_inputs(mode, dtype, grad)
    with mode:
        m = mask if mask_kind == "dataset" else None
        out = tcl_b200.temporal_loss(m, cur, prev, bf, loss=loss, validity=validity)
        meta(out, (), torch.float32)
        assert out.requires_grad == grad
        if grad:
            gp, gc = out.grad_fn.apply(torch.ones_like(out))[:2]
            meta(gp, prev.shape, dtype)
            meta(gc, cur.shape, dtype)
        g = tcl_b200.generateMask(cur, prev, bf)
        meta(g, (), torch.float32)


def test_temporal_loss_with_learnable_flow_and_computed_mask_under_fake_mode():
    mode = FakeTensorMode()
    prev, cur, ff, bf, mask = fake_inputs(mode, grad=True)
    with mode:
        bf.requires_grad_(True)
        out = tcl_b200.temporal_loss(tcl_b200.fbcCheckTorch(ff, bf.detach()), cur, prev, bf)
        meta(out, (), torch.float32)
        assert out.requires_grad


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16, torch.uint8])
def test_evaluation_helpers_under_fake_mode(dtype):
    mode = FakeTensorMode()
    prev, cur, ff, bf, mask = fake_inputs(mode)
    with mode:
        if dtype == torch.uint8:
            prev, cur = (prev * 255).to(torch.uint8), (cur * 255).to(torch.uint8)
        else:
            prev, cur = prev.to(dtype), cur.to(dtype)
        u8 = dict(u8_scale=[0.5, 0.25, 1.0], u8_offset=-0.5) if dtype == torch.uint8 else {}
        meta(tcl_b200.temporal_error(ff, bf, prev, cur, **u8), (), torch.float32)
        meta(tcl_b200.temporal_error_per_pair(ff, bf, prev, cur, **u8), (B,), torch.float32)
        meta(tcl_b200.temporal_rmse_per_sample(mask, cur, prev, bf, **u8), (B,), torch.float32)
        for kw in (dict(ff=ff), dict(ff=None, mask=mask), dict(ff=None)):
            for loss in (ops.L2, ops.L1):
                meta(tcl_b200.warping_error_per_pair(bf=bf, prev=prev, cur=cur, loss=loss, **kw, **u8), (B,), torch.float32)
        meta(tcl_b200.computeTCL_from_flows(ff, bf, prev, cur), (), torch.float32)
        if dtype != torch.uint8:
            meta(tcl_b200.warp_blend(mask, prev, bf, cur), prev.shape, dtype)
            m, pre = tcl_b200.long_term_blend_step(mask, ff, bf, prev, cur)
            meta(m, (B, 1, H, W), torch.float32)
            meta(pre, prev.shape, dtype)


@pytest.mark.parametrize("grad", [False, True])
@pytest.mark.parametrize("with_mask", [False, True])
def test_chains_under_fake_mode(grad, with_mask):
    mode = FakeTensorMode()
    prev, cur, ff, bf, mask = fake_inputs(mode, grad=grad)
    with mode:
        m = mask if with_mask else None
        img2, img1 = torch.rand(B, 3, H, W, device=CUDA), torch.rand(B, 3, H, W, device=CUDA)
        loss = tcl_b200.reconet_output_temporal_loss(m, cur, prev, img2, img1, bf)
        meta(loss, (), torch.float32)
        cat, warped = tcl_b200.ruder_network_input(img2, mask, prev, bf)
        meta(cat, (B, 7, H, W), torch.float32)
        meta(warped, (B, 3, H, W), torch.float32)
        if grad:
            g2, g1 = loss.grad_fn.apply(torch.ones_like(loss), torch.zeros(B, 1, H, W, device=CUDA))[:2]
            meta(g2, cur.shape, torch.float32)
            meta(g1, prev.shape, torch.float32)
            gp = cat.grad_fn.apply(torch.ones_like(cat), torch.ones_like(warped))[0]
            meta(gp, prev.shape, torch.float32)


def training_loss(prev, cur, flow, mask):
    """warp -> temporal_loss -> the backward of both, node by node."""
    w = tcl_b200.warp(prev, flow)
    loss = tcl_b200.temporal_loss(mask, cur, w, flow)
    g_w, g_cur = loss.grad_fn.apply(torch.ones_like(loss))[:2]
    g_prev = w.grad_fn.apply(g_w)[0]
    return loss, g_prev, g_cur


def symbolic_inputs():
    mode = FakeTensorMode(shape_env=ShapeEnv())

    def fake(shape, name):
        t = mode.from_tensor(torch.empty(shape), source=ConstantSource(name),
                             symbolic_context=StatelessSymbolicContext(dynamic_sizes=[DimDynamic.DYNAMIC] * len(shape)))
        with mode:
            return t.to(CUDA)
    prev, cur = fake((B, C, H, W), "prev").requires_grad_(), fake((B, C, H, W), "cur").requires_grad_()
    return prev, cur, fake((B, 2, H, W), "flow"), fake((B, 1, H, W), "mask")


@pytest.mark.parametrize("tracing_mode", ["fake", "symbolic"])
def test_make_fx_graph_calls_the_operators(tracing_mode):
    if tracing_mode == "fake":
        prev, cur, ff, bf, mask = fake_inputs(FakeTensorMode(), grad=True)
        args = (prev, cur, bf, mask)
    else:
        args = symbolic_inputs()
    gm = make_fx(training_loss, tracing_mode=tracing_mode)(*args)
    targets = [str(n.target) for n in gm.graph.nodes if n.op == "call_function"]
    for op in ("tcl_b200.warp.default", "tcl_b200.temporal_loss.default", "tcl_b200.temporal_loss_backward.default",
               "tcl_b200.warp_backward.default"):
        assert op in targets, targets
    assert all(t.startswith("tcl_b200.") or t in ("aten.ones_like.default", "<built-in function getitem>") for t in targets), targets
    if tracing_mode == "symbolic":
        shapes = [n.meta["val"].shape for n in gm.graph.nodes if n.op == "placeholder"]
        assert all(isinstance(d, torch.SymInt) for d in shapes[0]), shapes


def errors(fn):
    try:
        fn()
    except RuntimeError as e:
        return str(e)
    raise AssertionError("no error")


def test_validation_errors_match_eager_messages_under_fake_mode():
    # the eager messages, from the validation that runs before any routing (eager calls raise them before any launch)
    cases = [
        (lambda t: tcl_b200.warp(t["prev"], t["bf"][:, :, :8]), "do not match"),
        (lambda t: tcl_b200.warp(t["prev"].half(), t["bf"]), "frames must be float32 or bfloat16"),
        (lambda t: tcl_b200.temporal_loss(None, t["cur"][:1], t["prev"], t["bf"]), "must be (B,C,H,W) frames matching the flow"),
        (lambda t: tcl_b200.temporal_loss(t["mask"][:, :, :8], t["cur"], t["prev"], t["bf"]), "mask must be (B,1,H,W)"),
        (lambda t: tcl_b200.temporal_error(t["ff"], t["bf"], t["prev"], t["cur"].to(torch.bfloat16)), "same frame shape and dtype"),
        (lambda t: tcl_b200.temporal_error(t["ff"], t["bf"], t["prev"], t["cur"], u8_scale=0.5), "apply to uint8 frames only"),
        (lambda t: tcl_b200.temporal_error(t["ff"], t["bf"], (t["prev"] * 255).to(torch.uint8), (t["cur"] * 255).to(torch.uint8),
                                           u8_scale=float("inf")), "u8_scale must be finite"),
        (lambda t: tcl_b200.fbcCheckTorch(t["ff"][:1], t["bf"]), "do not match"),
        (lambda t: tcl_b200.upsample_flow(t["bf"], t["mask"]), "mask must be (N,576,H,W)"),
        (lambda t: tcl_b200.gradient(t["bf"]), "gradient expects (B,H,W)"),
        (lambda t: tcl_b200.ruder_network_input(t["cur"][:, :2], None, t["prev"], t["bf"]), "must be (B,3,H,W)"),
    ]
    mode = FakeTensorMode()
    prev, cur, ff, bf, mask = fake_inputs(mode)
    t = dict(prev=prev, cur=cur, ff=ff, bf=bf, mask=mask)
    for fn, text in cases:
        with mode:
            msg = errors(lambda: fn(t))
        assert text in msg, (text, msg)


def test_cpu_tensors_raise_before_routing():
    with pytest.raises(RuntimeError, match="expected CUDA tensors"):
        tcl_b200.warp(torch.zeros(1, 3, 4, 4), torch.zeros(1, 2, 4, 4))
    mode = FakeTensorMode()
    with mode:
        x, f = torch.zeros(1, 3, 4, 4), torch.zeros(1, 2, 4, 4)
        with pytest.raises(RuntimeError, match="expected CUDA tensors"):
            tcl_b200.warp(x, f)


def test_u8_normalisation_rounds_like_an_fp32_tensor():
    for v in (1.0 / 255.0, 0.1, 1e-30, 3.4028234663852886e38, -2.5):
        (s, _, _), _ = ops._u8_norm(ops.U8, v, None, 3)
        assert s == float(torch.tensor(v, dtype=torch.float32))
    for v in (float("nan"), float("inf"), 1e39):
        with pytest.raises(RuntimeError, match="u8_scale must be finite"):
            ops._u8_norm(ops.U8, v, None, 3)
