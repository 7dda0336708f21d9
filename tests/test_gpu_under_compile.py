"""GPU suite: the torch.library operators of ``library.py`` and the public functions under torch.compile.

opcheck of every operator; no graph break in functions calling each public entry; ``fullgraph=True`` compiles that give
the eager results (values, masks, warped frames, grad_cur / grad_f bit for bit; grad_prev / grad_x within the tolerance
of the backward tests, since the scatter's atomics reorder); a reduce-overhead (CUDA graph) training step of a stand-in
generator against the eager step; ``dynamic=True`` over two frame sizes.

The module's name sorts it after the other GPU modules.  The compiles leave process-wide state behind (dynamo and inductor
caches, cudagraph trees), and after them torch.profiler sessions in the same process were seen to miss kernels of the library,
which the launch-table tests (test_gpu_forward_plan.py, test_gpu_kept_pixels.py, test_gpu_u8_frames.py) read from the profile."""
import pytest
import torch
import torch._dynamo
from torch._dynamo.testing import CompileCounterWithBackend
from torch.fx.experimental.proxy_tensor import make_fx

import tcl_b200
from tcl_b200 import ops

# (attributes, not `from tcl_b200.ops import ...`: tcl_b200 is an alias, and importing a submodule by that name loads a second copy)
L1, L2, MOB, OCC, VALIDITY = ops.L1, ops.L2, ops.MOB, ops.OCC, ops.VALIDITY

pytestmark = pytest.mark.gpu

DEV = torch.device("cuda:0")
OPS = torch.ops.tcl_b200


def frames(B=2, C=3, H=24, W=40, dtype=torch.float32, seed=7, shift=4.0):
    ff, bf = tcl_b200.synth.make_flows(B, H, W, seed=seed, max_shift=shift, device=DEV)
    prev, cur = (t.to(DEV).to(dtype) for t in tcl_b200.synth.make_frames(B, C, H, W, seed=seed, kind="white"))
    mask = tcl_b200.fbcCheckTorch(ff, bf)
    return ff, bf, prev, cur, mask


def assert_bits(a, b):
    assert a.dtype == b.dtype and a.shape == b.shape
    assert torch.equal(a, b), float((a.float() - b.float()).abs().max())


def assert_scatter_close(a, b):
    """grad_prev / grad_x: fp32 within 1e-5 of the largest value (the atomics reorder); bf16 within one bf16 ulp."""
    assert a.dtype == b.dtype and a.shape == b.shape
    t = b.float()
    rel = 2.0 ** -7 if a.dtype == torch.bfloat16 else 1e-5
    err = (a.float() - t).abs() - (rel * t.abs() + 1e-5 * float(t.abs().max()))
    assert float(err.max()) <= 0.0


# ------------------------------------------------------------------------------------------------
# opcheck
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("flags", [0, VALIDITY])
def test_opcheck_warp(dtype, flags):
    ff, bf, prev, cur, mask = frames(dtype=dtype)
    torch.library.opcheck(OPS.warp, (prev.clone().requires_grad_(), bf.clone().requires_grad_(), flags))
    g = torch.randn_like(prev)
    for need in ((True, True), (True, False), (False, True)):
        torch.library.opcheck(OPS.warp_backward, (g, prev, bf, flags) + need)


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("loss", [L2, L1])
@pytest.mark.parametrize("flags", [0, VALIDITY])
def test_opcheck_temporal_loss(dtype, loss, flags):
    ff, bf, prev, cur, mask = frames(dtype=dtype)
    torch.library.opcheck(OPS.temporal_loss, (prev.clone().requires_grad_(), cur.clone().requires_grad_(), bf, mask, loss, flags))
    g = torch.tensor(0.75, device=DEV)
    for need in ((True, True), (True, False), (False, True)):
        torch.library.opcheck(OPS.temporal_loss_backward, (g, prev, cur, bf, mask, loss, flags) + need)


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16, torch.uint8])
@pytest.mark.parametrize("loss", [L2, L1])
def test_opcheck_fused_eval(dtype, loss):
    ff, bf, prev, cur, mask = frames()
    if dtype == torch.uint8:
        prev, cur = (prev * 255).round().to(torch.uint8), (cur * 255).round().to(torch.uint8)
        norm = ([0.5, 0.25, 1.0 / 255.0], [-0.5, 0.0, 0.0])
    else:
        prev, cur, norm = prev.to(dtype), cur.to(dtype), (None, None)
    for what in (ops.EVAL_TOTAL, ops.EVAL_PAIRS, ops.EVAL_KEPT):
        for f, m in ((ff, None), (None, mask), (None, None)):
            torch.library.opcheck(OPS.fused_eval, (bf, prev, cur, f, m, loss, ops.FIN_RMSE, what) + norm)
    if dtype != torch.uint8:
        torch.library.opcheck(OPS.fused_eval, (bf, prev, cur, None, mask, loss, ops.FIN_RMSE, ops.EVAL_BLEND, None, None))


def test_opcheck_fbcheck_gradient_upsample():
    ff, bf, prev, cur, mask = frames()
    for args in ((ff, bf, OCC | MOB, False), (ff, bf, OCC | MOB, True), (None, bf, MOB, False), (None, bf, MOB, True)):
        torch.library.opcheck(OPS.fbcheck, args)
    torch.library.opcheck(OPS.gradient, (bf[:, 0],))
    torch.library.opcheck(OPS.upsample_flow, (bf[:, :, :6, :8].contiguous(), torch.randn(2, 576, 6, 8, device=DEV)))


@pytest.mark.parametrize("with_mask", [False, True])
def test_opcheck_chains(with_mask):
    ff, bf, prev, cur, mask = frames()
    img2, img1 = torch.rand_like(cur), torch.rand_like(prev)
    m = mask if with_mask else None
    torch.library.opcheck(OPS.reconet_loss, (cur.clone().requires_grad_(), prev.clone().requires_grad_(), img2, img1, bf, m))
    loss, lum = OPS.reconet_loss(cur, prev, img2, img1, bf, m)
    g = torch.tensor(1.5, device=DEV)
    for need in ((True, True), (False, True)):
        torch.library.opcheck(OPS.reconet_loss_backward, (g, prev, cur, bf, m, lum) + need)
    torch.library.opcheck(OPS.ruder_input, (prev.clone().requires_grad_(), img2, m, bf))


# ------------------------------------------------------------------------------------------------
# graph breaks and fullgraph compiles against eager
# ------------------------------------------------------------------------------------------------
def entries():
    """{name: (fn, args, {index of an arg to differentiate: "bits" | "scatter"})} for every public entry routed through an
    operator; "scatter" marks the gradient of a warped frame."""
    ff, bf, prev, cur, mask = frames()
    u8p, u8c = (prev * 255).round().to(torch.uint8), (cur * 255).round().to(torch.uint8)
    img2, img1 = torch.rand_like(cur), torch.rand_like(prev)
    up_mask = torch.randn(2, 576, 6, 8, device=DEV)
    return {e[0]: e[1:] for e in [
        ("gradient", lambda f: tcl_b200.gradient(f[:, 0]), (bf,), {}),
        ("warp", tcl_b200.warp, (prev, bf), {0: "scatter", 1: "bits"}),
        ("fs_warp", tcl_b200.fs_warp, (prev, bf), {0: "scatter", 1: "bits"}),
        ("fbcCheckTorch", tcl_b200.fbcCheckTorch, (ff, bf), {}),
        ("fbcCheckTorch_mob", tcl_b200.fbcCheckTorch_mob, (ff, bf), {}),
        ("fbcheck_with_near_count", tcl_b200.fbcheck_with_near_count, (ff, bf), {}),
        ("upsample_flow", lambda f, m: tcl_b200.upsample_flow(f[:, :, :6, :8], m), (bf, up_mask), {}),
        ("temporal_loss_l2", lambda m, c, p, f: tcl_b200.temporal_loss(m, c, p, f), (mask, cur, prev, bf), {1: "bits", 2: "scatter"}),
        ("temporal_loss_l1_validity", lambda m, c, p, f: tcl_b200.temporal_loss(m, c, p, f, loss="l1", validity=True),
         (mask, cur, prev, bf), {1: "bits", 2: "scatter"}),
        ("temporal_loss_learnable_flow", lambda m, c, p, f: tcl_b200.temporal_loss(m, c, p, f), (mask, cur, prev, bf),
         {1: "bits", 2: "scatter", 3: "bits"}),
        ("generateMask", tcl_b200.generateMask, (cur, prev, bf), {0: "bits", 1: "scatter"}),
        ("temporal_error", tcl_b200.temporal_error, (ff, bf, prev, cur), {}),
        ("temporal_error_u8", lambda a, b, p, c: tcl_b200.temporal_error(a, b, p, c, u8_scale=0.5, u8_offset=[0.0, -0.25, 0.5]),
         (ff, bf, u8p, u8c), {}),
        ("temporal_error_per_pair", tcl_b200.temporal_error_per_pair, (ff, bf, prev, cur), {}),
        ("temporal_rmse_per_sample", tcl_b200.temporal_rmse_per_sample, (mask, cur, prev, bf), {}),
        ("warping_error_per_pair", tcl_b200.warping_error_per_pair, (ff, bf, prev, cur), {}),
        ("warping_error_per_pair_l1_mask", lambda b, p, c, m: tcl_b200.warping_error_per_pair(None, b, p, c, mask=m, loss=L1),
         (bf, prev, cur, mask), {}),
        ("warp_blend", tcl_b200.warp_blend, (mask, prev, bf, cur), {}),
        ("computeTCL_from_flows", tcl_b200.computeTCL_from_flows, (ff, bf, prev, cur), {}),
        ("reconet_output_temporal_loss", tcl_b200.reconet_output_temporal_loss, (mask, cur, prev, img2, img1, bf), {1: "bits", 2: "scatter"}),
        ("ruder_network_input", lambda i, m, s, f: sum(t.sum() for t in tcl_b200.ruder_network_input(i, m, s, f)),
         (img2, mask, prev, bf), {2: "scatter"}),
        ("long_term_blend_step", tcl_b200.long_term_blend_step, (mask, ff, bf, prev, cur), {}),
    ]}


def outputs(r):
    return list(r) if isinstance(r, (tuple, list)) else [r]


ENTRIES = ("gradient", "warp", "fs_warp", "fbcCheckTorch", "fbcCheckTorch_mob", "fbcheck_with_near_count", "upsample_flow",
           "temporal_loss_l2", "temporal_loss_l1_validity", "temporal_loss_learnable_flow", "generateMask", "temporal_error",
           "temporal_error_u8", "temporal_error_per_pair", "temporal_rmse_per_sample", "warping_error_per_pair",
           "warping_error_per_pair_l1_mask", "warp_blend", "computeTCL_from_flows", "reconet_output_temporal_loss",
           "ruder_network_input", "long_term_blend_step")


@pytest.mark.parametrize("name", ENTRIES)
def test_no_graph_break_and_fullgraph_equals_eager(name):
    fn, args, diff = entries()[name]
    torch._dynamo.reset()
    explain = torch._dynamo.explain(fn)(*args)
    assert explain.graph_break_count == 0, (name, explain.break_reasons)

    def run(f):
        a = [t.clone().requires_grad_(k in diff) for k, t in enumerate(args)]
        out = outputs(f(*a))
        grads = torch.autograd.grad(out[0].sum(), [a[k] for k in diff]) if diff else ()
        return out, grads

    want, want_g = run(fn)
    got, got_g = run(torch.compile(fn, fullgraph=True, backend="aot_eager"))
    for a, b in zip(got, want):
        assert_bits(a.detach(), b.detach())
    for k, a, b in zip(diff, got_g, want_g):
        (assert_scatter_close if diff[k] == "scatter" else assert_bits)(a, b)


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("loss", ["l2", "l1"])
@pytest.mark.parametrize("validity", [False, True])
def test_compiled_training_loss_equals_eager(dtype, loss, validity):
    ff, bf, prev, cur, mask = frames(B=4, H=64, W=96, dtype=dtype)

    def fn(p, c):
        return tcl_b200.temporal_loss(mask, c, p, bf, loss=loss, validity=validity) * 100.0

    def run(f):
        p, c = prev.clone().requires_grad_(), cur.clone().requires_grad_()
        v = f(p, c)
        return (v,) + torch.autograd.grad(v, (p, c))

    (v0, gp0, gc0), (v1, gp1, gc1) = run(fn), run(torch.compile(fn, fullgraph=True, backend="aot_eager"))
    assert_bits(v1, v0)
    assert_bits(gc1, gc0)
    assert_scatter_close(gp1, gp0)


def test_make_fx_of_a_training_loss_through_autograd_grad():
    ff, bf, prev, cur, mask = frames()

    def fn(p, c, f, m):
        loss = tcl_b200.temporal_loss(m, c, tcl_b200.warp(p, f), f) * 100.0
        return torch.autograd.grad(loss, (p, c))

    for mode in ("fake", "symbolic"):
        gm = make_fx(fn, tracing_mode=mode)(prev.clone().requires_grad_(), cur.clone().requires_grad_(), bf, mask)
        targets = {str(n.target) for n in gm.graph.nodes if n.op == "call_function"}
        assert {"tcl_b200.warp.default", "tcl_b200.temporal_loss.default", "tcl_b200.temporal_loss_backward.default",
                "tcl_b200.warp_backward.default"} <= targets, targets


def test_dynamic_shapes_compile_once():
    cnt = CompileCounterWithBackend("aot_eager")

    def fn(ff, bf, prev, cur):
        return tcl_b200.temporal_error_per_pair(ff, bf, prev, cur), tcl_b200.warp(prev, bf)

    torch._dynamo.reset()
    compiled = torch.compile(fn, backend=cnt, dynamic=True, fullgraph=True)
    for H, W in ((24, 40), (36, 56)):
        ff, bf, prev, cur, mask = frames(H=H, W=W)
        for a, b in zip(compiled(ff, bf, prev, cur), fn(ff, bf, prev, cur)):
            assert_bits(a, b)
    assert cnt.frame_count == 1


# ------------------------------------------------------------------------------------------------
# reduce-overhead training step (inductor, CUDA graphs)
# ------------------------------------------------------------------------------------------------
class StandIn(torch.nn.Module):
    """Two-layer conv stand-in for a generator."""

    def __init__(self):
        super().__init__()
        self.c1 = torch.nn.Conv2d(3, 8, 3, padding=1)
        self.c2 = torch.nn.Conv2d(8, 3, 3, padding=1)

    def forward(self, x):
        return torch.sigmoid(self.c2(torch.relu(self.c1(x))))


def tcl_step_loss(G, x_prev, x_cur, flow, mask):
    # StarGANv2AdvCon (core/solver.py:444-446): loss_tcl = ((mask * (fake2 - warp(fake1, flow)))**2).mean(); loss += loss_tcl * 100
    return tcl_b200.temporal_loss(mask, G(x_cur), G(x_prev), flow) * 100.0


def test_reduce_overhead_training_step_equals_eager():
    torch.manual_seed(0)
    G_eager = StandIn().to(DEV)
    G_comp = StandIn().to(DEV)
    G_comp.load_state_dict(G_eager.state_dict())
    opt_e = torch.optim.SGD(G_eager.parameters(), lr=0.05)
    opt_c = torch.optim.SGD(G_comp.parameters(), lr=0.05)
    torch._dynamo.reset()
    torch._dynamo.utils.counters.clear()
    step = torch.compile(tcl_step_loss, mode="reduce-overhead", fullgraph=True)
    for b in range(3):
        ff, bf, xp, xc, mask = frames(B=16, H=256, W=256, seed=100 + b, shift=12.0)
        opt_e.zero_grad(set_to_none=True)
        le = tcl_step_loss(G_eager, xp, xc, bf, mask)
        le.backward()
        opt_e.step()
        opt_c.zero_grad(set_to_none=True)
        if b == 0:
            lc = step(G_comp, xp, xc, bf, mask)
        else:
            with torch._dynamo.config.patch(error_on_recompile=True):
                lc = step(G_comp, xp, xc, bf, mask)
        lc.backward()
        opt_c.step()
        torch.testing.assert_close(lc.detach().clone(), le.detach(), rtol=1e-5, atol=0)
        for pc, pe in zip(G_comp.parameters(), G_eager.parameters()):
            torch.testing.assert_close(pc, pe, rtol=1e-5, atol=1e-6)
    assert torch._dynamo.utils.counters["inductor"]["cudagraph_skips"] == 0
    mgr = torch._inductor.cudagraph_trees.get_manager(DEV.index, create_if_none_exists=False)
    assert mgr is not None and sum(len(v) for v in mgr.roots.values()) > 0
