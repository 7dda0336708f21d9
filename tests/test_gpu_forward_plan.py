"""GPU suite: every forward kernel instantiation in the launch table of csrc/tcl_kernels.cu is reachable and correct.

Each case is the smallest call that selects one row: torch.profiler shows exactly that instantiation launched (with the
fold kernel when the call reduces).  The same call under tclb200_debug_force_generic(1) runs the generic exact kernel:
per-pixel outputs (warp, mask, blend, near-threshold count) are bit-equal, per-pair sums agree to the tolerance of
test_hot_path_equals_generic_kernel_on_a_large_sample (the tile shapes, and so the fixed summation trees, differ)."""
import ctypes
import re

import pytest
import torch

pytestmark = pytest.mark.gpu

OCC, MOB, VALIDITY = 1, 2, 4
L2, L1 = 0, 1
GEN, L2V, L1V, MOBV, OUTV = 0, 1, 2, 3, 4      # kVarGeneral, kVarL2, kVarL1, kVarMobOnly, kVarOutputs
F32, BF16 = "float", "__nv_bfloat16"
COMPUTED, GIVEN, NONE = 2, 1, 0                # MASK_COMPUTED, MASK_GIVEN, MASK_NONE


def _case(kernel, dtype=F32, mask=COMPUTED, frames=True, cur=True, sums=True, C=3, B=2, H=64, W=64, flags=OCC | MOB,
          loss=L2, warp=False, mask_out=False, blend=False, near=False):
    return dict(kernel=kernel, dtype=dtype, mask=mask, frames=frames, cur=cur, sums=sums, C=C, B=B, H=H, W=W, flags=flags,
                loss=loss, warp=warp, mask_out=mask_out, blend=blend, near=near)


BIG = dict(B=1, H=384, W=384)            # >= 384^2 px: the 8-warp rows
NODIRECT = dict(B=33, H=256, W=256)      # > 2 Mpx: the dataset-mask reductions leave the direct kernel
ALL_OUT = dict(warp=True, mask_out=True, blend=True)

CASES = {}
for T in (F32, BF16):
    t = "f32" if T == F32 else "bf16"
    # TMA kernel, computed mask
    CASES[f"tma-{t}-computed-l2"] = _case(("ws", T, COMPUTED, True, 3, L2V, 16), T)
    CASES[f"tma-{t}-computed-l1"] = _case(("ws", T, COMPUTED, True, 3, L1V, 16), T, loss=L1)
    CASES[f"tma-{t}-computed-outputs"] = _case(("ws", T, COMPUTED, True, 3, OUTV, 16), T, **ALL_OUT)
    CASES[f"tma-{t}-computed-general"] = _case(("ws", T, COMPUTED, True, 3, GEN, 16), T, near=True, **ALL_OUT)
    CASES[f"tma-{t}-computed-outputs-nosums"] = _case(("ws", T, COMPUTED, False, 3, OUTV, 16), T, sums=False, **ALL_OUT)
    CASES[f"tma-{t}-computed-general-nosums"] = _case(("ws", T, COMPUTED, False, 3, GEN, 16), T, sums=False, near=True, **ALL_OUT)
    CASES[f"tma-{t}-computed-maskonly-general"] = _case(("ws", T, COMPUTED, False, 0, GEN, 16), T, frames=False, cur=False,
                                                        sums=False, mask_out=True, flags=OCC)
    # TMA kernel, dataset mask
    CASES[f"tma-{t}-given-l2"] = _case(("ws", T, GIVEN, True, 3, L2V, 16), T, GIVEN, **NODIRECT)
    CASES[f"tma-{t}-given-l1"] = _case(("ws", T, GIVEN, True, 3, L1V, 16), T, GIVEN, loss=L1, **NODIRECT)
    CASES[f"tma-{t}-given-outputs"] = _case(("ws", T, GIVEN, True, 3, OUTV, 16), T, GIVEN, warp=True, blend=True)
    CASES[f"tma-{t}-given-general"] = _case(("ws", T, GIVEN, True, 3, GEN, 16), T, GIVEN, flags=VALIDITY, warp=True)
    CASES[f"tma-{t}-given-outputs-nosums"] = _case(("ws", T, GIVEN, False, 3, OUTV, 16), T, GIVEN, sums=False, warp=True, blend=True)
    CASES[f"tma-{t}-given-general-nosums"] = _case(("ws", T, GIVEN, False, 3, GEN, 16), T, GIVEN, sums=False, warp=True, mask_out=True)
    CASES[f"tma-{t}-given-maskonly"] = _case(("ws", T, GIVEN, False, 0, GEN, 16), T, GIVEN, frames=False, cur=False, sums=False,
                                             mask_out=True)
    # TMA kernel, no mask
    CASES[f"tma-{t}-none"] = _case(("ws", T, NONE, True, 3, GEN, 16), T, NONE)
    CASES[f"tma-{t}-none-nosums"] = _case(("ws", T, NONE, False, 3, GEN, 16), T, NONE, sums=False, warp=True, blend=True)
    CASES[f"tma-{t}-none-warponly"] = _case(("ws", T, NONE, False, 3, L2V, 16), T, NONE, cur=False, sums=False, warp=True)
    CASES[f"tma-{t}-none-maskonly"] = _case(("ws", T, NONE, False, 0, GEN, 16), T, NONE, frames=False, cur=False, sums=False,
                                            mask_out=True)
    # direct kernel
    CASES[f"direct-{t}-l2"] = _case(("direct", T, L2), T, GIVEN)
    CASES[f"direct-{t}-l1"] = _case(("direct", T, L1), T, GIVEN, loss=L1)
    # generic kernel: W % 4 != 0; CT == 0 is any C but 3
    for M, m in ((COMPUTED, "computed"), (GIVEN, "given"), (NONE, "none")):
        for R in (True, False):
            for C in (3, 1):
                CASES[f"generic-{t}-{m}-{'sums' if R else 'nosums'}-c{C}"] = _case(("generic", T, M, R, 3 if C == 3 else 0), T, M,
                                                                                  sums=R, C=C, W=62, warp=True)
# fp32 only: the 8-warp rows, and fbcCheckTorch on its own (an fp32 kernel whatever the dtype)
CASES["tma-f32-computed-l2-w8"] = _case(("ws", F32, COMPUTED, True, 3, L2V, 8), **BIG)
CASES["tma-f32-computed-l1-w8"] = _case(("ws", F32, COMPUTED, True, 3, L1V, 8), loss=L1, **BIG)
CASES["tma-f32-computed-maskonly-w8"] = _case(("ws", F32, COMPUTED, False, 0, L2V, 8), frames=False, cur=False, sums=False,
                                              mask_out=True, **BIG)
CASES["tma-f32-computed-maskonly"] = _case(("ws", F32, COMPUTED, False, 0, L2V, 16), frames=False, cur=False, sums=False, mask_out=True)
CASES["tma-bf16dtype-computed-maskonly"] = _case(("ws", F32, COMPUTED, False, 0, L2V, 16), BF16, frames=False, cur=False,
                                                 sums=False, mask_out=True)
CASES["tma-f32-computed-mobonly"] = _case(("ws", F32, COMPUTED, False, 0, MOBV, 16), frames=False, cur=False, sums=False,
                                          mask_out=True, flags=MOB)


def _parse(name):
    """(path, template arguments...) of a forward kernel's demangled name, None for any other kernel."""
    def targs(s):
        return [a.strip() for a in s.split(",")]
    m = re.search(r"fused_forward_ws_kernel<(.*?), tcl::WsCfg<([^>]*)>", name)
    if m:
        T, M, R, CT, V = targs(m.group(1))
        return ("ws", T, int(M), R == "true", int(CT), int(V), int(targs(m.group(2))[8]))
    m = re.search(r"fused_forward_direct_kernel<([^>]*)>", name)
    if m:
        T, loss = targs(m.group(1))
        return ("direct", T, int(loss))
    m = re.search(r"fused_forward_generic_kernel<([^>]*)>", name)
    if m:
        T, M, R, CT = targs(m.group(1))
        return ("generic", T, int(M), R == "true", int(CT))
    if re.search(r"fold_partials(_small)?_kernel", name):
        return ("fold",)
    return None


def _inputs(tcl, c):
    d = torch.device("cuda:0")
    dtype = torch.float32 if c["dtype"] == F32 else torch.bfloat16
    B, C, H, W = c["B"], c["C"], c["H"], c["W"]
    ff, bf = tcl.synth.make_flows(B, H, W, seed=31 + H + W, max_shift=12.0, max_rot_deg=3.0, n_rects=3, rect_shift=8.0, device=d)
    prev, cur = tcl.synth.make_frames(B, C, H, W, seed=31 + H + W, kind="white", device=d, dtype=dtype)
    mask = torch.rand(B, 1, H, W, device=d, generator=torch.Generator(device=d).manual_seed(5))
    return dict(ff=ff if c["mask"] == COMPUTED else None, bf=bf, mask=mask if c["mask"] == GIVEN else None,
                prev=prev if c["frames"] else None, cur=cur if c["cur"] else None, dtype=dtype)


def _forward(tcl, c, x):
    """One tclb200_tcl_forward call with fresh outputs; returns them."""
    B, C, H, W = c["B"], c["C"], c["H"], c["W"]
    d = x["bf"].device
    out = {}
    if c["sums"]:
        out["pair_sums"] = torch.empty(B, dtype=torch.float64, device=d)
        out["total_sums"] = torch.empty(2, dtype=torch.float64, device=d)
    if c["warp"]:
        out["warp"] = torch.full((B, C, H, W), float("nan"), dtype=x["dtype"], device=d)
    if c["blend"]:
        out["blend"] = torch.full((B, C, H, W), float("nan"), dtype=x["dtype"], device=d)
    if c["mask_out"]:
        out["mask"] = torch.full((B, 1, H, W), float("nan"), device=d)
    if c["near"]:
        out["near"] = torch.zeros(1, dtype=torch.int64, device=d)
    scratch = torch.zeros(tcl._cabi.lib().tclb200_scratch_bytes(B, H, W), dtype=torch.uint8, device=d) if c["sums"] else None
    p = tcl.ops._ptr
    a = tcl._cabi.TclArgs()
    a.ff, a.bf, a.mask_in, a.prev, a.cur = p(x["ff"]), p(x["bf"]), p(x["mask"]), p(x["prev"]), p(x["cur"])
    a.warp_out, a.mask_out, a.blend_out = p(out.get("warp")), p(out.get("mask")), p(out.get("blend"))
    a.pair_sums, a.total_sums, a.near_threshold = p(out.get("pair_sums")), p(out.get("total_sums")), p(out.get("near"))
    if scratch is not None:
        a.scratch, a.scratch_bytes = p(scratch), scratch.numel()
    a.B, a.C, a.H, a.W = B, C, H, W
    a.dtype = tcl._cabi.BF16 if x["dtype"] == torch.bfloat16 else tcl._cabi.F32
    a.flags, a.loss, a.finalize = c["flags"], c["loss"], tcl._cabi.FIN_MEAN
    tcl._cabi.check(tcl._cabi.lib().tclb200_tcl_forward(ctypes.byref(a), tcl.ops._stream_handle()))
    torch.cuda.synchronize()
    return out


@pytest.mark.parametrize("name", sorted(CASES))
def test_every_row_of_the_launch_table_is_selected_and_agrees_with_the_generic_kernel(tcl, name):
    c = CASES[name]
    x = _inputs(tcl, c)
    _forward(tcl, c, x)                   # warm-up: module load, shared-memory attribute
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        got = _forward(tcl, c, x)
    launched = [k for k in (_parse(e.name) for e in prof.events()) if k is not None]
    want = [c["kernel"]] + ([("fold",)] if c["sums"] and c["kernel"][0] != "generic" else [])
    assert launched == want, (launched, want)
    if c["kernel"][0] == "generic":
        return                            # (the generic kernel is the reference)
    lib = tcl._cabi.lib()
    lib.tclb200_debug_force_generic(1)
    try:
        ref = _forward(tcl, c, x)
    finally:
        lib.tclb200_debug_force_generic(0)
    rtol = 1e-6 if c["dtype"] == F32 else 1e-5
    for key, v in got.items():
        if key in ("pair_sums", "total_sums"):
            assert bool(torch.isfinite(v).all()), key
            assert torch.allclose(v, ref[key], rtol=rtol, atol=0.0), (key, v, ref[key])
        else:
            assert not bool(v.float().isnan().any()), key
            assert torch.equal(v, ref[key]), key
