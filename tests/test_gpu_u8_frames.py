"""GPU suite of uint8 frames: stored 8-bit video scored with a per-channel normalisation v = u * scale[c] + offset[c].

The contract: given the normalised frames (torch's u.float().mul(scale).add(offset)), the result is the fp32 path's -- masks
bit-identical, per-pair sums bit-identical when both calls run the generic kernel, within rtol 1e-6 otherwise (other tile
shapes, other summation trees).  grid_sample's zero padding applies to the normalised frame."""
import re

import pytest
import torch

from oracle import torch_port as tp

pytestmark = pytest.mark.gpu

NORMS = {"unit": (1 / 255, 0.0), "gan": (2 / 255, -1.0), "mean": (1.0, (-123.675, -116.28, -103.53))}
SHAPES = {"sintel": (2, 436, 1024), "crops": (4, 256, 256), "ragged": (3, 37, 53)}


def _dev():
    return torch.device("cuda:0")


def _norm_tensors(norm, d):
    s, o = norm
    s = torch.tensor([s] * 3 if not isinstance(s, tuple) else list(s), dtype=torch.float32, device=d).view(1, 3, 1, 1)
    o = torch.tensor([o] * 3 if not isinstance(o, tuple) else list(o), dtype=torch.float32, device=d).view(1, 3, 1, 1)
    return s, o


def _normalise(u, norm):
    s, o = _norm_tensors(norm, u.device)
    return u.float().mul(s).add(o)


def _u8_frames(B, H, W, seed, d):
    g = torch.Generator(device=d).manual_seed(seed)
    # smooth content plus noise, like decoded video: neighbouring pixels are correlated, every value 0..255 occurs
    base = torch.nn.functional.interpolate(torch.rand(B + 1, 3, H // 8 + 2, W // 8 + 2, device=d, generator=g) * 255,
                                           size=(H, W), mode="bilinear", align_corners=False)
    noise = torch.randint(-12, 13, (B + 1, 3, H, W), device=d, generator=g).float()
    u = (base + noise).round().clamp(0, 255).to(torch.uint8)
    return u[:B].contiguous(), u[1:].contiguous()


def _flows(tcl, B, H, W, seed, d):
    return tcl.synth.make_flows(B, H, W, seed=seed, max_shift=12.0, max_rot_deg=3.0, n_rects=3, rect_shift=8.0, device=d)


@pytest.fixture
def force_generic(tcl):
    lib = tcl._cabi.lib()
    yield lib.tclb200_debug_force_generic
    lib.tclb200_debug_force_generic(0)


def _pair(tcl, bf, prev, cur, mask_kind, ff, mask, loss, **kw):
    return tcl.fused_forward(bf, prev, cur, ff=ff if mask_kind == "computed" else None, mask=mask if mask_kind == "given" else None,
                             loss=loss, want_mask=mask_kind == "computed", **kw)


# ------------------------------------------------------------------ launch table
def _parse(name):
    m = re.search(r"fused_forward_generic_u8_kernel<(\d+)>", name)
    if m:
        return ("generic_u8", int(m.group(1)))
    m = re.search(r"fused_forward_ws_u8_kernel<(\d+), (true|false), (\d+), (\d+), tcl::WsCfg<([^>]*)>", name)
    if m:
        return ("ws_u8", int(m.group(1)), m.group(2) == "true", int(m.group(3)), int(m.group(4)),
                int([a.strip() for a in m.group(5).split(",")][8]))
    m = re.search(r"fused_forward_(ws|generic)_kernel<([^,>]*), (\d+), (true|false), (\d+)", name)
    if m:
        return (m.group(1), m.group(2), int(m.group(3)), m.group(4) == "true", int(m.group(5)))
    if re.search(r"fold_partials(_small)?_kernel", name):
        return ("fold",)
    return None


GEN, L2V, L1V, OUTV = 0, 1, 2, 4      # kVarGeneral, kVarL2, kVarL1, kVarOutputs
U8_ROWS = {   # the smallest call that selects each uint8 row: (kernel, mask kind, fused_forward keywords, W)
    "tma-computed-l2": (("ws_u8", 2, True, 3, L2V, 16), "computed", {}, 64),
    "tma-computed-l1": (("ws_u8", 2, True, 3, L1V, 16), "computed", {"loss": 1}, 64),
    "tma-computed-outputs": (("ws_u8", 2, True, 3, OUTV, 16), "computed", {"want_mask": True}, 64),
    "tma-computed-general": (("ws_u8", 2, True, 3, GEN, 16), "computed", {"want_mask": True, "want_near": True}, 64),
    "tma-given-l2": (("ws_u8", 1, True, 3, L2V, 16), "given", {}, 64),
    "tma-given-l1": (("ws_u8", 1, True, 3, L1V, 16), "given", {"loss": 1}, 64),
    "tma-given-general": (("ws_u8", 1, True, 3, GEN, 16), "given", {"want_mask": True}, 64),
    "tma-none-general": (("ws_u8", 0, True, 3, GEN, 16), "none", {}, 64),
    # W % 16 != 0: no uint8 tensor map (box rows are multiples of 16 bytes) -- the generic kernel
    "generic-computed": (("generic_u8", 2), "computed", {"want_mask": True}, 40),
    "generic-given": (("generic_u8", 1), "given", {}, 40),
    "generic-none": (("generic_u8", 0), "none", {}, 40),
}


@pytest.mark.parametrize("name", sorted(U8_ROWS))
def test_every_u8_row_is_selected_and_agrees_with_the_generic_kernel(tcl, force_generic, name):
    kernel, mask_kind, kw, W = U8_ROWS[name]
    d = _dev()
    B, H = 2, 64
    ff, bf = _flows(tcl, B, H, W, 31, d)
    prev, cur = _u8_frames(B, H, W, 31, d)
    mask = torch.rand(B, 1, H, W, device=d, generator=torch.Generator(device=d).manual_seed(5))
    norm = NORMS["gan"]

    def run(p, c, **extra):
        return tcl.fused_forward(bf, p, c, ff=ff if mask_kind == "computed" else None, mask=mask if mask_kind == "given" else None,
                                 **kw, **extra)
    run(prev, cur, u8_scale=norm[0], u8_offset=norm[1])
    torch.cuda.synchronize()
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        got = run(prev, cur, u8_scale=norm[0], u8_offset=norm[1])
        torch.cuda.synchronize()
    launched = [k for k in (_parse(e.name) for e in prof.events()) if k is not None]
    want = [kernel] + ([("fold",)] if kernel[0] == "ws_u8" else [])      # (the generic kernel folds its own partials)
    assert launched == want, (launched, want)
    force_generic(1)
    ref = run(prev, cur, u8_scale=norm[0], u8_offset=norm[1])            # the uint8 generic kernel
    f32 = run(_normalise(prev, norm), _normalise(cur, norm))             # the fp32 generic kernel on the normalised frames
    torch.cuda.synchronize()
    assert torch.equal(ref.pair_sums, f32.pair_sums) and torch.equal(ref.total_sums, f32.total_sums)
    assert bool(torch.isfinite(got.pair_sums).all())
    assert torch.allclose(got.pair_sums, ref.pair_sums, rtol=1e-6, atol=0.0), (got.pair_sums, ref.pair_sums)
    for key in ("mask", "near_threshold"):
        if getattr(got, key) is not None:
            assert torch.equal(getattr(got, key), getattr(ref, key)) and torch.equal(getattr(ref, key), getattr(f32, key)), key


def test_mask_only_calls_with_u8_dtype_take_the_fp32_mask_kernel(tcl):
    import ctypes
    d = _dev()
    B, H, W = 2, 64, 64
    ff, bf = _flows(tcl, B, H, W, 7, d)
    out = torch.full((B, 1, H, W), float("nan"), device=d)
    a = tcl._cabi.TclArgs()
    a.ff, a.bf, a.mask_out = ff.data_ptr(), bf.data_ptr(), out.data_ptr()
    a.B, a.H, a.W, a.dtype, a.flags = B, H, W, tcl._cabi.U8, tcl._cabi.OCC | tcl._cabi.MOB
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        tcl._cabi.check(tcl._cabi.lib().tclb200_tcl_forward(ctypes.byref(a), tcl.ops._stream_handle()))
        torch.cuda.synchronize()
    launched = [k for k in (_parse(e.name) for e in prof.events()) if k is not None]
    assert launched == [("ws", "float", 2, False, 0)], launched
    assert torch.equal(out, tcl.fbcCheckTorch(ff, bf))


# ------------------------------------------------------------------ against the fp32 path on the normalised frames
@pytest.mark.parametrize("shape", sorted(SHAPES))
@pytest.mark.parametrize("mask_kind", ["computed", "given", "none"])
@pytest.mark.parametrize("loss", ["l2", "l1"])
@pytest.mark.parametrize("norm", sorted(NORMS))
def test_u8_equals_fp32_on_normalised_frames(tcl, force_generic, shape, mask_kind, loss, norm):
    d = _dev()
    B, H, W = SHAPES[shape]
    ff, bf = _flows(tcl, B, H, W, 11 + H, d)
    prev, cur = _u8_frames(B, H, W, 11 + W, d)
    mask = torch.rand(B, 1, H, W, device=d, generator=torch.Generator(device=d).manual_seed(3))
    L = tcl._cabi.L2 if loss == "l2" else tcl._cabi.L1
    s, o = NORMS[norm]
    pf, cf = _normalise(prev, NORMS[norm]), _normalise(cur, NORMS[norm])
    got = _pair(tcl, bf, prev, cur, mask_kind, ff, mask, L, u8_scale=s, u8_offset=o)   # uint8: the TMA kernel where the shape allows
    fast = _pair(tcl, bf, pf, cf, mask_kind, ff, mask, L)                             # fp32: likewise
    force_generic(1)
    got_exact = _pair(tcl, bf, prev, cur, mask_kind, ff, mask, L, u8_scale=s, u8_offset=o)
    exact = _pair(tcl, bf, pf, cf, mask_kind, ff, mask, L)
    torch.cuda.synchronize()
    assert bool(torch.isfinite(got.pair_sums).all())
    assert torch.equal(got_exact.pair_sums, exact.pair_sums) and torch.equal(got_exact.pair_vals, exact.pair_vals)
    assert torch.allclose(got.pair_sums, exact.pair_sums, rtol=1e-6, atol=0.0), (got.pair_sums, exact.pair_sums)
    assert torch.allclose(got.pair_sums, fast.pair_sums, rtol=1e-6, atol=0.0), (got.pair_sums, fast.pair_sums)
    if mask_kind == "computed":
        assert torch.equal(got.mask, exact.mask) and torch.equal(got.mask, fast.mask) and torch.equal(got_exact.mask, exact.mask)


def test_default_normalisation_is_the_fp32_reciprocal_product(tcl):
    """The default scale is fp32(1/255): u8 frames with no arguments equal torch's u.float().mul(fp32(1/255))."""
    d = _dev()
    B, H, W = 2, 96, 128
    ff, bf = _flows(tcl, B, H, W, 2, d)
    prev, cur = _u8_frames(B, H, W, 2, d)
    scale = torch.tensor(1 / 255, dtype=torch.float32, device=d)
    lib = tcl._cabi.lib()
    lib.tclb200_debug_force_generic(1)    # (both on the generic kernel: the same summation tree)
    try:
        got = tcl.temporal_error_per_pair(ff, bf, prev, cur)
        ref = tcl.temporal_error_per_pair(ff, bf, prev.float().mul(scale), cur.float().mul(scale))
    finally:
        lib.tclb200_debug_force_generic(0)
    assert torch.equal(got, ref)


# ------------------------------------------------------------------ zero padding of the normalised frame
def _extreme_flows(d):
    B, H, W = 1, 24, 32
    bf = torch.zeros(B, 2, H, W)
    bf[:, 0, :8] = 1e6; bf[:, 1, 8:16] = -1e6; bf[:, 0, 16:20] = 3e9; bf[:, 1, 20:] = -40.25
    bf[:, 0, 20:, ::2] = 31.5
    return -bf.to(d), bf.to(d)


@pytest.mark.parametrize("flows", ["extreme", "nonfinite", "edge", "shifted"])
@pytest.mark.parametrize("mask_kind", ["computed", "none"])
def test_taps_outside_the_image_contribute_zero_not_the_offset(tcl, force_generic, flows, mask_kind):
    d = _dev()
    if flows == "extreme":
        ff, bf = _extreme_flows(d)
    elif flows == "shifted":   # several tiles, real flow plus a shift: the boxes of every border tile cross the image border
        ff, bf = _flows(tcl, 2, 128, 256, 12, d)
        bf[:, 0] += 5.5; bf[:, 1] -= 3.25; ff[:, 0] -= 5.5; ff[:, 1] += 3.25
    else:
        ff, bf = tcl.synth.make_flows(1, 32, 64, seed=8, max_shift=4.0, device=d)
        if flows == "nonfinite":
            bf[0, 0, 5, 7] = float("inf"); bf[0, 1, 9, 40] = float("-inf"); bf[0, 0, 20, 20] = float("nan")
        else:   # a uniform shift by 2.5 px: every pixel of a 3-px border band has taps outside
            bf[:, 0] = 2.5; bf[:, 1] = -2.5; ff = -bf
    B, _, H, W = bf.shape
    prev, cur = _u8_frames(B, H, W, 4, d)
    norm = NORMS["gan"]                                              # offset -1: an offset read outside would show
    pf, cf = _normalise(prev, norm), _normalise(cur, norm)
    got = _pair(tcl, bf, prev, cur, mask_kind, ff, None, tcl._cabi.L2, u8_scale=norm[0], u8_offset=norm[1])   # staged (TMA) path
    fast = _pair(tcl, bf, pf, cf, mask_kind, ff, None, tcl._cabi.L2)
    force_generic(1)
    got_exact = _pair(tcl, bf, prev, cur, mask_kind, ff, None, tcl._cabi.L2, u8_scale=norm[0], u8_offset=norm[1])
    exact = _pair(tcl, bf, pf, cf, mask_kind, ff, None, tcl._cabi.L2)
    torch.cuda.synchronize()
    assert torch.equal(torch.isnan(got_exact.pair_sums), torch.isnan(exact.pair_sums))
    assert torch.equal(torch.nan_to_num(got_exact.pair_sums), torch.nan_to_num(exact.pair_sums))
    assert torch.equal(torch.isnan(got.pair_sums), torch.isnan(fast.pair_sums))
    assert torch.allclose(torch.nan_to_num(got.pair_sums), torch.nan_to_num(fast.pair_sums), rtol=1e-6, atol=0.0), (got.pair_sums, fast.pair_sums)
    assert torch.allclose(torch.nan_to_num(got.pair_sums), torch.nan_to_num(exact.pair_sums), rtol=1e-6, atol=0.0)
    if mask_kind == "computed":
        assert torch.equal(got.mask, exact.mask)
    if flows != "nonfinite":
        # the reference's own expression on the normalised frames: taps outside are zeros of the fp32 frame
        w = tp.backward_warp(pf, bf)
        m = tp.fb_consistency(ff, bf) if mask_kind == "computed" else torch.ones_like(w[:, :1])
        want = ((m.double() * (cf.double() - w.double())) ** 2).sum(dim=(1, 2, 3))
        assert torch.allclose(got.pair_sums, want, rtol=1e-5, atol=0.0), (got.pair_sums, want)
    if flows != "nonfinite" and mask_kind == "none":
        # and the offset read in place of the zero padding would have changed the sums (with a computed mask the pixels whose
        # taps leave the image are occluded anyway)
        w = tp.backward_warp(pf, bf)
        want = ((cf.double() - w.double()) ** 2).sum(dim=(1, 2, 3))
        wrong = tp.backward_warp(pf - norm[1], bf) + norm[1]
        bad = ((cf.double() - wrong.double()) ** 2).sum(dim=(1, 2, 3))
        assert not torch.allclose(want, bad, rtol=1e-5, atol=0.0)


# ------------------------------------------------------------------ the reference
@pytest.mark.parametrize("norm", sorted(NORMS))
def test_reference_on_normalised_frames(tcl, norm):
    d = _dev()
    B, H, W = 2, 96, 160
    ff, bf = tcl.synth.make_flows(B, H, W, seed=1234, max_shift=8.0, device=d)
    prev, cur = _u8_frames(B, H, W, 1234, d)
    s, o = NORMS[norm]
    got = tcl.temporal_error(ff, bf, prev, cur, u8_scale=s, u8_offset=o)
    want = tp.temporal_error(ff, bf, _normalise(prev, NORMS[norm]), _normalise(cur, NORMS[norm]))
    assert abs(float(got) - float(want)) <= 1e-5 * abs(float(want)), (float(got), float(want))


# ------------------------------------------------------------------ clip, window and band modes
def test_clip_mode_with_a_u8_bank_equals_independent_pairs(tcl):
    d = _dev()
    T, H, W = 6, 96, 128
    ff, bf = _flows(tcl, T - 1, H, W, 21, d)
    frames = torch.cat(_u8_frames(T - 1, H, W, 21, d)[:1] + (_u8_frames(T - 1, H, W, 21, d)[1][-1:],)).contiguous()
    norm = NORMS["mean"]
    got = tcl.temporal_error_clip(frames, ff, bf, u8_scale=norm[0], u8_offset=norm[1])
    want = tcl.temporal_error_per_pair(ff, bf, frames[:-1], frames[1:], u8_scale=norm[0], u8_offset=norm[1])
    assert torch.equal(got, want)


def test_window_mode_with_a_u8_bank_equals_independent_pairs(tcl):
    d = _dev()
    T, H, W = 6, 64, 96
    idx = tcl.ops.window_evaluations(T, 4)
    J = idx["field_t"].numel()
    g = torch.Generator(device=d).manual_seed(9)
    bank = (torch.randn(2 * J, 2, H, W, device=d, generator=g) * 3).contiguous()
    frames = torch.randint(0, 256, (T, 3, H, W), device=d, generator=g, dtype=torch.uint8)
    norm = NORMS["gan"]
    got = tcl.temporal_error_window(frames, bank, 4, idx, u8_scale=norm[0], u8_offset=norm[1])
    at = lambda k: idx[k].to(d).long()
    want = tcl.temporal_error_per_pair(bank[at("ff_index")], bank[at("bf_index")], frames[at("prev_index")], frames[at("cur_index")],
                                       u8_scale=norm[0], u8_offset=norm[1])
    assert torch.equal(got, want)


def test_band_mode_sums_add_up_to_the_whole_frame(tcl):
    d = _dev()
    B, H, W = 2, 200, 96
    ff, bf = _flows(tcl, B, H, W, 13, d)
    prev, cur = _u8_frames(B, H, W, 13, d)
    whole = tcl.fused_forward(bf, prev, cur, ff=ff).pair_sums
    parts = sum(tcl.sharding.evaluate_banded(ff, bf, prev, cur, rank=r, world=3)["pair_sums"] for r in range(3))
    assert torch.allclose(parts, whole, rtol=1e-12, atol=0.0), (parts, whole)


def test_sharded_evaluation_takes_u8_frames(tcl):
    d = _dev()
    B, H, W = 3, 64, 64
    ff, bf = _flows(tcl, B, H, W, 17, d)
    prev, cur = _u8_frames(B, H, W, 17, d)
    seq = torch.tensor([0, 0, 1], device=d)
    got = tcl.sharding.evaluate_sharded(ff, bf, prev, cur, seq, 2, u8_scale=1.0, u8_offset=-128.0)
    vals = tcl.temporal_error_per_pair(ff, bf, prev, cur, u8_scale=1.0, u8_offset=-128.0).double()
    assert torch.allclose(got["per_sequence_mean"], torch.stack([vals[:2].mean(), vals[2:].mean()]), rtol=1e-12, atol=0.0)


# ------------------------------------------------------------------ host-buffer entry
@pytest.mark.parametrize("ring", [False, True])
def test_host_entry_with_u8_clips_equals_the_device_clip_path(tcl, ring):
    d = _dev()
    T, H, W = 16, 96, 128
    ff, bf = _flows(tcl, T - 1, H, W, 41, d)
    frames = torch.randint(0, 256, (T, 3, H, W), device=d, dtype=torch.uint8, generator=torch.Generator(device=d).manual_seed(41))
    norm = NORMS["mean"]
    want = tcl.temporal_error_clip(frames, ff, bf, u8_scale=norm[0], u8_offset=norm[1]).cpu()
    kw = dict(chunk_pairs=2, max_device_frames=10) if ring else {}
    got = tcl.temporal_error_host(frames.cpu().pin_memory(), ff.cpu().pin_memory(), bf.cpu().pin_memory(), u8_scale=norm[0],
                                  u8_offset=norm[1], **kw)
    assert torch.equal(got, want)
    got2 = tcl.sharding.evaluate_sharded_host(frames.cpu(), ff.cpu(), bf.cpu(), torch.arange(T - 1, dtype=torch.int32),
                                              torch.arange(1, T, dtype=torch.int32), torch.zeros(T - 1, dtype=torch.long), 1,
                                              u8_scale=norm[0], u8_offset=norm[1])
    assert torch.allclose(got2["mean_over_pairs"].cpu(), want.double().mean(), rtol=1e-12, atol=0.0)


# ------------------------------------------------------------------ refusals
def test_python_refusals(tcl):
    d = _dev()
    B, H, W = 1, 32, 64
    ff, bf = _flows(tcl, B, H, W, 3, d)
    prev, cur = _u8_frames(B, H, W, 3, d)
    err = tcl._cabi.TclB200Error
    with pytest.raises(err, match="warp_out"):
        tcl.fused_forward(bf, prev, cur, ff=ff, want_warp=True)
    with pytest.raises(err, match="blend_out"):
        tcl.fused_forward(bf, prev, cur, ff=ff, want_blend=True)
    with pytest.raises(err, match="reduction"):
        tcl.fused_forward(bf, prev, cur, ff=ff, want_sums=False, want_mask=True)
    with pytest.raises(RuntimeError, match="3 channels"):
        tcl.fused_forward(bf, prev[:, :1], cur[:, :1], ff=ff)
    with pytest.raises(RuntimeError, match="uint8 frames only"):
        tcl.temporal_error(ff, bf, prev.float(), cur.float(), u8_scale=1 / 255)
    with pytest.raises(RuntimeError, match="finite"):
        tcl.temporal_error(ff, bf, prev, cur, u8_offset=float("nan"))
    for fn in (lambda: tcl.warp(prev, bf), lambda: tcl.fs_warp(prev, bf), lambda: tcl.temporal_loss(None, cur, prev, bf),
               lambda: tcl.warp_blend(torch.ones(B, 1, H, W, device=d), prev, bf, cur), lambda: tcl.generateMask(cur, prev, bf),
               lambda: tcl.temporal_error(ff, bf, prev.half(), cur.half())):
        with pytest.raises(RuntimeError, match="float32 or bfloat16"):
            fn()
