"""GPU suite of the kept-pixel sums (ABI v9): pair b's sum of the mask over its evaluated pixels, from the fused evaluation
(`fused_forward(want_kept=True)`, `warping_error_per_pair`) and from the host-buffer entry (`temporal_error_host(return_kept=True)`).

* every kept row of the launch table is selected (torch.profiler, the scheme of test_gpu_forward_plan.py) and agrees with the
  generic kept kernel, and its pair_sums are bit for bit those of the same call without kept sums;
* kept sums equal the mask oracle: fbcCheckTorch's mask summed in fp64 (exact), a binary dataset mask's fp64 sum (exact), a soft
  one's to rtol 1e-6;
* the masked warping error S_b / (C * kept_b) matches the expression built from oracle.torch_port on the same GPU;
* clip, window, band, cropped flow views, bf16 and uint8 frames, and the host entry across chunkings, a frame ring and
  channels-last inputs all give the same kept sums."""
import re

import pytest
import torch

from oracle import torch_port as tp

pytestmark = pytest.mark.gpu

L2, L1 = 0, 1
FIN_MEAN, FIN_RMSE = 0, 1
GEN, L2V, L1V = 0, 1, 2                 # kVarGeneral, kVarL2, kVarL1
COMPUTED, GIVEN = 2, 1                  # MASK_COMPUTED, MASK_GIVEN
F32, BF16, U8 = "float", "__nv_bfloat16", "u8"


def _dev():
    return torch.device("cuda:0")


def _row(kernel, T=F32, mask=COMPUTED, loss=L2, B=2, C=3, H=64, W=64):
    return dict(kernel=kernel, T=T, mask=mask, loss=loss, B=B, C=C, H=H, W=W)


ROWS = {}
for T, t in ((F32, "f32"), (BF16, "bf16"), (U8, "u8")):
    for M, m in ((COMPUTED, "computed"), (GIVEN, "given")):
        ROWS[f"tma-{t}-{m}-l2"] = _row(("ws", T, M, 3, L2V, 16), T, M)
        ROWS[f"tma-{t}-{m}-l1"] = _row(("ws", T, M, 3, L1V, 16), T, M, L1)
        # the generic kernel: a width TMA cannot describe; C != 3 (CT == 0) for the frame types that allow it
        ROWS[f"generic-{t}-{m}-c3"] = _row(("generic", T, M, 3), T, M, W=62)
        if T != U8:
            ROWS[f"generic-{t}-{m}-c1"] = _row(("generic", T, M, 0), T, M, C=1, W=62)
# the 8-warp rows of large fp32 frames with a computed mask
ROWS["tma-f32-computed-l2-w8"] = _row(("ws", F32, COMPUTED, 3, L2V, 8), B=1, H=384, W=384)
ROWS["tma-f32-computed-l1-w8"] = _row(("ws", F32, COMPUTED, 3, L1V, 8), loss=L1, B=1, H=384, W=384)


def _parse(name):
    """(path, template arguments...) of a kept-pixel kernel; ("fold",) for its fold; ("other", name) for any other forward or
    fold kernel (none may run in a kept call); None for everything else."""
    targs = lambda s: [a.strip() for a in s.split(",")]
    m = re.search(r"fused_forward_ws_kept_kernel<(.*?), tcl::WsCfg<([^>]*)>", name)
    if m:
        T, M, CT, V = targs(m.group(1))
        return ("ws", T, int(M), int(CT), int(V), int(targs(m.group(2))[8]))
    m = re.search(r"fused_forward_ws_u8_kept_kernel<(.*?), tcl::WsCfg<([^>]*)>", name)
    if m:
        M, CT, V = targs(m.group(1))
        return ("ws", U8, int(M), int(CT), int(V), int(targs(m.group(2))[8]))
    m = re.search(r"fused_forward_generic_kept_kernel<([^>]*)>", name)
    if m:
        T, M, CT = targs(m.group(1))
        return ("generic", T, int(M), int(CT))
    m = re.search(r"fused_forward_generic_u8_kept_kernel<([^>]*)>", name)
    if m:
        return ("generic", U8, int(m.group(1)), 3)
    if re.search(r"fold_partials(_small)?_kept_kernel", name):
        return ("fold",)
    if re.search(r"fused_forward_|fold_partials|fill_kept", name):
        return ("other", name)
    return None


def _frames(T, B, C, H, W, seed):
    d = _dev()
    if T == U8:
        g = torch.Generator(device=d).manual_seed(seed)
        return (torch.randint(0, 256, (B, C, H, W), device=d, dtype=torch.uint8, generator=g),
                torch.randint(0, 256, (B, C, H, W), device=d, dtype=torch.uint8, generator=g))
    import tcl_b200
    return tcl_b200.synth.make_frames(B, C, H, W, seed=seed, kind="white", device=d,
                                      dtype=torch.float32 if T == F32 else torch.bfloat16)


def _inputs(tcl, c, seed=31):
    d = _dev()
    B, C, H, W = c["B"], c["C"], c["H"], c["W"]
    ff, bf = tcl.synth.make_flows(B, H, W, seed=seed + H + W, max_shift=12.0, max_rot_deg=3.0, n_rects=3, rect_shift=8.0, device=d)
    prev, cur = _frames(c["T"], B, C, H, W, seed)
    mask = torch.rand(B, 1, H, W, device=d, generator=torch.Generator(device=d).manual_seed(seed + 5))   # soft
    return dict(ff=ff if c["mask"] == COMPUTED else None, bf=bf, mask=mask if c["mask"] == GIVEN else None, prev=prev, cur=cur)


def _call(tcl, c, x, kept=True, **kw):
    r = tcl.fused_forward(x["bf"], x["prev"], x["cur"], ff=x["ff"], mask=x["mask"], loss=c["loss"], want_kept=kept, **kw)
    torch.cuda.synchronize()
    return r


def _forced(tcl, mode, fn):
    lib = tcl._cabi.lib()
    lib.tclb200_debug_force_generic(mode)
    try:
        return fn()
    finally:
        lib.tclb200_debug_force_generic(0)


def _mask_of(tcl, x):
    return tcl.fbcCheckTorch(x["ff"], x["bf"]) if x["ff"] is not None else x["mask"]


@pytest.mark.parametrize("name", sorted(ROWS))
def test_every_kept_row_is_selected_and_agrees_with_the_generic_kernel_and_the_oracle(tcl, name):
    c = ROWS[name]
    x = _inputs(tcl, c)
    _call(tcl, c, x)                      # warm-up: module load, shared-memory attribute
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        got = _call(tcl, c, x)
    launched = [k for k in (_parse(e.name) for e in prof.events()) if k is not None]
    want = [c["kernel"]] + ([("fold",)] if c["kernel"][0] == "ws" else [])
    assert launched == want, (launched, want)
    # kept sums: the mask oracle (the computed mask's verdicts are exact integers; a soft mask is summed in another order)
    oracle = _mask_of(tcl, x).double().sum((1, 2, 3))
    if c["mask"] == COMPUTED:
        assert torch.equal(got.pair_kept, oracle), (got.pair_kept, oracle)
        assert float(got.total_kept) == float(oracle.sum())
    else:
        assert torch.allclose(got.pair_kept, oracle, rtol=1e-6, atol=0.0), (got.pair_kept, oracle)
        assert abs(float(got.total_kept) - float(oracle.sum())) <= 1e-6 * float(oracle.sum())
    # pair_sums: bit for bit those of the same call without kept sums (same kernel body, tile geometry and consumer warps;
    # mode 2 keeps dataset-mask calls off the direct kernel, which reduces in another order)
    plain = _forced(tcl, 2, lambda: _call(tcl, c, x, kept=False))
    assert torch.equal(got.pair_sums, plain.pair_sums), (got.pair_sums, plain.pair_sums)
    assert torch.equal(got.pair_vals, plain.pair_vals) and torch.equal(got.total_sums, plain.total_sums)
    if c["kernel"][0] == "generic":
        return                            # (the generic kernel is the reference)
    ref = _forced(tcl, 1, lambda: _call(tcl, c, x))
    if c["mask"] == COMPUTED:
        assert torch.equal(got.pair_kept, ref.pair_kept)
    else:
        assert torch.allclose(got.pair_kept, ref.pair_kept, rtol=1e-6, atol=0.0)
    rtol = 1e-6 if c["T"] != BF16 else 1e-5
    assert torch.allclose(got.pair_sums, ref.pair_sums, rtol=rtol, atol=0.0)


@pytest.mark.parametrize("W", [64, 62])
def test_binary_dataset_masks_are_counted_exactly(tcl, W):
    c = _row(None, F32, GIVEN, W=W, B=3)
    x = _inputs(tcl, c)
    x["mask"] = (x["mask"] > 0.3).float()
    got = _call(tcl, c, x)
    assert torch.equal(got.pair_kept, x["mask"].double().sum((1, 2, 3)))


def test_calls_without_a_mask_keep_every_pixel(tcl):
    c = _row(None, F32, GIVEN)
    x = _inputs(tcl, c)
    x["mask"] = None
    got = _call(tcl, c, x)
    assert got.pair_kept.tolist() == [64.0 * 64.0] * 2 and float(got.total_kept) == 2 * 64.0 * 64.0
    band = _call(tcl, c, x, rows=(8, 40))
    assert band.pair_kept.tolist() == [32.0 * 64.0] * 2


@pytest.mark.parametrize("mask_kind", ["computed", "given"])
@pytest.mark.parametrize("loss", [L2, L1])
def test_warping_error_matches_the_torch_expression(tcl, mask_kind, loss):
    d = _dev()
    B, C, H, W = 3, 3, 128, 192
    ff, bf = tcl.synth.make_flows(B, H, W, seed=11, max_shift=16.0, device=d)
    prev, cur = tcl.synth.make_frames(B, C, H, W, seed=11, kind="smooth", device=d)
    with torch.no_grad():
        if mask_kind == "computed":
            m = tp.fb_consistency(ff, bf)
            assert torch.equal(tcl.fbcCheckTorch(ff, bf), m)     # (no verdict within 1e-6 of its threshold here)
        else:
            m = torch.rand(B, 1, H, W, device=d, generator=torch.Generator(device=d).manual_seed(3))
        w = tp.backward_warp(prev, bf)
        if loss == L2:
            want = (((m * (cur - w)) ** 2).sum((1, 2, 3)) / (C * m.sum((1, 2, 3)))).sqrt()
        else:
            want = (m * (w - cur).abs()).sum((1, 2, 3)) / (C * m.sum((1, 2, 3)))
    finalize = FIN_RMSE if loss == L2 else FIN_MEAN
    got = tcl.warping_error_per_pair(ff if mask_kind == "computed" else None, bf, prev, cur, mask=None if mask_kind == "computed" else m,
                                     loss=loss, finalize=finalize)
    assert got.shape == (B,) and got.dtype == torch.float32
    assert torch.allclose(got.double(), want.double(), rtol=1e-5, atol=0.0), (got, want)
    # ... and it is not the mean over all C*H*W values whenever the mask drops pixels
    plain = tcl.fused_forward(bf, prev, cur, ff=ff if mask_kind == "computed" else None, mask=None if mask_kind == "computed" else m,
                              loss=loss, finalize=finalize).pair_vals
    assert bool((got > plain).all())


def test_a_mask_that_keeps_nothing_gives_nan(tcl):
    d = _dev()
    B, H, W = 2, 64, 64
    _, bf = tcl.synth.make_flows(B, H, W, seed=2, device=d)
    prev, cur = tcl.synth.make_frames(B, 3, H, W, seed=2, device=d)
    m = torch.ones(B, 1, H, W, device=d)
    m[0] = 0.0
    got = tcl.warping_error_per_pair(None, bf, prev, cur, mask=m)
    with torch.no_grad():
        want = (((m * (cur - tp.backward_warp(prev, bf))) ** 2).sum((1, 2, 3)) / (3 * m.sum((1, 2, 3)))).sqrt()
    assert bool(torch.isnan(got[0])) and bool(torch.isnan(want[0]))
    assert torch.allclose(got[1:].double(), want[1:].double(), rtol=1e-5, atol=0.0)


# ------------------------------------------------------------------ modes
def _clip(tcl, T, H, W, seed=21, dtype=torch.float32):
    d = _dev()
    ff, bf = tcl.synth.make_flows(T - 1, H, W, seed=seed, max_shift=12.0, device=d)
    frames, _ = tcl.synth.make_frames(T, 3, H, W, seed=seed, kind="white", device=d, dtype=dtype)
    return frames, ff, bf


@pytest.mark.parametrize("H,W", [(96, 128), (37, 53)])
def test_clip_and_window_kept_sums_are_those_of_independent_pairs(tcl, H, W):
    T = 6
    frames, ff, bf = _clip(tcl, T, H, W)
    idx = torch.arange(T, dtype=torch.int32, device=frames.device)
    clip = tcl.fused_forward(bf, frames, frames, ff=ff, prev_index=idx[:-1], cur_index=idx[1:], want_kept=True)
    pairs = tcl.fused_forward(bf, frames[:-1], frames[1:], ff=ff, want_kept=True)
    assert torch.equal(clip.pair_kept, pairs.pair_kept) and torch.equal(clip.total_kept, pairs.total_kept)
    index = tcl.window_evaluations(T, 4)
    J = index["field_t"].numel()
    bank_ff, bank_bf = tcl.synth.make_flows(2 * J, H, W, seed=4, max_shift=12.0, device=frames.device)
    bank = bank_bf   # (field 2j and 2j+1 are the two directions; any fields serve the comparison)
    to = lambda k: index[k].to(frames.device)
    win = tcl.fused_forward(bank, frames, frames, ff=bank_ff, prev_index=to("prev_index"), cur_index=to("cur_index"), bf_index=to("bf_index"),
                            ff_index=to("ff_index"), pair_group=index["group"], want_kept=True)
    lk = lambda k: index[k].long().to(frames.device)
    ind = tcl.fused_forward(bank[lk("bf_index")], frames[lk("prev_index")], frames[lk("cur_index")], ff=bank_ff[lk("ff_index")], want_kept=True)
    assert torch.equal(win.pair_kept, ind.pair_kept)
    assert torch.equal(win.pair_sums, ind.pair_sums)


@pytest.mark.parametrize("kind", ["computed", "binary"])
def test_band_kept_sums_add_up_to_the_whole_frame(tcl, kind):
    d = _dev()
    B, H, W = 3, 192, 256
    ff, bf = tcl.synth.make_flows(B, H, W, seed=9, max_shift=12.0, device=d)
    prev, cur = tcl.synth.make_frames(B, 3, H, W, seed=9, device=d)
    mask = None if kind == "computed" else (torch.rand(B, 1, H, W, device=d) > 0.4).float()
    ffm = ff if kind == "computed" else None
    whole = tcl.fused_forward(bf, prev, cur, ff=ffm, mask=mask, want_kept=True)
    for cuts in ((0, 64, 192), (0, 96, 160, 192), (0, 7, 192)):
        parts = [tcl.fused_forward(bf, prev, cur, ff=ffm, mask=mask, rows=(a, b), want_kept=True) for a, b in zip(cuts[:-1], cuts[1:])]
        assert torch.equal(sum(p.pair_kept for p in parts), whole.pair_kept)
        assert float(sum(float(p.total_kept) for p in parts)) == float(whole.total_kept)
    want = (tcl.fbcCheckTorch(ff, bf) if kind == "computed" else mask)[:, :, 64:].double().sum((1, 2, 3))
    assert torch.equal(tcl.fused_forward(bf, prev, cur, ff=ffm, mask=mask, rows=(64, 192), want_kept=True).pair_kept, want)


def test_cropped_flow_views(tcl):
    d = _dev()
    B, H, W = 2, 100, 128
    ffp, bfp = tcl.synth.make_flows(B, 104, W, seed=13, max_shift=12.0, device=d)
    ff, bf = ffp[:, :, :H, :], bfp[:, :, :H, :]
    assert not ff.is_contiguous()
    prev, cur = tcl.synth.make_frames(B, 3, H, W, seed=13, device=d)
    got = tcl.fused_forward(bf, prev, cur, ff=ff, want_kept=True)
    want = tcl.fused_forward(bf.contiguous(), prev, cur, ff=ff.contiguous(), want_kept=True)
    assert torch.equal(got.pair_kept, want.pair_kept) and torch.equal(got.pair_sums, want.pair_sums)
    assert torch.equal(got.pair_kept, tcl.fbcCheckTorch(ff.contiguous(), bf.contiguous()).double().sum((1, 2, 3)))


@pytest.mark.parametrize("W", [128, 62])
@pytest.mark.parametrize("mask_kind", ["computed", "binary", "soft"])
def test_uint8_and_bf16_frames_give_the_fp32_kept_sums(tcl, W, mask_kind):
    d = _dev()
    B, H = 2, 96
    ff, bf = tcl.synth.make_flows(B, H, W, seed=17, max_shift=12.0, device=d)
    g = torch.Generator(device=d).manual_seed(17)
    u_prev = torch.randint(0, 256, (B, 3, H, W), device=d, dtype=torch.uint8, generator=g)
    u_cur = torch.randint(0, 256, (B, 3, H, W), device=d, dtype=torch.uint8, generator=g)
    m = torch.rand(B, 1, H, W, device=d, generator=g)
    if mask_kind == "binary":
        m = (m > 0.5).float()
    ffm, mm = (ff, None) if mask_kind == "computed" else (None, m)
    s, o = (2 / 255, -1.0)
    scale = torch.tensor(s, dtype=torch.float32, device=d)
    f_prev, f_cur = u_prev.float().mul(scale).add(o), u_cur.float().mul(scale).add(o)
    ref = tcl.fused_forward(bf, f_prev, f_cur, ff=ffm, mask=mm, want_kept=True)
    u8 = tcl.fused_forward(bf, u_prev, u_cur, ff=ffm, mask=mm, want_kept=True, u8_scale=s, u8_offset=o)
    b16 = tcl.fused_forward(bf, f_prev.bfloat16(), f_cur.bfloat16(), ff=ffm, mask=mm, want_kept=True)
    assert torch.equal(u8.pair_kept, ref.pair_kept) and torch.equal(u8.total_kept, ref.total_kept)
    assert torch.equal(b16.pair_kept, ref.pair_kept)


# ------------------------------------------------------------------ host entry
@pytest.mark.parametrize("H,W", [(96, 128), (37, 53)])
@pytest.mark.parametrize("mask_kind", ["computed", "given", "none"])
def test_host_entry_kept_sums_are_the_device_paths(tcl, H, W, mask_kind):
    d = _dev()
    T = 9
    frames, ff, bf = _clip(tcl, T, H, W, seed=29)
    m = torch.rand(T - 1, 1, H, W, device=d, generator=torch.Generator(device=d).manual_seed(1))
    ffm = ff if mask_kind == "computed" else None
    mm = m if mask_kind == "given" else None
    idx = torch.arange(T, dtype=torch.int32, device=d)
    dev = tcl.fused_forward(bf, frames, frames, ff=ffm, mask=mm, prev_index=idx[:-1], cur_index=idx[1:], want_kept=True)
    want_kept, want_sums = dev.pair_kept.cpu(), dev.pair_sums.cpu()
    h = lambda t: None if t is None else t.cpu().pin_memory()
    hcl = lambda t: t.cpu().permute(0, 2, 3, 1).contiguous().pin_memory().permute(0, 3, 1, 2)
    fr_h, ff_h, bf_h, m_h = h(frames), h(ffm), h(bf), h(mm)
    runs = {
        "default": dict(),
        "chunk3": dict(chunk_pairs=3),
        "chunk5-ring": dict(chunk_pairs=1, max_device_frames=5),
    }
    for name, kw in runs.items():
        vals, sums, kept = tcl.temporal_error_host(fr_h, ff_h, bf_h, mask=m_h, return_sums=True, return_kept=True, **kw)
        assert torch.equal(kept, want_kept), name
        assert torch.equal(sums, want_sums), name
        assert kept.is_pinned() and kept.dtype == torch.float64
    vals, kept = tcl.temporal_error_host(hcl(frames), None if ffm is None else hcl(ffm), hcl(bf), mask=m_h, return_kept=True, chunk_pairs=3)
    assert torch.equal(kept, want_kept)
    plain = tcl.temporal_error_host(fr_h, ff_h, bf_h, mask=m_h)
    assert torch.equal(plain, vals)
