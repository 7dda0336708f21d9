"""GPU suite of channels-last host data in the host-buffer entry: (F,H,W,C) frames and (P,H,W,2) flows, handed over as
`.permute(0, 3, 1, 2)` views, are read in place and de-interleaved on the device.  The contract: pair values and pair sums
are bit for bit those of the same call on `.contiguous()` copies, for every frame type, mask kind, chunk size and ring
size -- the de-interleave permutes elements, and the fused launches then see the same planar data chunk for chunk."""
import ctypes

import pytest
import torch

pytestmark = pytest.mark.gpu

CL_FRAMES, CL_FF, CL_BF = 1, 2, 4
NORMS = {"unit": (1 / 255, 0.0), "gan": (2 / 255, -1.0), "mean": (1.0, (-123.675, -116.28, -103.53))}   # test_gpu_u8_frames.py
KINDS = ["fp32", "bf16", "u8-unit", "u8-gan", "u8-mean"]
SHAPES = {"sintel": (436, 1024), "ragged": (37, 53)}   # the staged TMA kernel; the generic kernel, odd planes, unaligned runs
BITS = {"frames": CL_FRAMES, "flows": CL_FF | CL_BF, "all": CL_FRAMES | CL_FF | CL_BF}


def _dev():
    return torch.device("cuda:0")


def _frames(kind, T, H, W, seed):
    d = _dev()
    g = torch.Generator(device=d).manual_seed(seed)
    u = torch.randint(0, 256, (T, 3, H, W), device=d, dtype=torch.uint8, generator=g)
    if kind.startswith("u8"):
        s, o = NORMS[kind[3:]]
        return u.cpu(), dict(u8_scale=s, u8_offset=o)
    f = u.float().mul(torch.tensor(1 / 255, dtype=torch.float32, device=d)) + torch.rand(T, 3, H, W, device=d, generator=g) * 1e-3
    return (f if kind == "fp32" else f.to(torch.bfloat16)).cpu(), {}


def _flows(tcl, P, H, W, seed):
    ff, bf = tcl.synth.make_flows(P, H, W, seed=seed, max_shift=12.0, max_rot_deg=3.0, n_rects=3, rect_shift=8.0, device=_dev())
    return ff.cpu(), bf.cpu()


def _hwc(t, pinned):
    """The same values as a channels-last view of interleaved (N,H,W,C) memory, pinned or pageable."""
    a = t.permute(0, 2, 3, 1).contiguous()
    return (a.pin_memory() if pinned else a).permute(0, 3, 1, 2)


def _host(t, pinned):
    return t.pin_memory() if pinned else t


def _layout(frames, ff, bf, bits, pinned):
    """The call's inputs with the layouts of `bits`: channels-last where a bit is set, planar elsewhere."""
    pick = lambda t, b: None if t is None else (_hwc(t, pinned) if bits & b else _host(t.contiguous(), pinned))
    return pick(frames, CL_FRAMES), pick(ff, CL_FF), pick(bf, CL_BF)


def _both(tcl, frames, ff, bf, bits, pinned=True, **kw):
    """(channels-last call, planar call) on the same values; asserts the channels-last inputs were not written."""
    fr_c, ff_c, bf_c = _layout(frames, ff, bf, bits, pinned)
    for t, b in ((fr_c, CL_FRAMES), (ff_c, CL_FF), (bf_c, CL_BF)):
        if t is not None:
            assert tcl.ops._is_channels_last(t) == bool(bits & b)
    before = [None if t is None else t.clone() for t in (fr_c, ff_c, bf_c)]
    got = tcl.temporal_error_host(fr_c, ff_c, bf_c, return_sums=True, **kw)
    want = tcl.temporal_error_host(_host(frames.contiguous(), pinned), None if ff is None else _host(ff.contiguous(), pinned),
                                   _host(bf.contiguous(), pinned), return_sums=True, **kw)
    for t, b in zip((fr_c, ff_c, bf_c), before):
        if t is not None:
            assert torch.equal(t, b), "host input mutated"
    return got, want


def _assert_same(got, want):
    assert got[0].shape == want[0].shape and torch.equal(got[0], want[0]), (got[0], want[0])
    assert torch.equal(got[1], want[1]), (got[1], want[1])
    assert bool(torch.isfinite(got[1]).all())


@pytest.mark.parametrize("shape", sorted(SHAPES))
@pytest.mark.parametrize("bits", sorted(BITS))
@pytest.mark.parametrize("kind", KINDS)
def test_computed_mask_equals_planar(tcl, kind, bits, shape):
    H, W = SHAPES[shape]
    T = 8
    frames, norm = _frames(kind, T, H, W, H + T)
    ff, bf = _flows(tcl, T - 1, H, W, W + T)
    # chunks of 1 and 2 pairs: the ring's three slots (and their staging areas) and both copy streams are reused several times
    for chunk in (1, 2, 0):
        _assert_same(*_both(tcl, frames, ff, bf, BITS[bits], chunk_pairs=chunk, **norm))


@pytest.mark.parametrize("shape", sorted(SHAPES))
@pytest.mark.parametrize("bits", [CL_FRAMES, CL_BF, CL_FRAMES | CL_BF])
@pytest.mark.parametrize("kind", ["fp32", "bf16", "u8-gan"])
def test_dataset_mask_equals_planar(tcl, kind, bits, shape):
    H, W = SHAPES[shape]
    T = 7
    frames, norm = _frames(kind, T, H, W, 3 + T)
    _, bf = _flows(tcl, T - 1, H, W, 5 + T)
    mask = (torch.rand(T - 1, 1, H, W, generator=torch.Generator().manual_seed(4)) > 0.3).float()
    for chunk in (1, 3):
        _assert_same(*_both(tcl, frames, None, bf, bits, chunk_pairs=chunk, mask=mask, **norm))


@pytest.mark.parametrize("pinned", [True, False])
@pytest.mark.parametrize("kind", ["fp32", "bf16", "u8-mean"])
def test_window_indices_and_frame_ring_equal_planar(tcl, kind, pinned):
    """The evaluations of temporal windows: a chunk uploads up to two frames per pair, in several runs, and a ring of 8 slots
    for 12 frames hands slots out again out of order, so staged runs start anywhere in the staging area."""
    H, W, T = 37, 53, 12
    idx = tcl.ops.window_evaluations(T, 4)
    frames, norm = _frames(kind, T, H, W, 17)
    J = idx["field_t"].numel()
    bank_ff, bank_bf = _flows(tcl, 2 * J, H, W, 19)
    ff, bf = bank_ff[idx["ff_index"].long()], bank_bf[idx["bf_index"].long()]
    pi, ci = idx["prev_index"], idx["cur_index"]
    for chunk, slots in ((2, 8), (3, 8), (1, None), (5, None)):
        got, want = _both(tcl, frames, ff, bf, BITS["all"], pinned, prev_index=pi, cur_index=ci, chunk_pairs=chunk,
                          max_device_frames=slots, **norm)
        _assert_same(got, want)


@pytest.mark.parametrize("kind", ["fp32", "u8-unit"])
def test_sintel_frame_ring_equals_planar(tcl, kind):
    H, W, T = 436, 1024, 9
    frames, norm = _frames(kind, T, H, W, 23)
    ff, bf = _flows(tcl, T - 1, H, W, 29)
    for bits in (CL_FRAMES, BITS["all"]):
        _assert_same(*_both(tcl, frames, ff, bf, bits, chunk_pairs=1, max_device_frames=4, **norm))


def test_clip_without_pairs(tcl):
    frames, _ = _frames("u8-unit", 1, 37, 53, 1)
    ff, bf = _flows(tcl, 1, 37, 53, 1)
    v, s = tcl.temporal_error_host(_hwc(frames, True), _hwc(ff[:0], True), _hwc(bf[:0], True), return_sums=True)
    assert v.shape == (0,) and s.shape == (0,)


def test_caller_storage_reaches_the_c_abi_and_is_converted_on_the_device(tcl, monkeypatch):
    """The channels-last tensors' own data_ptr() is what the C ABI receives (no host copy), with the bits set; the profile
    shows the device conversions running, and none for planar inputs."""
    H, W, T = 64, 96, 6
    frames, norm = _frames("u8-gan", T, H, W, 31)
    ff, bf = _flows(tcl, T - 1, H, W, 31)
    fr_c, ff_c, bf_c = _hwc(frames, True), _hwc(ff, True), _hwc(bf, True)
    real = tcl._cabi.lib()
    seen = []

    class Spy:
        def __getattr__(self, name):
            return getattr(real, name)

        def tclb200_tcl_forward_host(self, ref, stream):
            a = ref._obj
            seen.append((a.frames, a.ff, a.bf, a.channels_last))
            return real.tclb200_tcl_forward_host(ref, stream)

    monkeypatch.setattr(tcl._cabi, "lib", lambda: Spy())
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        got = tcl.temporal_error_host(fr_c, ff_c, bf_c, **norm)
    names = [e.name for e in prof.events()]
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof_planar:
        want = tcl.temporal_error_host(frames.pin_memory(), ff.pin_memory(), bf.pin_memory(), **norm)
    names_planar = [e.name for e in prof_planar.events()]
    assert seen[0] == (fr_c.data_ptr(), ff_c.data_ptr(), bf_c.data_ptr(), CL_FRAMES | CL_FF | CL_BF)
    assert seen[1][3] == 0
    assert torch.equal(got, want)
    assert any("hwc_to_chw_kernel" in n for n in names), names
    assert any("hwc2_split_kernel" in n for n in names), names
    assert not any("hwc_to_chw_kernel" in n or "split_kernel" in n for n in names_planar), names_planar


def test_sync_false_keeps_the_callers_tensors_alive(tcl):
    H, W, T = 37, 53, 6
    frames, _ = _frames("bf16", T, H, W, 37)
    ff, bf = _flows(tcl, T - 1, H, W, 37)
    fr_c, ff_c, bf_c = _hwc(frames, True), _hwc(ff, True), _hwc(bf, True)
    out = tcl.temporal_error_host(fr_c, ff_c, bf_c, sync=False)
    assert out._tcl_keepalive[0] is fr_c and out._tcl_keepalive[1] is ff_c and out._tcl_keepalive[2] is bf_c
    torch.cuda.current_stream().synchronize()
    assert torch.equal(out, tcl.temporal_error_host(frames, ff, bf))


def test_sharded_host_evaluation_takes_channels_last_inputs(tcl):
    H, W, T = 37, 53, 9
    frames, norm = _frames("u8-mean", T, H, W, 41)
    ff, bf = _flows(tcl, T - 1, H, W, 41)
    pi, ci = torch.arange(T - 1, dtype=torch.int32), torch.arange(1, T, dtype=torch.int32)
    seq = torch.tensor([0] * 4 + [1] * (T - 5), dtype=torch.long)
    got = tcl.sharding.evaluate_sharded_host(_hwc(frames, True), _hwc(ff, True), _hwc(bf, True), pi, ci, seq, 2, chunk_pairs=3, **norm)
    want = tcl.sharding.evaluate_sharded_host(frames, ff, bf, pi, ci, seq, 2, chunk_pairs=3, **norm)
    assert set(got) == set(want)
    for k in want:
        assert torch.equal(got[k], want[k]), k
