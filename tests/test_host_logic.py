"""CPU suite: host-side logic of the wrappers that needs no GPU (file formats, argument checks, no-fallback behaviour)."""
import numpy as np
import pytest
import torch


def test_flo_round_trip_matches_flowlib_layout(tcl, tmp_path):
    # utils/flowlib.py:33-55: 'PIEH', int32 width, int32 height, H x W x 2 float32
    rng = np.random.default_rng(0)
    flow = rng.standard_normal((7, 13, 2)).astype(np.float32)
    path = str(tmp_path / "a.flo")
    tcl.ingest.write_flo(path, flow)
    raw = open(path, "rb").read()
    assert raw[:4] == b"PIEH" and np.frombuffer(raw[4:12], np.int32).tolist() == [13, 7]
    assert len(raw) == 12 + flow.nbytes
    assert np.array_equal(tcl.ingest.read_flo(path), flow)
    open(path, "wb").write(b"XXXX" + raw[4:])
    with pytest.raises(Exception):
        tcl.ingest.read_flo(path)


def test_wrappers_refuse_cpu_tensors_instead_of_falling_back(tcl):
    x, f = torch.zeros(1, 3, 8, 8), torch.zeros(1, 2, 8, 8)
    for call in (lambda: tcl.warp(x, f), lambda: tcl.fs_warp(x, f), lambda: tcl.fbcCheckTorch(f, f),
                 lambda: tcl.gradient(f[:, 0]), lambda: tcl.temporal_error(f, f, x, x),
                 lambda: tcl.temporal_loss(torch.ones(1, 1, 8, 8), x, x, f), lambda: tcl.hwc_split(torch.zeros(1, 8, 8, 9), tcl.ingest.FC2_LAYOUT),
                 lambda: tcl.upsample_flow(f, torch.zeros(1, 576, 8, 8)), lambda: tcl.temporal_error_clip(x.repeat(2, 1, 1, 1), f, f),
                 lambda: tcl.long_term_blend_step(torch.ones(1, 1, 8, 8), f, f, x, x)):
        with pytest.raises(RuntimeError):
            call()


def test_fc2_layout_is_the_reference_slicing(tcl):
    # core/data_loader.py:243-245 / learning-based/datasets.py:52-54: imgs 0:6, mask 6:7, flow 7:9
    assert tcl.ingest.FC2_LAYOUT == (("img1", 0, 3), ("img2", 3, 3), ("mask", 6, 1), ("flow", 7, 2))
    assert sum(c for _, _, c in tcl.ingest.FC2_LAYOUT) == 9


# ------------------------------------------------------------------ host-side logic added around the kernels (no GPU needed)
def test_flow_view_recognises_row_dense_views(tcl):
    """ops._flow_view: cropped views of a padded flow (InputPadder.unpad, flow_up[:,:,:H,:]) are handed over through their
    strides; anything that is not row-dense is made contiguous."""
    import torch
    fv = tcl.ops._flow_view
    B, H, W = 3, 10, 16
    dense = torch.randn(B, 2, H, W)
    t, plane, batch = fv(dense)
    assert t is dense and (plane, batch) == (0, 0)                                  # dense: nothing to say
    big = torch.randn(B, 2, H + 4, W)
    for view in (big[:, :, 2:H + 2, :], big[:, :, :H, :]):
        t, plane, batch = fv(view)
        assert t.data_ptr() == view.data_ptr() and plane == (H + 4) * W and batch == 2 * (H + 4) * W
    one = torch.randn(1, 2, H + 8, W)[:, :, 3:H + 3, :]                             # B == 1: the pair stride follows the plane stride
    t, plane, batch = fv(one)
    assert t.data_ptr() == one.data_ptr() and plane == (H + 8) * W and batch == 2 * plane
    wide = torch.randn(B, 2, H, W + 8)[:, :, :, 4:W + 4]                            # cropped columns: rows are not dense
    t, plane, batch = fv(wide)
    assert t.is_contiguous() and (plane, batch) == (0, 0) and torch.equal(t, wide)
    half = torch.randn(B, 2, H, W, dtype=torch.float64)[:, :, :, :]                 # wrong dtype -> converted copy
    t, plane, batch = fv(half)
    assert t.dtype == torch.float32 and (plane, batch) == (0, 0)
    import pytest
    with pytest.raises(RuntimeError):
        fv(torch.randn(B, 3, H, W))


def test_no_gpu_means_loud_errors_not_fallbacks(tcl):
    import numpy as np
    import pytest
    import torch
    if torch.cuda.is_available():
        pytest.skip("this check is for the GPU-less build container")
    z = np.zeros((4, 5, 2), np.float32)
    with pytest.raises(RuntimeError):
        tcl.cv2compat.warp_flow(z, z)
    with pytest.raises(RuntimeError):
        tcl.cv2compat.fb_check(z, z)
    with pytest.raises(RuntimeError):
        tcl.temporal_error_host(torch.zeros(2, 3, 4, 8), torch.zeros(1, 2, 4, 8), torch.zeros(1, 2, 4, 8))
    with pytest.raises(RuntimeError):
        tcl.sintel_occlusion_mask(torch.zeros(4, 8, dtype=torch.uint8))
    with pytest.raises(RuntimeError):
        tcl.warp(torch.zeros(1, 3, 4, 8), torch.zeros(1, 2, 4, 8))


def test_aggregation_and_ingest_entries_validate_arguments(tcl):
    lib = tcl._cabi.lib()
    assert lib.tclb200_pack_sequence_sums(None, None, None, 0, 0, 1.0, None, None) == 1
    assert lib.tclb200_pack_sequence_sums(None, None, None, 5, 3, 1.0, 8, None) == 1        # pairs without values
    assert lib.tclb200_unpack_sequence_means(None, 3, None, None) == 1
    assert lib.tclb200_occlusion_u8_to_mask(None, None, 16, None) == 1
    assert lib.tclb200_cv2_remap(None, None, None, 1, 4, 4, 3, None) == 1
    assert lib.tclb200_cv2_fb_check(None, None, None, 1, 4, 4, 3, 0, None, None) == 1
    assert lib.tclb200_gradient_strided(8, 4, 8, 1, 4, 4, None) == 1                         # stride below H*W
    assert b"stride" in lib.tclb200_last_error()


def test_cpu_and_device_forms_of_the_aggregation_share_one_definition(tcl):
    """sharding.pack_local / unpack on CPU tensors (what the gloo tests exercise) against hand-computed numbers."""
    import torch
    sh = tcl.sharding
    vals = torch.tensor([1.0, 3.0, 5.0, 7.0])
    seq = torch.tensor([0, 0, 2, 2])
    packed = sh.pack_local(vals, torch.tensor(8.0, dtype=torch.float64), seq, 3, 2)
    assert packed.tolist() == [4.0, 0.0, 12.0, 2.0, 0.0, 2.0, 8.0, 8.0]
    u = sh.unpack(packed, 3)
    assert u["per_sequence_mean"].tolist() == [2.0, 0.0, 6.0]
    assert float(u["mean_over_sequences"]) == 4.0 and float(u["mean_over_pairs"]) == 4.0       # the empty sequence does not count
    assert float(u["pooled_rmse"]) == 1.0 and float(u["n_pairs"]) == 4.0


def _raft_pad(ht, wd, mode):
    """InputPadder._pad as RAFT publishes it (core/utils/utils.py; vendored upstream as utils/raft/raft/utils/utils.py:7-24)."""
    pad_ht = (((ht // 8) + 1) * 8 - ht) % 8
    pad_wd = (((wd // 8) + 1) * 8 - wd) % 8
    if mode == "sintel":
        return [pad_wd // 2, pad_wd - pad_wd // 2, pad_ht // 2, pad_ht - pad_ht // 2]
    return [pad_wd // 2, pad_wd - pad_wd // 2, 0, pad_ht]


def test_input_padder_is_the_reference_one(tcl):
    """sintel_eval.InputPadder against RAFT's InputPadder (its padding, replicate-padded images and unpad) and against
    its definition: replicate padding to multiples of 8, rows split top / bottom in 'sintel' mode."""
    import torch.nn.functional as F
    ours = tcl.sintel_eval.InputPadder
    g = torch.Generator().manual_seed(3)
    for H, W in ((436, 1024), (432, 1024), (44, 61), (8, 8), (7, 9), (1080, 1920)):
        x = torch.rand(1, 3, H, W, generator=g)
        for mode in ("sintel", "kitti"):
            p = ours(x.shape, mode)
            (y,) = p.pad(x)
            assert y.shape[-2] % 8 == 0 and y.shape[-1] % 8 == 0 and y.shape[-2] - H < 8 and y.shape[-1] - W < 8
            assert torch.equal(p.unpad(y), x)
            q = _raft_pad(H, W, mode)
            assert q == p._pad and torch.equal(F.pad(x, q, mode="replicate"), y)
            assert torch.equal(y[..., q[2]:y.shape[-2] - q[3], q[0]:y.shape[-1] - q[1]], x)
    assert ours((436, 1024))._pad == [0, 0, 2, 2] and ours((436, 1024), "kitti")._pad == [0, 0, 0, 4]


def test_computeRAFT_pads_then_crops_from_the_top(tcl):
    seen = {}

    def model(a, b, iters=20, test_mode=True):
        seen["shape"], seen["iters"] = tuple(a.shape), iters
        return None, torch.arange(a.shape[-2], dtype=torch.float32).view(1, 1, -1, 1).expand(1, 2, a.shape[-2], a.shape[-1])
    img = torch.zeros(1, 3, 436, 64)
    f = tcl.sintel_eval.computeRAFT(model, img, img, it=12)
    assert seen == {"shape": (1, 3, 440, 64), "iters": 12}
    assert f.shape == (1, 2, 436, 64) and float(f[0, 0, 0, 0]) == 0.0 and float(f[0, 0, -1, 0]) == 435.0   # flow_up[:, :, :H, :]
    assert tcl.sintel_eval.computeRAFT(model, img, img, crop=False).shape == (1, 2, 440, 64)
