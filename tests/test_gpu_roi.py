"""GPU parity: b200 ROI Align (through the C ABI) against the oracle, the golden fixtures
from the live reference, and the installed torchvision op."""
import numpy as np
import pytest
import torch

from conftest import assert_close, load_golden, load_roi_wrappers_golden
from oracle import native

pytestmark = pytest.mark.gpu

import alufe_b200  # noqa: E402,F401
from alufe_b200 import roi, synth  # noqa: E402


def _run(feat, rois, ps, scale, sr, al, nhwc=False):
    f = torch.from_numpy(feat).cuda()
    if nhwc:
        f = f.contiguous(memory_format=torch.channels_last)
    out = roi.roi_align(f, torch.from_numpy(rois).cuda(), ps, scale, sr, al)
    torch.cuda.synchronize()
    return out.cpu().numpy()


@pytest.mark.parametrize("nhwc", [False, True])
def test_roi_vs_golden(nhwc):
    g = load_golden("roi")
    for tag in "abcd":
        ph, pw, sr, al = (int(v) for v in g["arg_" + tag])
        got = _run(g["feat"], g["rois"], (ph, pw), 20 / 640.0, sr, bool(al), nhwc)
        assert_close(got, g["out_" + tag], what="golden roi %s nhwc=%s" % (tag, nhwc))


@pytest.mark.parametrize("nhwc", [False, True])
@pytest.mark.parametrize("cfg", ["c1", "c2", "c5"])
@pytest.mark.parametrize("ps", [(10, 10), (7, 7)])
def test_roi_vs_oracle_named_shapes(cfg, ps, nhwc):
    Hf, Wf, H_in, W_in, n = synth.CONFIGS[cfg]
    C = 512 if cfg != "c5" else 96
    feat = synth.feature_map(0, 1, C, Hf, Wf)
    rng = np.random.default_rng(3)
    boxes = np.concatenate([synth.random_boxes(rng, n, H_in, W_in), synth.edge_case_boxes(H_in, W_in)])
    rois = np.concatenate([np.zeros((len(boxes), 1)), boxes], 1).astype(np.float32)
    scale = Hf / float(H_in)
    want = native.roi_align(feat, rois, ps, scale, 2, True)
    assert_close(_run(feat, rois, ps, scale, 2, True, nhwc), want, what=cfg)


@pytest.mark.parametrize("nhwc", [False, True])
def test_roi_batched_maps_odd_shapes(nhwc):
    """c3-style batch indices, C not a multiple of 32, W not a multiple of 4, large boxes
    (slow path), adaptive sampling, not-aligned mode, out-of-range batch index -> zeros."""
    rng = np.random.default_rng(5)
    feat = rng.standard_normal((5, 70, 23, 37), dtype=np.float32)
    boxes = rng.uniform(-100, 1300, (64, 4))
    boxes[:8] = [0, 0, 1184, 736]                       # whole-map boxes
    boxes[8:16, 2:] = boxes[8:16, :2] + rng.uniform(200, 600, (8, 2))
    rois = np.concatenate([rng.integers(0, 5, (64, 1)).astype(np.float64), boxes], 1).astype(np.float32)
    for ps, sr, al in [((10, 10), 2, True), ((7, 7), 2, False), ((10, 10), -1, True), ((7, 7), 0, False),
                       ((10, 10), 3, True), ((4, 6), 2, True), ((1, 1), -1, False)]:
        want = native.roi_align(feat, rois, ps, 1 / 32.0, sr, al)
        assert_close(_run(feat, rois, ps, 1 / 32.0, sr, al, nhwc), want, what="odd %s %s %s" % (ps, sr, al))
    bad = rois.copy()
    bad[3, 0] = 9
    got = _run(feat, bad, (10, 10), 1 / 32.0, 2, True, nhwc)
    assert np.all(got[3] == 0) and np.isfinite(got).all()


def test_roi_vs_torchvision_cuda_and_cpu():
    tv = pytest.importorskip("torchvision")
    feat = synth.feature_map(1, 2, 512, 40, 40)
    rng = np.random.default_rng(9)
    boxes = synth.random_boxes(rng, 64, 1280, 1280)
    rois = np.concatenate([rng.integers(0, 2, (64, 1)).astype(np.float64), boxes], 1).astype(np.float32)
    got = _run(feat, rois, (10, 10), 40 / 1280.0, 2, True)
    cpu = tv.ops.roi_align(torch.from_numpy(feat), torch.from_numpy(rois), (10, 10), 40 / 1280.0, 2, True).numpy()
    assert_close(got, cpu, what="tv cpu")
    gpu = tv.ops.roi_align(torch.from_numpy(feat).cuda(), torch.from_numpy(rois).cuda(), (10, 10), 40 / 1280.0, 2, True)
    # torchvision's own CUDA kernel is only a second opinion: it differs from its CPU op (the
    # parity contract) by up to ~2e-5 absolute on these inputs, so it gets a looser bound.
    assert_close(got, gpu.cpu().numpy(), rtol=1e-4, atol=1e-4, what="tv cuda")


def test_roi_wrappers_match_reference_call_conventions():
    """tracking.py:193-221 and trainingCard.py:24-79 calling conventions."""
    feat = synth.feature_map(2, 1, 64, 20, 20)
    boxes = synth.random_boxes(np.random.default_rng(2), 8, 640, 640)
    f = torch.from_numpy(feat).cuda()
    got = roi.roi_align_from_input_boxes(f, boxes.tolist(), (640, 640)).cpu().numpy()
    rois = np.concatenate([np.zeros((8, 1)), boxes], 1).astype(np.float32)
    assert got.shape == (8, 64, 7, 7)
    assert_close(got, native.roi_align(feat, rois, (7, 7), 20 / 640.0, 2, True))
    # _preprocess_roi: sorted, scaled per axis, clamped, min size 1, spatial_scale 1
    b = boxes.copy()
    b[0] = [300, 300, 250, 240]
    b[1] = [630, 630, 700, 700]
    got = roi.preprocess_roi(f, torch.from_numpy(b), (640, 640)).cpu().numpy()
    x1, x2 = np.minimum(b[:, 0], b[:, 2]), np.maximum(b[:, 0], b[:, 2])
    y1, y2 = np.minimum(b[:, 1], b[:, 3]), np.maximum(b[:, 1], b[:, 3])
    fb = np.stack([x1, y1, x2, y2], 1).astype(np.float32) * np.float32(20 / 640.0)
    fb = np.clip(fb, 0, 19)
    fb[:, 2] = np.clip(np.maximum(fb[:, 2], fb[:, 0] + 1), 0, 19)
    fb[:, 3] = np.clip(np.maximum(fb[:, 3], fb[:, 1] + 1), 0, 19)
    r2 = np.concatenate([np.zeros((8, 1), np.float32), fb], 1)
    assert_close(got, native.roi_align(feat, r2, (10, 10), 1.0, 2, True))
    with pytest.raises(AssertionError):
        roi.preprocess_roi(torch.zeros(2, 4, 5, 5).cuda(), torch.zeros(1, 4), (10, 10))


def test_roi_wrappers_vs_reference_golden():
    """roi_align_from_input_boxes / preprocess_roi against fixtures recorded from the reference's OWN methods
    (tracking.py:193-221, trainingCard.py:24-79; tests/golden/make_golden.py::run_roi_wrapper_cases)."""
    g = load_roi_wrappers_golden()
    for tag in ("sq", "wide"):
        boxes, hw = g[tag + "_boxes"], tuple(int(v) for v in g[tag + "_hw"])
        f = torch.from_numpy(g[tag + "_feat"]).cuda()
        for ps in (7, 10):
            got = roi.roi_align_from_input_boxes(f, boxes.tolist(), hw, out_size=(ps, ps))
            assert_close(got.cpu().numpy(), g["%s_r1_%d" % (tag, ps)], what="%s r1 %d" % (tag, ps))
        got = roi.roi_align_from_input_boxes(f, torch.from_numpy(boxes).cuda(), hw)          # device boxes, default 7x7
        assert_close(got.cpu().numpy(), g[tag + "_r1_7"], what=tag + " r1 device boxes")
        got = roi.preprocess_roi(f, torch.from_numpy(boxes), hw)
        assert_close(got.cpu().numpy(), g[tag + "_r2_10"], what=tag + " r2")
        got = roi.preprocess_roi(f, torch.from_numpy(boxes).cuda(), hw, output_size=(7, 7), enforce_min_size=0.0)
        assert_close(got.cpu().numpy(), g[tag + "_r2_7_nomin"], what=tag + " r2 nomin")


def test_roi_box_prep_kernel_bit_exact_and_batched_c3():
    """b200_roi_boxes_prep_f32 (one launch instead of the wrappers' eager tensor ops) against the oracle's restatement
    of trainingCard.py:38-69, bit for bit (inverted, out-of-image, sub-pixel, NaN boxes, strided [N,6] rows), and
    BASELINE config 3 as ONE call: 256 maps x 16 boxes with a per-box image index == 256 reference-shaped calls."""
    from oracle import roi_wrappers_ref
    from alufe_b200.roi import _prep_boxes
    from alufe_b200 import _lib
    rng = np.random.default_rng(31)
    b = synth.random_boxes(rng, 300, 720, 1280).astype(np.float32)
    edge = synth.edge_case_boxes(720, 1280).astype(np.float32)
    b[:len(edge)] = edge
    b[40] = [500, 400, 100, 50]                       # inverted
    b[41] = [-50, -20, 3000, 2000]                    # far outside
    b[42] = [10.25, 10.25, 10.5, 10.5]                # smaller than the minimum size
    b[43] = [np.nan, 5, 50, 60]
    for min_size in (1.0, 0.0, 2.5):
        want = roi_wrappers_ref.preprocess_rois(b, (23, 40), (720, 1280), min_size)
        got = _prep_boxes(torch.from_numpy(b).cuda(), "cuda:0", _lib.BOXES_TRAINING, None, (720, 1280), (23, 40), min_size)
        np.testing.assert_array_equal(got.cpu().numpy(), want)
    six = torch.from_numpy(np.concatenate([b, rng.random((300, 2), dtype=np.float32)], 1)).cuda()
    idx = rng.integers(0, 7, 300).astype(np.int32)
    got = _prep_boxes(six, "cuda:0", _lib.BOXES_INPUT, idx).cpu().numpy()
    np.testing.assert_array_equal(got[:, 1:], b)
    np.testing.assert_array_equal(got[:, 0], idx.astype(np.float32))
    assert _prep_boxes(torch.zeros((0, 4)), "cuda:0", _lib.BOXES_INPUT).shape == (0, 5)
    # config 3 in one call
    Bm, per, Cc = 256, 16, 32
    feat = torch.randn((Bm, Cc, 40, 40), device="cuda", generator=torch.Generator(device="cuda").manual_seed(3))
    boxes = np.concatenate([synth.random_boxes(rng, per, 1280, 1280) for _ in range(Bm)]).astype(np.float32)
    bi = np.repeat(np.arange(Bm), per)
    one = roi.preprocess_roi(feat, torch.from_numpy(boxes), (1280, 1280), batch_index=bi)
    assert one.shape == (Bm * per, Cc, 10, 10)
    for m in (0, 17, 255):                             # the reference's loop body (trainingCard.py:86-129), image by image
        ref_call = roi.preprocess_roi(feat[m:m + 1], torch.from_numpy(boxes[m * per:(m + 1) * per]), (1280, 1280))
        assert torch.equal(one[m * per:(m + 1) * per], ref_call)
        want = roi_wrappers_ref.preprocess_roi(feat[m:m + 1].cpu().numpy(), boxes[m * per:(m + 1) * per], (1280, 1280))
        assert_close(ref_call.cpu().numpy(), want, what="c3 image %d" % m)
    a = roi.roi_align_from_input_boxes(feat, torch.from_numpy(boxes).cuda(), (1280, 1280), out_size=(10, 10), batch_index=bi)
    assert torch.equal(a[16:32], roi.roi_align_from_input_boxes(feat[1:2], boxes[16:32].tolist(), (1280, 1280), out_size=(10, 10)))


@pytest.mark.parametrize("nhwc", [False, True])
def test_roi_c5_full_width_vs_oracle(nhwc):
    """BASELINE config 5 at full width: 64 maps [512,34,60], 128 boxes each = 8 192 ROIs in ONE launch (the prep +
    multi-tile / TMA / pipelined kernels), every ROI against the oracle."""
    S, C, Hf, Wf, H_in, W_in, n = 64, 512, 34, 60, 1088, 1920, 128
    rng = np.random.default_rng(17)
    gen = torch.Generator(device="cuda").manual_seed(5)
    f = torch.randn((S, C, Hf, Wf), device="cuda", generator=gen)
    boxes = np.concatenate([synth.random_boxes(rng, n, H_in, W_in) for _ in range(S)])
    edge = synth.edge_case_boxes(H_in, W_in)
    boxes[:len(edge)] = edge
    rois = np.concatenate([np.repeat(np.arange(S), n)[:, None].astype(np.float64), boxes], 1).astype(np.float32)
    fin = f.contiguous(memory_format=torch.channels_last) if nhwc else f
    got = roi.roi_align(fin, torch.from_numpy(rois).cuda(), (10, 10), Hf / float(H_in), 2, True)
    assert got.shape == (S * n, C, 10, 10)
    for s0 in range(0, S, 8):                                        # eight maps at a time keeps host memory modest
        sub = rois[s0 * n:(s0 + 8) * n].copy()
        sub[:, 0] -= s0
        want = native.roi_align(f[s0:s0 + 8].cpu().numpy(), sub, (10, 10), Hf / float(H_in), 2, True)
        assert_close(got[s0 * n:(s0 + 8) * n].cpu().numpy(), want, rtol=1e-5, atol=2e-6, what="c5 maps %d.." % s0)


def test_roi_full_size_properties():
    """BASELINE config 3 size ([4096,512,10,10]): size-independent checks only.
    (i) a constant map gives the constant for fully-inside boxes; (ii) linearity in the map;
    (iii) a random subset of ROIs agrees with the oracle."""
    Bm, C, Hf, Wf = 256, 512, 40, 40
    rng = np.random.default_rng(0)
    boxes = np.concatenate([synth.random_boxes(rng, 16, 1280, 1280) for _ in range(Bm)])
    rois = np.concatenate([np.repeat(np.arange(Bm), 16)[:, None].astype(np.float64), boxes], 1).astype(np.float32)
    r = torch.from_numpy(rois).cuda()
    gen = torch.Generator(device="cuda").manual_seed(0)
    a = torch.randn((Bm, C, Hf, Wf), device="cuda", generator=gen)
    b = torch.randn((Bm, C, Hf, Wf), device="cuda", generator=gen)
    ya = roi.roi_align(a, r, (10, 10), 40 / 1280.0, 2, True)
    yb = roi.roi_align(b, r, (10, 10), 40 / 1280.0, 2, True)
    ys = roi.roi_align(a * 2 + b, r, (10, 10), 40 / 1280.0, 2, True)
    assert ya.shape == (4096, 512, 10, 10)
    assert torch.allclose(ys, 2 * ya + yb, rtol=1e-5, atol=1e-5)
    ones = roi.roi_align(torch.full_like(a, 3.25), r, (10, 10), 40 / 1280.0, 2, True)
    assert torch.allclose(ones, torch.full_like(ones, 3.25), rtol=1e-6, atol=0)
    pick = rng.choice(4096, 24, replace=False)
    maps = np.unique(rois[pick, 0].astype(int))
    sub_feat = a[maps].cpu().numpy()
    sub_rois = rois[pick].copy()
    sub_rois[:, 0] = np.searchsorted(maps, sub_rois[:, 0].astype(int))
    want = native.roi_align(sub_feat, sub_rois, (10, 10), 40 / 1280.0, 2, True)
    assert_close(ya[torch.from_numpy(pick).cuda()].cpu().numpy(), want, what="c3 subset")


@pytest.mark.parametrize("nhwc", [False, True])
@pytest.mark.parametrize("ps", [(10, 10), (7, 7)])
def test_roi_large_launch_path_vs_oracle(ps, nhwc):
    """More than 16 384 (ROI, channel-tile) pairs: the per-ROI prep pass + the persistent producer/consumer
    kernel.  Every ROI is checked against the oracle; the list mixes ordinary boxes, the reference's edge
    cases, boxes whose footprint is too large to stage (handled inside a consumer warp), bad batch indices,
    and a channel count with a ragged last tile."""
    rng = np.random.default_rng(17)
    Bm, C, Hf, Wf = 3, 150, 40, 48
    feat = rng.standard_normal((Bm, C, Hf, Wf), dtype=np.float32)
    n = 3400                                            # x 5 channel tiles = 17 000 tiles
    boxes = synth.random_boxes(rng, n, 1280, 1536)
    edge = synth.edge_case_boxes(1280, 1536)
    boxes[100:100 + len(edge)] = edge
    boxes[500:540] = [[0, 0, 1536, 1280]] * 40          # whole map
    boxes[900:940, 2:] = boxes[900:940, :2] + rng.uniform(300, 700, (40, 2))
    bidx = rng.integers(0, Bm, (n, 1)).astype(np.float64)
    bidx[1200:1204] = [[-1], [3], [7], [-2]]
    rois = np.concatenate([bidx, boxes], 1).astype(np.float32)
    good = (bidx[:, 0] >= 0) & (bidx[:, 0] < Bm)
    want = np.zeros((n, C, ps[0], ps[1]), np.float32)
    want[good] = native.roi_align(feat, rois[good], ps, 40 / 1280.0, 2, True)
    got = _run(feat, rois, ps, 40 / 1280.0, 2, True, nhwc)
    assert_close(got, want, rtol=1e-5, atol=2e-6, what="large launch %s nhwc=%s" % (ps, nhwc))


@pytest.mark.parametrize("nhwc", [False, True])
def test_roi_huge_footprints_take_the_exact_fallbacks(nhwc):
    """Whole-map boxes on a 150x140 map: the weight tables no longer fit next to the output tile, so the
    kernel's per-bin path runs; medium boxes on the same map use the unstaged separable path."""
    rng = np.random.default_rng(11)
    feat = rng.standard_normal((1, 40, 150, 140), dtype=np.float32)
    boxes = np.array([[0, 0, 140, 150], [3.5, 2.25, 138.0, 149.0], [10, 20, 60, 90], [100, 5, 139, 40],
                      [50, 50, 58, 57], [-20, -30, 200, 220]], dtype=np.float64)
    rois = np.concatenate([np.zeros((len(boxes), 1)), boxes], 1).astype(np.float32)
    for ps, sr in [((10, 10), 2), ((7, 7), 2), ((10, 10), -1)]:
        want = native.roi_align(feat, rois, ps, 1.0, sr, True)
        assert_close(_run(feat, rois, ps, 1.0, sr, True, nhwc), want, rtol=1e-5, atol=2e-6, what="huge %s %s" % (ps, sr))


@pytest.mark.parametrize("nhwc", [False, True])
@pytest.mark.parametrize("ps", [(10, 10), (7, 7), (5, 4)])
def test_roi_float16_storage(ps, nhwc):
    """float16 map / float16 output (tracking.py:177-178): contract = float32 sampling of the half-rounded map,
    rounded to half once, i.e. within half an ulp (2^-11 relative) of the float32 oracle on the same values."""
    rng = np.random.default_rng(21)
    feat16 = rng.standard_normal((2, 96, 40, 40)).astype(np.float16)
    boxes = np.concatenate([synth.random_boxes(rng, 40, 1280, 1280), synth.edge_case_boxes(1280, 1280)])
    boxes = boxes.astype(np.float16).astype(np.float64)              # the reference builds rois in half
    rois = np.concatenate([rng.integers(0, 2, (len(boxes), 1)).astype(np.float64), boxes], 1).astype(np.float32)
    f = torch.from_numpy(feat16).cuda()
    if nhwc:
        f = f.contiguous(memory_format=torch.channels_last)
    got = roi.roi_align(f, torch.from_numpy(rois).cuda().half(), ps, 40 / 1280.0, 2, True)
    assert got.dtype == torch.float16 and got.shape == (len(boxes), 96, ps[0], ps[1])
    want = native.roi_align(feat16.astype(np.float32), rois, ps, 40 / 1280.0, 2, True)
    assert_close(got.float().cpu().numpy(), want, rtol=1e-3, atol=2e-4, what="fp16 %s" % (ps,))


@pytest.mark.parametrize("dtype", [torch.float32, torch.float16])
@pytest.mark.parametrize("in_cl", [False, True])
def test_roi_channels_last_output_equals_nchw_output(in_cl, dtype):
    """out_channels_last=True (ROI -> encoder hand-off): same values, element for element, as the NCHW result, for
    the tiled sizes (10x10, 7x7), a generic size, small and large launches, ragged channel counts, edge boxes,
    huge footprints and bad batch indices; the returned tensor is a channels_last [K,C,PH,PW] view."""
    rng = np.random.default_rng(31)
    for (Bm, C, Hf, Wf, n) in [(2, 70, 23, 37, 60), (3, 150, 40, 48, 3400)]:
        feat = torch.from_numpy(rng.standard_normal((Bm, C, Hf, Wf), dtype=np.float32)).cuda().to(dtype)
        if in_cl:
            feat = feat.contiguous(memory_format=torch.channels_last)
        boxes = synth.random_boxes(rng, n, 32 * Hf, 32 * Wf)
        edge = synth.edge_case_boxes(32 * Hf, 32 * Wf)
        boxes[:len(edge)] = edge
        boxes[len(edge):len(edge) + 4] = [[0, 0, 32 * Wf, 32 * Hf]] * 4
        bidx = rng.integers(0, Bm, (n, 1)).astype(np.float64)
        bidx[-3:] = [[-1], [Bm], [9]]
        rois = torch.from_numpy(np.concatenate([bidx, boxes], 1).astype(np.float32)).cuda()
        for ps, sr in [((10, 10), 2), ((7, 7), 2), ((5, 4), -1)]:
            a = roi.roi_align(feat, rois, ps, 1 / 32.0, sr, True)
            b = roi.roi_align(feat, rois, ps, 1 / 32.0, sr, True, out_channels_last=True)
            assert b.shape == a.shape and b.is_contiguous(memory_format=torch.channels_last)
            assert torch.equal(a, b.contiguous()), (Bm, C, ps, in_cl, dtype)


def test_roi_device_boxes_hand_off():
    """roi_align_from_input_boxes with the detector's [N,6] output still on the device == the list form."""
    rng = np.random.default_rng(9)
    feat = torch.from_numpy(synth.feature_map(2, 1, 64, 40, 40)).cuda()
    boxes = synth.random_boxes(rng, 20, 1280, 1280)
    det = torch.from_numpy(np.concatenate([boxes, rng.random((20, 2))], 1).astype(np.float32)).cuda()
    a = roi.roi_align_from_input_boxes(feat, boxes.astype(np.float32).tolist(), (1280, 1280), out_size=(10, 10))
    b = roi.roi_align_from_input_boxes(feat, det, (1280, 1280), out_size=(10, 10))
    c = roi.roi_align_from_input_boxes(feat.contiguous(memory_format=torch.channels_last), det, (1280, 1280),
                                       out_size=(10, 10), out_channels_last=True)
    assert torch.equal(a, b) and torch.allclose(a, c.contiguous(), rtol=1e-6, atol=1e-6)


@pytest.mark.parametrize("out_cl", [False, True])
@pytest.mark.parametrize("nhwc", [False, True])
def test_roi_float16_large_launch_vs_oracle(nhwc, out_cl):
    """Half storage at launch sizes that take the prep + multi-tile (NCHW) / pipelined (channels-last) kernels:
    float32 sampling of the half-rounded map, one rounding at the end (within half an ulp of the float32 oracle).
    C = 136 gives four full channel tiles and a ragged one."""
    rng = np.random.default_rng(23)
    Bm, C, Hf, Wf, n = 2, 136, 40, 48, 3400
    feat16 = rng.standard_normal((Bm, C, Hf, Wf)).astype(np.float16)
    boxes = synth.random_boxes(rng, n, 1280, 1536)
    edge = synth.edge_case_boxes(1280, 1536)
    boxes[:len(edge)] = edge
    boxes[100:104] = [[0, 0, 1536, 1280]] * 4
    boxes = boxes.astype(np.float16).astype(np.float64)
    rois = np.concatenate([rng.integers(0, Bm, (n, 1)).astype(np.float64), boxes], 1).astype(np.float32)
    f = torch.from_numpy(feat16).cuda()
    if nhwc:
        f = f.contiguous(memory_format=torch.channels_last)
    got = roi.roi_align(f, torch.from_numpy(rois).cuda(), (10, 10), 40 / 1280.0, 2, True, out_channels_last=out_cl)
    assert got.dtype == torch.float16
    want = native.roi_align(feat16.astype(np.float32), rois, (10, 10), 40 / 1280.0, 2, True)
    assert_close(got.contiguous().float().cpu().numpy(), want, rtol=1e-3, atol=2e-4, what="fp16 large nhwc=%s cl=%s" % (nhwc, out_cl))
