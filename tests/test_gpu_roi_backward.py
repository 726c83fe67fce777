"""GPU: the ROI Align backward kernels (b200_roi_align_bwd_ex through roi_align_backward) against the double-accumulating
oracle with the bound |g - ref| <= 1e-5 * sum|contrib| + 1e-6 per cell, and roi_align's autograd path."""
import warnings

import numpy as np
import pytest
import torch

from roi_backward_oracle import assert_grad_close, roi_align_backward as oracle_bwd

pytestmark = pytest.mark.gpu

import alufe_b200  # noqa: E402,F401
from alufe_b200 import roi, synth  # noqa: E402


def _bad_rows(rois, B):
    """Appends a NaN box and ROIs with a batch index outside [0, B)."""
    extra = np.array([[0, np.nan, 10, 40, 40], [B, 0, 0, 64, 64], [-1, 0, 0, 64, 64]], np.float32)
    return np.concatenate([rois, extra]).astype(np.float32)


def _gpu_grad(g, rois, shape, ps, scale, sr, al, nhwc=False, go_cl=False, dtype=torch.float32):
    gt = torch.from_numpy(g).cuda()
    if go_cl:
        gt = gt.contiguous(memory_format=torch.channels_last)
    mf = torch.channels_last if nhwc else torch.contiguous_format
    out = roi.roi_align_backward(gt, torch.from_numpy(rois).cuda(), shape, ps, scale, sr, al, dtype=dtype,
                                 memory_format=mf)
    assert out.is_contiguous(memory_format=mf) and out.dtype == dtype
    torch.cuda.synchronize()
    return out.float().cpu().numpy()


def _named(cfg, C, seed=3):
    Hf, Wf, H_in, W_in, n = synth.CONFIGS[cfg]
    rng = np.random.default_rng(seed)
    boxes = np.concatenate([synth.random_boxes(rng, n, H_in, W_in), synth.edge_case_boxes(H_in, W_in)])
    rois = _bad_rows(np.concatenate([np.zeros((len(boxes), 1)), boxes], 1).astype(np.float32), 1)
    return (1, C, Hf, Wf), rois, Hf / float(H_in)


def _grouped(maps, per_map, C, Hf=40, Wf=40, H_in=1280, W_in=1280, seed=0):
    """bench-style launch: `maps` maps with `per_map` boxes each, plus edge cases (whole-map = unstaged footprints)."""
    rng = np.random.default_rng(seed)
    boxes = np.concatenate([synth.random_boxes(rng, per_map, H_in, W_in) for _ in range(maps)])
    idx = np.repeat(np.arange(maps), per_map)[:, None].astype(np.float64)
    edge = synth.edge_case_boxes(H_in, W_in)
    rois = np.concatenate([np.concatenate([idx, boxes], 1),
                           np.concatenate([rng.integers(0, maps, (len(edge), 1)), edge], 1)]).astype(np.float32)
    return (maps, C, Hf, Wf), _bad_rows(rois, maps), Hf / float(H_in)


def _g(rois, C, ps, seed=1):
    return np.random.default_rng(seed).standard_normal((len(rois), C) + tuple(ps)).astype(np.float32)


@pytest.mark.parametrize("go_cl", [False, True], ids=["go_nchw", "go_cl"])
@pytest.mark.parametrize("nhwc", [False, True], ids=["nchw", "nhwc"])
@pytest.mark.parametrize("ps", [(10, 10), (7, 7)])
@pytest.mark.parametrize("cfg", ["c1", "c2", "c5"])
def test_bwd_fused_named_shapes(cfg, ps, nhwc, go_cl):
    shape, rois, scale = _named(cfg, 512 if cfg != "c5" else 96)
    g = _g(rois, shape[1], ps)
    got = _gpu_grad(g, rois, shape, ps, scale, 2, True, nhwc, go_cl)
    assert_grad_close(got, g, rois, shape, ps, scale, 2, True, what="%s %s nhwc=%s go_cl=%s" % (cfg, ps, nhwc, go_cl))


@pytest.mark.parametrize("go_cl", [False, True], ids=["go_nchw", "go_cl"])
@pytest.mark.parametrize("nhwc", [False, True], ids=["nchw", "nhwc"])
@pytest.mark.parametrize("ps", [(10, 10), (7, 7)])
@pytest.mark.parametrize("launch", ["g64", "c3"])
def test_bwd_large_launches(launch, ps, nhwc, go_cl):
    """Prep + TMA reduce (NCHW grad_in) / prep + tile kernel (channels-last grad_in); 128 channels keep the oracle fast
    while staying above the prep kernel's launch threshold."""
    shape, rois, scale = _grouped(64, 64, 128) if launch == "g64" else _grouped(256, 16, 128, seed=4)
    g = _g(rois, shape[1], ps)
    got = _gpu_grad(g, rois, shape, ps, scale, 2, True, nhwc, go_cl)
    assert_grad_close(got, g, rois, shape, ps, scale, 2, True, what="%s %s nhwc=%s go_cl=%s" % (launch, ps, nhwc, go_cl))


@pytest.mark.parametrize("nhwc", [False, True], ids=["nchw", "nhwc"])
@pytest.mark.parametrize("ps, sr, al", [((10, 10), -1, True), ((7, 7), 2, False), ((10, 10), 0, False),
                                        ((7, 7), 3, True), ((5, 4), 2, True), ((5, 4), -1, False)])
@pytest.mark.parametrize("C, W", [(100, 40), (128, 37)], ids=["C100", "W37"])
def test_bwd_odd_shapes_and_parameters(C, W, ps, sr, al, nhwc):
    """C not a multiple of 32, W not a multiple of 4 (no TMA), adaptive sampling, aligned=False, an output size without a
    tile kernel -- on launches large enough for the prep path."""
    shape, rois, scale = _grouped(64, 64, C, Wf=W)
    g = _g(rois, C, ps, seed=5)
    got = _gpu_grad(g, rois, shape, ps, scale, sr, al, nhwc)
    assert_grad_close(got, g, rois, shape, ps, scale, sr, al, what="C=%d W=%d %s sr=%d al=%s" % (C, W, ps, sr, al))


@pytest.mark.parametrize("nhwc", [False, True], ids=["nchw", "nhwc"])
@pytest.mark.parametrize("launch", ["c2", "g64"])
def test_bwd_half_grad_output(launch, nhwc):
    ps = (10, 10)
    shape, rois, scale = _named("c2", 512) if launch == "c2" else _grouped(64, 64, 128)
    g = _g(rois, shape[1], ps).astype(np.float16).astype(np.float32)       # half-rounded grad_output
    gh = torch.from_numpy(g).cuda().half()
    r = torch.from_numpy(rois).cuda()
    mf = torch.channels_last if nhwc else torch.contiguous_format
    f32 = roi.roi_align_backward(gh, r, shape, ps, scale, 2, True, memory_format=mf).cpu().numpy()
    ref, mag = assert_grad_close(f32, g, rois, shape, ps, scale, 2, True, what="half grad_output, float32 result")
    h = roi.roi_align_backward(gh, r, shape, ps, scale, 2, True, dtype=torch.float16, memory_format=mf)
    assert h.dtype == torch.float16 and h.is_contiguous(memory_format=mf)
    h = h.cpu().numpy().astype(np.float64)
    ulp = np.spacing(np.abs(ref).astype(np.float16)).astype(np.float64)
    assert np.all(np.abs(h - ref) <= 0.5 * ulp + 1e-5 * mag + 1e-6)


def test_bwd_adjoint_identity_g64():
    shape, rois, scale = _grouped(64, 64, 512)
    ps = (10, 10)
    x = torch.randn(shape, device="cuda", generator=torch.Generator("cuda").manual_seed(0))
    r = torch.from_numpy(rois).cuda()
    g = torch.randn((len(rois), shape[1]) + ps, device="cuda", generator=torch.Generator("cuda").manual_seed(1))
    lhs = (roi.roi_align(x, r, ps, scale, 2, True).double() * g.double()).sum().item()
    gx = roi.roi_align_backward(g, r, shape, ps, scale, 2, True)
    rhs = (x.double() * gx.double()).sum().item()
    # every bilinear weight is >= 0, so backward(|g|) is sum|contrib| per cell: <|x|, backward(|g|)> bounds both sides' sums
    bound = (x.double().abs() * roi.roi_align_backward(g.abs(), r, shape, ps, scale, 2, True).double()).sum().item()
    assert abs(lhs - rhs) <= 1e-5 * bound, (lhs, rhs, bound)


@pytest.mark.parametrize("launch", ["c2", "g64"])
def test_bwd_vs_torchvision_cuda(launch):
    torchvision = pytest.importorskip("torchvision")  # noqa: F841
    ps = (10, 10)
    shape, rois, scale = _named("c2", 512) if launch == "c2" else _grouped(64, 64, 128)
    rois = rois[np.isfinite(rois).all(1) & (rois[:, 0] >= 0) & (rois[:, 0] < shape[0])]   # torchvision: valid rows only
    g = torch.from_numpy(_g(rois, shape[1], ps)).cuda()
    r = torch.from_numpy(rois).cuda()
    B, C, H, W = shape
    tv = torch.ops.torchvision._roi_align_backward(g, r, scale, ps[0], ps[1], B, C, H, W, 2, True).cpu().numpy()
    got = roi.roi_align_backward(g, r, shape, ps, scale, 2, True).cpu().numpy()
    _, mag = oracle_bwd(g.cpu().numpy(), rois, shape, ps, scale, 2, True, with_magnitude=True)
    assert np.all(np.abs(got - tv) <= 1e-4 * mag + 1e-5)


@pytest.mark.parametrize("nhwc", [False, True], ids=["nchw", "nhwc"])
@pytest.mark.parametrize("launch", ["c2", "g64"])
def test_autograd_roi_align(launch, nhwc):
    ps = (10, 10)
    shape, rois, scale = _named("c2", 512) if launch == "c2" else _grouped(64, 64, 128)
    x0 = torch.from_numpy(synth.feature_map(2, *shape)).cuda()
    if nhwc:
        x0 = x0.contiguous(memory_format=torch.channels_last)
    r = torch.from_numpy(rois).cuda()
    plain = roi.roi_align(x0, r, ps, scale, 2, True)
    x = x0.clone().requires_grad_()
    out = roi.roi_align(x, r, ps, scale, 2, True)
    assert out.grad_fn is not None
    assert torch.equal(out.detach(), plain)                    # the forward values do not depend on grad mode
    g = _g(rois, shape[1], ps, seed=7)
    out.backward(torch.from_numpy(g).cuda())
    mf = torch.channels_last if nhwc else torch.contiguous_format
    assert x.grad.dtype == x.dtype and x.grad.is_contiguous(memory_format=mf)
    assert_grad_close(x.grad.cpu().numpy(), g, rois, shape, ps, scale, 2, True, what="autograd")
    with torch.no_grad():
        assert roi.roi_align(x, r, ps, scale, 2, True).grad_fn is None


def test_autograd_half_map():
    shape, rois, scale = _named("c2", 64)
    x = torch.from_numpy(synth.feature_map(2, *shape)).cuda().half().requires_grad_()
    out = roi.roi_align(x, torch.from_numpy(rois).cuda(), (10, 10), scale, 2, True)
    g = _g(rois, shape[1], (10, 10)).astype(np.float16)
    out.backward(torch.from_numpy(g).cuda())
    assert x.grad.dtype == torch.float16
    ref, mag = oracle_bwd(g.astype(np.float32), rois, shape, (10, 10), scale, 2, True, with_magnitude=True)
    ulp = np.spacing(np.abs(ref).astype(np.float16)).astype(np.float64)
    assert np.all(np.abs(x.grad.cpu().numpy().astype(np.float64) - ref) <= 0.5 * ulp + 1e-5 * mag + 1e-6)


def test_autograd_wrappers_with_device_boxes():
    Hf, Wf, H_in, W_in, n = synth.CONFIGS["c2"]
    rng = np.random.default_rng(9)
    boxes = synth.random_boxes(rng, n, H_in, W_in).astype(np.float32)
    feat = torch.from_numpy(synth.feature_map(4, 1, 64, Hf, Wf)).cuda().requires_grad_()
    db = torch.from_numpy(boxes).cuda()
    out = roi.roi_align_from_input_boxes(feat, db, (H_in, W_in), out_size=(7, 7))
    g = _g(boxes, 64, (7, 7))
    out.backward(torch.from_numpy(g).cuda())
    rois = np.concatenate([np.zeros((n, 1), np.float32), boxes], 1)
    assert_grad_close(feat.grad.cpu().numpy(), g, rois, (1, 64, Hf, Wf), (7, 7), Hf / float(H_in), 2, True,
                      what="roi_align_from_input_boxes")

    feat.grad = None
    out = roi.preprocess_roi(feat, db, (H_in, W_in))
    g = _g(boxes, 64, (10, 10), seed=3)
    out.backward(torch.from_numpy(g).cuda())
    rois = roi._prep_boxes(db, feat.device, alufe_b200._lib.BOXES_TRAINING, None, (H_in, W_in), (Hf, Wf), 1.0)
    assert_grad_close(feat.grad.cpu().numpy(), g, rois.cpu().numpy(), (1, 64, Hf, Wf), (10, 10), 1.0, 2, True,
                      what="preprocess_roi")


def test_autograd_deterministic_mode_and_double_backward():
    shape, rois, scale = _named("c1", 32)
    x = torch.from_numpy(synth.feature_map(2, *shape)).cuda().requires_grad_()
    r = torch.from_numpy(rois).cuda()
    old, old_warn = torch.are_deterministic_algorithms_enabled(), torch.is_deterministic_algorithms_warn_only_enabled()
    try:
        torch.use_deterministic_algorithms(True)
        with pytest.raises(RuntimeError, match="deterministic"):
            roi.roi_align(x, r, (7, 7), scale, 2, True).sum().backward()
        torch.use_deterministic_algorithms(True, warn_only=True)
        with warnings.catch_warnings(record=True) as w:
            warnings.simplefilter("always")
            roi.roi_align(x, r, (7, 7), scale, 2, True).sum().backward()
        assert any("deterministic" in str(m.message) for m in w)
    finally:
        torch.use_deterministic_algorithms(old, warn_only=old_warn)
    out = roi.roi_align(x, r, (7, 7), scale, 2, True)
    (gx,) = torch.autograd.grad(out.square().sum(), x, create_graph=True)
    with pytest.raises(RuntimeError):
        gx.sum().backward()


@pytest.mark.parametrize("launch", ["c2", "g64"])
def test_bwd_replays_as_cuda_graph(launch):
    ps = (10, 10)
    shape, rois, scale = _named("c2", 512) if launch == "c2" else _grouped(64, 64, 128)
    r = torch.from_numpy(rois).cuda()
    g = torch.zeros((len(rois), shape[1]) + ps, device="cuda")
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        for _ in range(2):
            roi.roi_align_backward(g, r, shape, ps, scale, 2, True)
    torch.cuda.current_stream().wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        out = roi.roi_align_backward(g, r, shape, ps, scale, 2, True)
    for seed in (1, 2):
        gn = _g(rois, shape[1], ps, seed=seed)
        g.copy_(torch.from_numpy(gn))
        graph.replay()
        torch.cuda.synchronize()
        assert_grad_close(out.cpu().numpy(), gn, rois, shape, ps, scale, 2, True, what="graph replay %d" % seed)

