"""CPU: the ROI Align backward oracle against torchvision's CPU _roi_align_backward, the adjoint identity
<roi_align(x), g> = <x, roi_align_backward(g)>, and the argument checks of b200_roi_align_bwd_ex."""
import ctypes

import numpy as np
import pytest
import torch

from conftest import ROOT  # noqa: F401  (puts the repository on sys.path)
from oracle import native
from roi_backward_oracle import roi_align_backward as oracle_bwd

import alufe_b200  # noqa: E402,F401
from alufe_b200 import _lib, synth  # noqa: E402

torchvision = pytest.importorskip("torchvision")


def _cases():
    rng = np.random.default_rng(11)
    Hf, Wf, H_in, W_in, n = synth.CONFIGS["c1"]
    boxes = np.concatenate([synth.random_boxes(rng, n, H_in, W_in), synth.edge_case_boxes(H_in, W_in)])
    rois = np.concatenate([np.zeros((len(boxes), 1)), boxes], 1).astype(np.float32)
    yield "c1 edge cases", (1, 6, Hf, Wf), rois, (10, 10), Hf / float(H_in), 2, True
    yield "c1 7x7 not aligned", (1, 6, Hf, Wf), rois, (7, 7), Hf / float(H_in), 2, False
    yield "c1 adaptive", (1, 6, Hf, Wf), rois, (10, 10), Hf / float(H_in), -1, True
    b = rng.uniform(-100, 1300, (40, 4))
    b[:4] = [0, 0, 1184, 736]                           # whole-map boxes
    b[4:12, 2:] = b[4:12, :2] + rng.uniform(200, 600, (8, 2))
    rois = np.concatenate([rng.integers(0, 3, (40, 1)).astype(np.float64), b], 1).astype(np.float32)
    yield "batched adaptive not aligned", (3, 5, 23, 37), rois, (7, 7), 1 / 32.0, 0, False
    yield "batched (5,4) sr 3", (3, 5, 23, 37), rois, (5, 4), 1 / 32.0, 3, True


@pytest.mark.parametrize("case", list(_cases()), ids=lambda c: c[0])
def test_oracle_matches_torchvision_cpu(case):
    _, shape, rois, ps, scale, sr, al = case
    B, C, H, W = shape
    g = np.random.default_rng(1).standard_normal((len(rois), C) + ps).astype(np.float32)
    want = torch.ops.torchvision._roi_align_backward(torch.from_numpy(g), torch.from_numpy(rois), scale, ps[0], ps[1],
                                                     B, C, H, W, sr, al).double().numpy()
    got, mag = oracle_bwd(g, rois, shape, ps, scale, sr, al, with_magnitude=True)
    assert np.all(np.abs(got - want) <= 1e-5 * mag + 1e-6)
    assert np.all(mag >= np.abs(got) - 1e-9)
    assert mag.max() > 0


@pytest.mark.parametrize("case", list(_cases()), ids=lambda c: c[0])
def test_oracle_adjoint_identity(case):
    _, shape, rois, ps, scale, sr, al = case
    rng = np.random.default_rng(2)
    x = rng.standard_normal(shape).astype(np.float32)
    g = rng.standard_normal((len(rois), shape[1]) + ps).astype(np.float32)
    lhs = float(np.sum(native.roi_align(x, rois, ps, scale, sr, al).astype(np.float64) * g))
    gx, mag = oracle_bwd(g, rois, shape, ps, scale, sr, al, with_magnitude=True)
    rhs = float(np.sum(x.astype(np.float64) * gx))
    bound = float(np.sum(np.abs(x) * mag))
    assert abs(lhs - rhs) <= 1e-5 * bound + 1e-6


def test_oracle_skips_bad_batch_index():
    rois = np.array([[3, 0, 0, 8, 8], [-1, 0, 0, 8, 8], [np.nan, 0, 0, 8, 8]], np.float32)
    g = np.ones((3, 2, 7, 7), np.float32)
    assert not oracle_bwd(g, rois, (2, 2, 9, 9), (7, 7), 1.0, 2, True).any()


def test_bwd_entry_point_arguments_without_gpu():
    _lib.build()
    assert hasattr(ctypes.CDLL(_lib.LIB_PATH), "b200_roi_align_bwd_ex")
    lib = _lib.lib()
    rc = lib.b200_roi_align_bwd_ex(None, 0, 0, None, 0, 7, 7, 1.0, 2, 1, None, 9, 1, 1, 1, 1, None)
    assert rc == _lib.EINVAL and b"layout" in lib.b200_last_error()
    rc = lib.b200_roi_align_bwd_ex(None, 0, 5, None, 0, 7, 7, 1.0, 2, 1, None, 0, 1, 1, 1, 1, None)
    assert rc == _lib.EINVAL and b"layout" in lib.b200_last_error()
    rc = lib.b200_roi_align_bwd_ex(None, 7, 0, None, 1, 7, 7, 1.0, 2, 1, None, 0, 1, 1, 1, 1, None)
    assert rc == _lib.EINVAL and b"dtype" in lib.b200_last_error()
    rc = lib.b200_roi_align_bwd_ex(None, 0, 0, None, 1, 7, 7, 1.0, 2, 1, None, 0, 0, 1, 1, 1, None)
    assert rc == _lib.EINVAL and b"shape" in lib.b200_last_error()
    rc = lib.b200_roi_align_bwd_ex(None, 0, 0, None, 0, 10, 10, 1.0, 2, 1, None, 0, 1, 1, 1, 1, None)
    assert rc == _lib.OK                      # K == 0 is a no-op
    assert lib.b200_version() == 100


def test_backward_has_no_cpu_fallback():
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    with pytest.raises(_lib.B200Error):
        alufe_b200.roi_align_backward(torch.zeros(1, 4, 2, 2), torch.zeros(1, 5), (1, 4, 5, 5), (2, 2))
