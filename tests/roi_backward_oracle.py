"""Oracle (test-only) for the ROI Align backward pass: loads tests/roi_align_bwd_ref.c, built with gcc into a
temporary directory on first use (the repository tree is left untouched)."""
import ctypes
import hashlib
import os
import subprocess
import tempfile

import numpy as np

_SRC = os.path.join(os.path.dirname(os.path.abspath(__file__)), "roi_align_bwd_ref.c")
_lib = None


def lib():
    global _lib
    if _lib is None:
        tag = hashlib.sha1(open(_SRC, "rb").read()).hexdigest()[:12]
        out = os.path.join(tempfile.gettempdir(), "roi_align_bwd_ref_%d_%s.so" % (os.getuid(), tag))
        if not os.path.exists(out):
            tmp = out + ".%d" % os.getpid()
            subprocess.run(["gcc", "-O2", "-fPIC", "-shared", "-ffp-contract=off", "-o", tmp, _SRC, "-lm"], check=True)
            os.replace(tmp, out)
        _lib = ctypes.CDLL(out)
        _lib.oracle_roi_align_bwd_f32.restype = None
    return _lib


def _p(a):
    return a.ctypes.data_as(ctypes.c_void_p)


def roi_align_backward(grad_out, rois, input_shape, output_size, spatial_scale=1.0, sampling_ratio=-1, aligned=False,
                       with_magnitude=False):
    """float64 [B,C,H,W] gradient of roi_align w.r.t. its float32 input for the float32 grad_out [K,C,PH,PW]
    (NCHW).  ``with_magnitude=True`` returns (gradient, per-cell sum of the magnitudes of the contributions)."""
    g = np.ascontiguousarray(grad_out, dtype=np.float32)
    r = np.ascontiguousarray(rois, dtype=np.float32).reshape(-1, 5)
    B, C, H, W = (int(v) for v in input_shape)
    PH, PW = output_size
    assert g.shape == (r.shape[0], C, PH, PW), g.shape
    out = np.zeros((B, C, H, W), dtype=np.float64)
    mag = np.zeros_like(out) if with_magnitude else None
    lib().oracle_roi_align_bwd_f32(_p(g), B, C, H, W, _p(r), ctypes.c_int64(r.shape[0]), PH, PW,
                                   ctypes.c_float(spatial_scale), int(sampling_ratio), int(bool(aligned)), _p(out),
                                   _p(mag) if with_magnitude else None)
    return (out, mag) if with_magnitude else out


def assert_grad_close(got, grad_out, rois, input_shape, output_size, spatial_scale, sampling_ratio, aligned,
                      rel=1e-5, what=""):
    """|got - ref| <= rel * sum|contributions| + 1e-6 per cell: the bound for a float32 sum in any order."""
    ref, mag = roi_align_backward(grad_out, rois, input_shape, output_size, spatial_scale, sampling_ratio, aligned,
                                  with_magnitude=True)
    got = np.asarray(got, dtype=np.float64)
    assert got.shape == ref.shape, "%s: shape %s vs %s" % (what, got.shape, ref.shape)
    err = np.abs(got - ref)
    tol = rel * mag + 1e-6
    bad = ~(err <= tol)
    if bad.any():
        i = np.unravel_index(np.argmax(np.where(np.isnan(err), np.inf, err - tol)), got.shape)
        raise AssertionError("%s: %d/%d cells out of tolerance; worst at %s: got %r want %r (sum|contrib| %r)" %
                             (what, int(bad.sum()), got.size, i, got[i], ref[i], mag[i]))
    return ref, mag
