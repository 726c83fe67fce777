import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

GOLDEN = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")


def load_golden(name):
    return np.load(os.path.join(GOLDEN, name + ".npz"))


def load_roi_wrappers_golden():
    """roi_wrappers.npz keeps a preprocess_roi output only for the ROIs where it differs from the
    roi_align_from_input_boxes output named by ``<key>_base`` (``<key>_rows`` lists those ROIs; every other row
    is equal bit for bit), so that the fixture stays small.  Returns every output in full."""
    g = dict(load_golden("roi_wrappers"))
    for key in [k[:-len("_rows")] for k in g if k.endswith("_rows")]:
        full = g[str(g.pop(key + "_base"))].copy()
        full[g.pop(key + "_rows")] = g[key]
        g[key] = full
    return g


def assert_close(a, b, rtol=1e-5, atol=1e-6, what=""):
    """The parity bar of BASELINE.json north_star: 1e-5 relative in fp32, with an absolute
    floor for outputs near zero (SURVEY.md section 7, hard parts)."""
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    assert a.shape == b.shape, "%s shape %s vs %s" % (what, a.shape, b.shape)
    if a.size == 0:
        return
    err = np.abs(a - b)
    tol = atol + rtol * np.abs(b)
    bad = err > tol
    if bad.any():
        i = np.unravel_index(np.argmax(err - tol), a.shape)
        raise AssertionError("%s: %d/%d out of tolerance; worst at %s: got %r want %r" %
                             (what, int(bad.sum()), a.size, i, a[i], b[i]))
