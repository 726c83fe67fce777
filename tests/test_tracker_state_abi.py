"""CPU: argument errors of b200_tracker_export_device / b200_tracker_import_device that need no device (the image's own
checks and the null handle; the checks against a live handle are in test_gpu_tracker_state.py)."""
import ctypes

import pytest

from alufe_b200 import _lib

ENTRY_POINTS = ["b200_tracker_export_device", "b200_tracker_import_device"]


def _image(n_rows=1, cap=4, hist_max=30):
    im = _lib.tracker_state()
    for n, _, _ in _lib.STATE_LAYOUT:
        setattr(im, n, 256)                 # never dereferenced: every failing check is made on the host
    im.n_rows, im.cap, im.hist_max = n_rows, cap, hist_max
    return im


def _call(fn, handle, im):
    lib = _lib.lib()
    rc = getattr(lib, fn)(handle, None, ctypes.byref(im) if im is not None else None, None, None)
    return rc, lib.b200_last_error()


@pytest.mark.parametrize("fn", ENTRY_POINTS)
def test_null_handle(fn):
    rc, msg = _call(fn, None, _image())
    assert rc == _lib.EINVAL and b"null handle" in msg and fn[5:].encode() in msg


@pytest.mark.parametrize("fn", ENTRY_POINTS)
def test_null_image(fn):
    rc, msg = _call(fn, ctypes.c_void_p(16), None)
    assert rc == _lib.EINVAL and b"null image" in msg


@pytest.mark.parametrize("fn", ENTRY_POINTS)
def test_bad_image_shape(fn):
    rc, msg = _call(fn, ctypes.c_void_p(16), _image(cap=0))
    assert rc == _lib.EINVAL and b"cap 0" in msg
    rc, msg = _call(fn, ctypes.c_void_p(16), _image(n_rows=-1))
    assert rc == _lib.EINVAL and b"n_rows -1" in msg


@pytest.mark.parametrize("fn", ENTRY_POINTS)
def test_image_fields(fn):
    im = _image()
    im.bank = None
    rc, msg = _call(fn, ctypes.c_void_p(16), im)
    assert rc == _lib.EINVAL and b"null image field" in msg
    im = _image()
    im.P = 264                              # 8-byte aligned only
    rc, msg = _call(fn, ctypes.c_void_p(16), im)
    assert rc == _lib.EINVAL and b"16-byte aligned" in msg


def test_struct_matches_the_header():
    """Every field of b200_tracker_state, in order, as include/b200track.h declares it."""
    import os
    import re
    from conftest import ROOT
    text = open(os.path.join(ROOT, "include", "b200track.h")).read()
    body = re.search(r"typedef struct b200_tracker_state \{(.*?)\} b200_tracker_state;", text, flags=re.S).group(1)
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    names = re.findall(r"\*\s*(\w+)\s*;", body) + list(re.findall(r"int32_t\s+(n_rows),\s*(cap),\s*(hist_max);", body)[0])
    assert [n for n, _ in _lib.tracker_state._fields_] == list(names)
    assert ctypes.sizeof(_lib.tracker_state) == 14 * 8 + 3 * 4 + 4
