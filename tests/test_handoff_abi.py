"""CPU: argument errors of b200_tracker_step_packed that need no device."""
import ctypes

from alufe_b200 import _lib


def test_step_packed_null_handle():
    lib = _lib.lib()
    p = ctypes.c_void_p(16)                  # never dereferenced: the handle is checked first
    rc = lib.b200_tracker_step_packed(None, 1, p, 6, p, 6, _lib.DTYPE_F32, p, _lib.DTYPE_F32, None, None, p, p, None, None)
    assert rc == _lib.EINVAL
    assert b"tracker_step_packed" in lib.b200_last_error() and b"null handle" in lib.b200_last_error()
