"""ctypes loader for libb200track.so (the C ABI of include/b200track.h).

There is no CPU fallback: every operator in this package goes through this library and
raises if it cannot be loaded or if no CUDA device is present.
"""
import ctypes
import os
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
# B200TRACK_LIB: load another build of the same library (e.g. another commit's, to compare against); unset = the product
LIB_PATH = os.environ.get("B200TRACK_LIB") or os.path.join(_HERE, "libb200track.so")
CSRC = os.path.join(_HERE, "csrc")

OK, EINVAL, ECUDA, ECAPACITY, ENUMERIC, EINFEASIBLE = 0, -1, -2, -3, -4, -5
LAYOUT_NCHW, LAYOUT_NHWC = 0, 1
DTYPE_F32, DTYPE_F16 = 0, 1
BOXES_INPUT, BOXES_TRAINING = 0, 1

_lib = None


class B200Error(RuntimeError):
    pass


def build(force=False, verbose=False):
    """Compiles csrc/*.cu for sm_100a into libb200track.so (nvcc cross-compiles without a GPU)."""
    cmd = ["make", "-C", CSRC, "-j8"] + (["-B"] if force else [])
    res = subprocess.run(cmd, capture_output=not verbose, text=True)
    if res.returncode != 0:
        raise B200Error("building libb200track.so failed:\n%s\n%s" % (res.stdout, res.stderr))
    return LIB_PATH


class tracker_conf(ctypes.Structure):
    _fields_ = [(n, ctypes.c_double) for n in (
        "init_conf_min", "w_app", "w_bbox", "w_conf", "alpha", "beta", "cost_max", "ema_alpha",
        "conf_update_min", "cost_update_max", "maha_thr", "reid_only_cost_max")] + [
        (n, ctypes.c_int32) for n in ("hist_max", "emb_top_k", "max_age", "lost_reid_after")]


_P, _I, _L, _F, _D = ctypes.c_void_p, ctypes.c_int, ctypes.c_int64, ctypes.c_float, ctypes.c_double

# b200_tracker_state: (field, element type, shape after the row dimension; "cap" / "hist_max" are the image's), in the
# struct's order.  n_live and next_id are [n_rows]; every other field is [n_rows, cap, ...].
STATE_LAYOUT = (
    ("n_live", "int32", ()), ("next_id", "int32", ()), ("ids", "int32", ("cap",)), ("x", "float64", ("cap", 8)),
    ("P", "float64", ("cap", 8, 8)), ("stage", "uint8", ("cap",)), ("ema", "float32", ("cap", 128)),
    ("bank", "float32", ("cap", "hist_max", 128)), ("bank_len", "int32", ("cap",)), ("miss", "int32", ("cap",)),
    ("age", "int32", ("cap",)), ("last_bbox", "float64", ("cap", 4)), ("last_conf", "float64", ("cap",)),
    ("last_cost", "float64", ("cap",)))


class tracker_state(ctypes.Structure):
    _fields_ = [(n, _P) for n, _, _ in STATE_LAYOUT] + [(n, ctypes.c_int32) for n in ("n_rows", "cap", "hist_max")]

SIGNATURES = {
    "b200_version": (ctypes.c_int, []),
    "b200_last_error": (ctypes.c_char_p, []),
    "b200_launch_count": (ctypes.c_int64, []),
    "b200_roi_align_fwd_f32": (_I, [_P, _I, _I, _I, _I, _I, _P, _L, _I, _I, _F, _I, _I, _P, _P]),
    "b200_roi_align_fwd_f16": (_I, [_P, _I, _I, _I, _I, _I, _P, _L, _I, _I, _F, _I, _I, _P, _P]),
    "b200_roi_align_fwd_ex": (_I, [_P, _I, _I, _I, _I, _I, _I, _P, _L, _I, _I, _F, _I, _I, _P, _I, _P]),
    "b200_roi_align_bwd_ex": (_I, [_P, _I, _I, _P, _L, _I, _I, _F, _I, _I, _P, _I, _I, _I, _I, _I, _P]),
    "b200_roi_boxes_prep_f32": (_I, [_P, _L, _I, _P, _I, _I, _I, _I, _I, _F, _P, _P]),
    "b200_app_cost_topk_f32": (_I, [_P, _P, _P, _P, _I, _I, _I, _I, _I, _P, _I, _P]),
    "b200_pair_cost_f32": (_I, [_P, _P, _P, _P, _P, _I, _I, _F, _F, _F, _F, _F, _F, _P, _P, _P, _P, _P, _I, _P]),
    "b200_kalman_init": (_I, [_P, _I, _P, _P, _P, _P]),
    "b200_kalman_predict": (_I, [_P, _P, _P, _I, _P, _P, _P]),
    "b200_kalman_update": (_I, [_P, _P, _P, _I, _P, _P, _I, _P, _P]),
    "b200_maha_gate": (_I, [_P, _P, _P, _I, _P, _I, _P, _D, _F, _P, _I, _P, _I, _P]),
    "b200_lsap_f32": (_I, [_P, _I, _L, _I, _I, _I, _D, _P, _P, _P, _P]),
    "b200_tracker_create": (_I, [ctypes.POINTER(_P), _I, _I, _I, ctypes.POINTER(tracker_conf)]),
    "b200_tracker_destroy": (None, [_P]),
    "b200_tracker_reset": (_I, [_P, _P]),
    "b200_tracker_result_stride": (_I, [_P]),
    "b200_tracker_live_counts": (_I, [_P, _P, _P, _P]),
    "b200_tracker_step": (_I, [_P, _P, _P, _P, _P, _P, _P, _P]),
    "b200_tracker_step_packed": (_I, [_P, _L, _P, _I, _P, _I, _I, _P, _I, _P, _P, _P, _P, _P, _P]),
    "b200_tracker_step_host": (_I, [_P, _P, _P, _P, _P, _P, _P, _P]),
    "b200_tracker_step_host_async": (_I, [_P, _P, _P, _P, _P, _P, ctypes.POINTER(ctypes.c_int64), _P]),
    "b200_tracker_step_pinned_async": (_I, [_P, _P, _P, _P, _P, _P, ctypes.POINTER(ctypes.c_int64), _P]),
    "b200_tracker_step_result": (_I, [_P, ctypes.c_int64, _P]),
    "b200_tracker_predict_all": (_I, [_P, _I, _P]),
    "b200_tracker_mark_missed": (_I, [_P, _I, _P, _I, _P]),
    "b200_tracker_purge_dead": (_I, [_P, _I, _P]),
    "b200_tracker_create_tracks": (_I, [_P, _I, _P, _I, _P, _P, _P, _I, _I, _P]),
    "b200_tracker_update_matched": (_I, [_P, _I, _P, _P, _P, _I, _P, _P, _P, _I, _I, _D, _D, _D, _D, _P]),
    "b200_peer_gather_create": (_I, [ctypes.POINTER(_P), _I, _I, _L, _I]),
    "b200_peer_gather_handle": (_I, [_P, _P]),
    "b200_peer_gather_connect": (_I, [_P, _P]),
    "b200_peer_gather_push": (_I, [_P, _P, _L, _L, _P]),
    "b200_peer_gather_collect": (_I, [_P, _P, _L, _L, _P]),
    "b200_peer_gather_destroy": (None, [_P]),
    "b200_tracker_export": (_I, [_P, _I] + [_P] * 14),
    "b200_tracker_import": (_I, [_P, _I, _I] + [_P] * 12 + [_I, _P]),
    "b200_tracker_export_device": (_I, [_P, _P, ctypes.POINTER(tracker_state), _P, _P]),
    "b200_tracker_import_device": (_I, [_P, _P, ctypes.POINTER(tracker_state), _P, _P]),
}


def lib():
    """Returns the loaded library; raises B200Error when it is missing (no fallback)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise B200Error(
                "%s not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(or `make -C %s`). This package has no CPU fallback." % (LIB_PATH, CSRC))
        h = ctypes.CDLL(LIB_PATH)
        missing = [n for n in SIGNATURES if not hasattr(h, n)]
        if missing:
            raise B200Error("%s does not export %s: rebuild it" % (LIB_PATH, ", ".join(missing)))
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(h, name)
            fn.restype, fn.argtypes = res, args
        _lib = h
    return _lib


def check(rc, exc_map=None):
    if rc == OK:
        return
    msg = lib().b200_last_error().decode("utf-8", "replace")
    exc = (exc_map or {}).get(rc)
    if exc is not None:
        raise exc(msg)
    if rc == EINVAL:
        raise ValueError(msg)
    raise B200Error("libb200track error %d: %s" % (rc, msg))


def require_cuda(t, name):
    if not t.is_cuda:
        raise B200Error("%s must be a CUDA tensor: this package has no CPU path" % name)


def stream_ptr(device=None):
    import torch
    return ctypes.c_void_p(torch.cuda.current_stream(device).cuda_stream)


def ptr(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else None
