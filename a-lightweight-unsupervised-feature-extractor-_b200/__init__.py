"""B200-native tracker hot path: ROI Align + association step (cost, gate, Kalman, assignment).

Every operator calls hand-written sm_100a kernels through ``libb200track.so`` (C ABI in
``include/b200track.h``).  There is no CPU fallback: importing is cheap, but using any operator
without the built library or without a CUDA device raises.

Reference surface mirrored here (SURVEY.md section 8b):
    roi_align, roi_align_from_input_boxes, preprocess_roi            (roi.py)
    roi_align_backward (the gradient of roi_align; roi_align is differentiable)
    bbox_cost, conf_cost, cal_cost, app_cost_topk                    (cost.py)
    bbox_xyxy_to_z, x_to_bbox_xyxy, init_kf_from_bbox,
    gating_distance_maha, BatchedKalman                              (kalman.py)
    hungarian_assign, lsap_batched                                   (hung.py)
    Tracking, MultiStreamTracker                                     (tracking.py)
"""
from . import _lib  # noqa: F401
from .roi import roi_align, roi_align_backward, roi_align_from_input_boxes, preprocess_roi  # noqa: F401
from .cost import bbox_cost, conf_cost, cal_cost, app_cost_topk  # noqa: F401
from .kalman import (bbox_xyxy_to_z, x_to_bbox_xyxy, init_kf_from_bbox, gating_distance_maha,  # noqa: F401
                     BatchedKalman, KalmanState)
from .hung import hungarian_assign, lsap_batched  # noqa: F401
from .tracking import Tracking, MultiStreamTracker, SHIPPED_CONF, CODE_DEFAULTS, load_conf  # noqa: F401

__all__ = ["roi_align", "roi_align_backward", "roi_align_from_input_boxes", "preprocess_roi", "bbox_cost", "conf_cost", "cal_cost",
           "app_cost_topk", "bbox_xyxy_to_z", "x_to_bbox_xyxy", "init_kf_from_bbox", "gating_distance_maha",
           "BatchedKalman", "KalmanState", "hungarian_assign", "lsap_batched", "Tracking", "MultiStreamTracker",
           "SHIPPED_CONF", "CODE_DEFAULTS", "load_conf"]
