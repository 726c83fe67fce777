"""ROI Align operators with the reference's Python surface, backed by libb200track.

* ``roi_align``                  - torchvision.ops.roi_align signature (tracking.py:203,214).
* ``roi_align_from_input_boxes`` - MainInfer.roi_align_from_input_boxes, tracking.py:193-221
                                   (= tracking_win.py:239-267, infer.py:143-170).
* ``preprocess_roi``             - PreProcess._preprocess_roi, trainingCard.py:24-79.
"""
import warnings
from typing import Sequence, Tuple, Union

import numpy as np
import torch
from torch.autograd.function import once_differentiable

from . import _lib


def _pair(v):
    return (int(v), int(v)) if isinstance(v, int) else (int(v[0]), int(v[1]))


def _boxes_to_rois(boxes, device):
    if isinstance(boxes, (list, tuple)):
        parts = []
        for i, b in enumerate(boxes):
            if b.dim() != 2 or b.size(1) != 4:
                raise ValueError("each element of the box list must be Tensor[L, 4]")
            idx = torch.full((b.size(0), 1), float(i), dtype=torch.float32, device=b.device)
            parts.append(torch.cat([idx, b.to(torch.float32)], dim=1))
        rois = torch.cat(parts, dim=0) if parts else torch.zeros((0, 5), dtype=torch.float32)
    else:
        if boxes.dim() != 2 or boxes.size(1) != 5:
            raise ValueError("boxes must be Tensor[K, 5] (batch index in column 0) or a list of Tensor[L, 4]")
        rois = boxes
    return rois.to(device=device, dtype=torch.float32).contiguous()


def roi_align(input: torch.Tensor, boxes: Union[torch.Tensor, Sequence[torch.Tensor]],
              output_size: Union[int, Tuple[int, int]], spatial_scale: float = 1.0,
              sampling_ratio: int = -1, aligned: bool = False, *, out_channels_last: bool = False) -> torch.Tensor:
    """Drop-in for ``torchvision.ops.roi_align``, differentiable with respect to ``input`` like torchvision's op.

    ``input`` may be contiguous NCHW or ``torch.channels_last``; both are read in place.  float32 maps are
    the parity contract; float16 maps (what the reference's live CUDA path feeds, tracking.py:177-178) are
    read as stored, sampled with float32 arithmetic and rounded to float16 once at the end.  Boxes of any
    float dtype are used at float32 (half-rounded boxes keep their half-rounded values).
    Returns a new contiguous ``[K, C, PH, PW]`` tensor of ``input``'s dtype on ``input``'s device.

    ``out_channels_last=True`` (extension; SURVEY 8f-3, the ROI -> encoder hand-off) returns the same values as a
    ``[K, C, PH, PW]`` tensor in ``torch.channels_last`` memory format, which a channels_last encoder
    (model/utils/encoder/card.py:24-41) consumes without a copy and which the kernel writes as whole cache lines.

    When grad mode is on and ``input`` requires grad, the result carries a ``grad_fn`` whose backward is
    ``roi_align_backward``: ``input.grad`` gets ``input``'s dtype and memory format, the boxes get no gradient.  The
    gradient is summed with atomic additions in an order that is not fixed (not bit-reproducible, and refused under
    ``torch.use_deterministic_algorithms(True)`` as torchvision's CUDA backward is); a float16 map's gradient is
    accumulated in float32 and rounded once.  Otherwise exactly the forward kernel runs, as before.
    """
    _lib.require_cuda(input, "input")
    if input.dim() != 4:
        raise ValueError("input must be [B, C, H, W]")
    if input.dtype not in (torch.float32, torch.float16):
        raise TypeError("roi_align: float32 or float16 feature maps only (got %s)" % input.dtype)
    if torch.is_grad_enabled() and input.requires_grad:
        rois = _boxes_to_rois(boxes, input.device)
        return _RoIAlign.apply(input, rois, _pair(output_size), spatial_scale, sampling_ratio, aligned, out_channels_last)
    return _roi_align_forward(input, boxes, output_size, spatial_scale, sampling_ratio, aligned, out_channels_last)


def _roi_align_forward(input, boxes, output_size, spatial_scale, sampling_ratio, aligned, out_channels_last):
    B, C, H, W = input.shape
    if input.is_contiguous():
        layout = _lib.LAYOUT_NCHW
    elif input.is_contiguous(memory_format=torch.channels_last):
        layout = _lib.LAYOUT_NHWC
    else:
        input, layout = input.contiguous(), _lib.LAYOUT_NCHW
    rois = _boxes_to_rois(boxes, input.device)
    PH, PW = _pair(output_size)
    K = rois.size(0)
    out = torch.empty((K, C, PH, PW), dtype=input.dtype, device=input.device,
                      memory_format=torch.channels_last if out_channels_last else torch.contiguous_format)
    dtype = _lib.DTYPE_F32 if input.dtype == torch.float32 else _lib.DTYPE_F16
    with torch.cuda.device(input.device):
        rc = _lib.lib().b200_roi_align_fwd_ex(
            _lib.ptr(input), dtype, layout, B, C, H, W, _lib.ptr(rois), K, PH, PW, float(spatial_scale),
            int(sampling_ratio), int(bool(aligned)), _lib.ptr(out),
            _lib.LAYOUT_NHWC if out_channels_last else _lib.LAYOUT_NCHW, _lib.stream_ptr(input.device))
    _lib.check(rc)
    return out


def _memory_format_of(t):
    if not t.is_contiguous() and t.is_contiguous(memory_format=torch.channels_last):
        return torch.channels_last
    return torch.contiguous_format


class _RoIAlign(torch.autograd.Function):
    """roi_align with a gradient for the map.  Saves the float32 rois and the input's metadata, not the input."""

    @staticmethod
    def forward(ctx, input, rois, output_size, spatial_scale, sampling_ratio, aligned, out_channels_last):
        ctx.save_for_backward(rois)
        ctx.input_shape = tuple(input.shape)
        ctx.dtype, ctx.memory_format = input.dtype, _memory_format_of(input)
        ctx.args = (output_size, spatial_scale, sampling_ratio, aligned)
        return _roi_align_forward(input, rois, output_size, spatial_scale, sampling_ratio, aligned, out_channels_last)

    @staticmethod
    @once_differentiable
    def backward(ctx, grad_output):
        if torch.are_deterministic_algorithms_enabled():
            msg = ("roi_align_backward does not have a deterministic implementation, but you set "
                   "'torch.use_deterministic_algorithms(True)'.")
            if not torch.is_deterministic_algorithms_warn_only_enabled():
                raise RuntimeError(msg)
            warnings.warn(msg)
        rois, = ctx.saved_tensors
        grad_input = roi_align_backward(grad_output, rois, ctx.input_shape, *ctx.args, dtype=ctx.dtype,
                                        memory_format=ctx.memory_format)
        return grad_input, None, None, None, None, None, None


def roi_align_backward(grad_output: torch.Tensor, boxes: Union[torch.Tensor, Sequence[torch.Tensor]],
                       input_shape: Sequence[int], output_size: Union[int, Tuple[int, int]], spatial_scale: float = 1.0,
                       sampling_ratio: int = -1, aligned: bool = False, *, dtype: torch.dtype = torch.float32,
                       memory_format: torch.memory_format = torch.contiguous_format) -> torch.Tensor:
    """Gradient of ``roi_align`` with respect to its input (torchvision's ``_roi_align_backward``).

    ``grad_output``: ``[K, C, PH, PW]`` float32 or float16 on a CUDA device, read in place when it is contiguous or
    ``torch.channels_last`` (otherwise copied); ``boxes`` and the scalar arguments exactly as given to ``roi_align``;
    ``input_shape``: ``(B, C, H, W)`` of the map.  Returns a new ``[B, C, H, W]`` tensor of ``dtype`` (float32 or
    float16) in ``memory_format`` (contiguous or channels_last): zeros plus the contributions of every ROI whose batch
    index is in ``[0, B)``.  The contributions are accumulated in float32 with atomic additions in an order that is not
    fixed, then rounded to ``dtype`` once; torchvision's float16 backward accumulates in float16 and differs.
    """
    _lib.require_cuda(grad_output, "grad_output")
    B, C, H, W = (int(v) for v in input_shape)
    PH, PW = _pair(output_size)
    if grad_output.dim() != 4 or tuple(grad_output.shape[1:]) != (C, PH, PW):
        raise ValueError("grad_output must be [K, %d, %d, %d] (got %s)" % (C, PH, PW, tuple(grad_output.shape)))
    if grad_output.dtype not in (torch.float32, torch.float16):
        raise TypeError("roi_align_backward: float32 or float16 grad_output only (got %s)" % grad_output.dtype)
    if dtype not in (torch.float32, torch.float16):
        raise TypeError("roi_align_backward: float32 or float16 result only (got %s)" % dtype)
    if memory_format not in (torch.contiguous_format, torch.channels_last):
        raise ValueError("roi_align_backward: memory_format must be contiguous_format or channels_last")
    rois = _boxes_to_rois(boxes, grad_output.device)
    K = rois.size(0)
    if grad_output.size(0) != K:
        raise ValueError("grad_output has %d ROIs, boxes %d" % (grad_output.size(0), K))
    if grad_output.is_contiguous():
        go_layout = _lib.LAYOUT_NCHW
    elif grad_output.is_contiguous(memory_format=torch.channels_last):
        go_layout = _lib.LAYOUT_NHWC
    else:
        grad_output, go_layout = grad_output.contiguous(), _lib.LAYOUT_NCHW
    grad_input = torch.empty((B, C, H, W), dtype=torch.float32, device=grad_output.device,
                             memory_format=memory_format).zero_()
    layout = _lib.LAYOUT_NHWC if memory_format == torch.channels_last else _lib.LAYOUT_NCHW
    gdtype = _lib.DTYPE_F32 if grad_output.dtype == torch.float32 else _lib.DTYPE_F16
    with torch.cuda.device(grad_output.device):
        rc = _lib.lib().b200_roi_align_bwd_ex(
            _lib.ptr(grad_output), gdtype, go_layout, _lib.ptr(rois), K, PH, PW, float(spatial_scale),
            int(sampling_ratio), int(bool(aligned)), _lib.ptr(grad_input), layout, B, C, H, W,
            _lib.stream_ptr(grad_output.device))
    _lib.check(rc)
    return grad_input if dtype == torch.float32 else grad_input.to(dtype)


def _prep_boxes(boxes: torch.Tensor, device, mode: int, batch_index=None, img_hw=(0, 0), map_hw=(0, 0),
                enforce_min_size: float = 0.0) -> torch.Tensor:
    """[N, >=4] boxes -> device [N, 5] roi records in ONE launch (b200_roi_boxes_prep_f32)."""
    b = boxes.reshape(-1, boxes.shape[-1]) if boxes.numel() else boxes.reshape(0, 4)
    if b.shape[1] < 4:
        raise ValueError("boxes must have at least four columns (x1, y1, x2, y2)")
    b = b.to(device=device, dtype=torch.float32)
    if b.stride(1) != 1 or (b.shape[0] > 1 and b.stride(0) < b.shape[1]):
        b = b.contiguous()
    n = b.shape[0]
    bi = None
    if batch_index is not None:
        bi = torch.as_tensor(batch_index).reshape(-1).to(device=device, dtype=torch.int32).contiguous()
        if bi.shape[0] != n:
            raise ValueError("batch_index must have one entry per box")
    rois = torch.empty((n, 5), dtype=torch.float32, device=device)
    with torch.cuda.device(device):
        rc = _lib.lib().b200_roi_boxes_prep_f32(_lib.ptr(b), n, int(b.stride(0)) if n > 1 else int(b.shape[1]), _lib.ptr(bi),
                                                mode, int(img_hw[0]), int(img_hw[1]), int(map_hw[0]), int(map_hw[1]),
                                                float(enforce_min_size), _lib.ptr(rois), _lib.stream_ptr(device))
    _lib.check(rc)
    return rois


def roi_align_from_input_boxes(feat: torch.Tensor, boxes_in, input_hw: Tuple[int, int],
                               out_size=(7, 7), aligned: bool = True, sampling_ratio: int = 2, *,
                               out_channels_last: bool = False, batch_index=None) -> torch.Tensor:
    """tracking.py:193-221: boxes are in letterboxed-input pixels, scale = Hf / H_in, batch 0.

    ``boxes_in`` is the reference's ``List[[x1, y1, x2, y2]]`` or (extension; SURVEY 8f-4, the detector -> ROI
    hand-off) a ``[N, >=4]`` tensor whose first four columns are the box -- e.g. the detector's NMS output still
    on the device, which then never visits the host (yoloDetects2.py:135-157 does ``.cpu().tolist()`` per box); the
    roi records are then built by one kernel.  ``batch_index`` (extension, int [N]): the map each box belongs to when
    ``feat`` holds several maps; the reference always passes one map, i.e. index 0.
    """
    _lib.require_cuda(feat, "feat")
    H_in, _ = input_hw
    Hf = feat.shape[2]
    if isinstance(boxes_in, torch.Tensor):
        rois = _prep_boxes(boxes_in, feat.device, _lib.BOXES_INPUT, batch_index)
    else:
        b = np.asarray(boxes_in, dtype=np.float32).reshape(-1, 4) if len(boxes_in) else np.zeros((0, 4), np.float32)
        r = np.zeros((b.shape[0], 5), np.float32)                     # batch index 0 (tracking.py:209-213)
        r[:, 1:] = b
        if batch_index is not None:
            r[:, 0] = np.asarray(batch_index, dtype=np.float32).reshape(-1)
        rois = torch.from_numpy(r).to(feat.device)
    return roi_align(feat, rois, out_size, Hf / float(H_in), sampling_ratio, aligned,
                     out_channels_last=out_channels_last)


def preprocess_roi(feat: torch.Tensor, bboxes_xyxy: torch.Tensor, img_hw: Tuple[int, int],
                   output_size=(10, 10), sampling_ratio: int = 2, aligned: bool = True,
                   enforce_min_size: float = 1.0, *, batch_index=None) -> torch.Tensor:
    """trainingCard.py:24-79: box prep in feature coordinates (one kernel: corner sort, scale, clamp, minimum size --
    float32 operation for operation), then roi_align(scale=1).

    Like the reference, ``feat`` is one map ``[1,C,H,W]``.  Extension for BASELINE config 3 (the training-time
    extraction loops 256 images, trainingCard.py:86-129): with ``batch_index`` (int [N], the image each box belongs to)
    ``feat`` may be ``[B,C,H,W]`` and the whole batch is one box-prep launch + one ROI Align launch."""
    _lib.require_cuda(feat, "feat")
    if batch_index is None:
        assert feat.dim() == 4 and feat.size(0) == 1, f"feat shape expected [1,C,H,W], got {feat.shape}"
    elif feat.dim() != 4:
        raise ValueError("feat must be [B,C,H,W]")
    _, _, Hf, Wf = feat.shape
    rois = _prep_boxes(bboxes_xyxy, feat.device, _lib.BOXES_TRAINING, batch_index, img_hw, (Hf, Wf), enforce_min_size)
    return roi_align(feat, rois, output_size, 1.0, sampling_ratio, aligned)
