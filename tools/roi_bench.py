"""Micro-benchmark of the ROI Align kernel at the BASELINE.json shapes (CUDA events, L2 flushed
or inputs larger than L2).  Prints one JSON line per case.  Not the headline bench (bench.py).

--backward times the gradient instead: the public roi_align_backward call (zero fill of grad_in included; "nhwc" =
channels-last grad_in) against torchvision's CUDA _roi_align_backward (which zero-fills too).  Algorithmic bytes are
the forward's formula -- each upstream gradient read once, each input gradient written once -- a floor that the zero
fill and the read-modify-write of the additions in L2 put out of reach; the fraction is reported against it anyway."""
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import alufe_b200  # noqa: E402,F401
from alufe_b200 import roi, synth  # noqa: E402

PEAK = 6548.5
if os.path.exists(os.path.join(ROOT, "MEASURED_PEAKS.json")):
    PEAK = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"]


def timed(fn, iters, flush):
    start = [torch.cuda.Event(enable_timing=True) for _ in range(iters)]
    stop = [torch.cuda.Event(enable_timing=True) for _ in range(iters)]
    for i in range(iters):
        if flush is not None:
            flush.zero_()
        start[i].record()
        fn()
        stop[i].record()
    torch.cuda.synchronize()
    t = sorted(s.elapsed_time(e) for s, e in zip(start, stop))
    return t[len(t) // 2] * 1e-3, t[0] * 1e-3


def case(name, Bm, Hf, Wf, H_in, W_in, per_map, ps=(10, 10), nhwc=False, tv=False, iters=20, half=False, out_cl=False,
         backward=False):
    rng = np.random.default_rng(0)
    boxes = np.concatenate([synth.random_boxes(rng, per_map, H_in, W_in) for _ in range(Bm)])
    rois = np.concatenate([np.repeat(np.arange(Bm), per_map)[:, None].astype(np.float64), boxes], 1).astype(np.float32)
    r = torch.from_numpy(rois).cuda()
    feat = torch.randn((Bm, 512, Hf, Wf), device="cuda")
    if half:
        feat = feat.half()
    if nhwc:
        feat = feat.contiguous(memory_format=torch.channels_last)
    K = r.shape[0]
    es = 2 if half else 4
    alg = K * 512 * ps[0] * ps[1] * es + Bm * 512 * Hf * Wf * es + K * 20
    flush = torch.empty(256 * 1024 * 1024 // 4, device="cuda") if alg < 512e6 else None
    if backward:
        alg = K * 512 * ps[0] * ps[1] * es + Bm * 512 * Hf * Wf * 4 + K * 20      # grad_in is float32
        flush = torch.empty(256 * 1024 * 1024 // 4, device="cuda") if alg < 512e6 else None
        g = torch.randn((K, 512) + tuple(ps), device="cuda", dtype=torch.float16 if half else torch.float32)
        if tv:
            import torchvision  # noqa: F401  (registers torch.ops.torchvision)
            fn = lambda: torch.ops.torchvision._roi_align_backward(g, r, Hf / float(H_in), ps[0], ps[1], Bm, 512, Hf, Wf, 2,
                                                                   True)
        else:
            mf = torch.channels_last if nhwc else torch.contiguous_format
            fn = lambda: roi.roi_align_backward(g, r, (Bm, 512, Hf, Wf), ps, Hf / float(H_in), 2, True, memory_format=mf)
    elif tv:
        import torchvision
        fn = lambda: torchvision.ops.roi_align(feat, r, ps, Hf / float(H_in), 2, True)
    else:
        fn = lambda: roi.roi_align(feat, r, ps, Hf / float(H_in), 2, True, out_channels_last=out_cl)
    for _ in range(3):
        fn()
    med, best = timed(fn, iters, flush)
    print(json.dumps({**({"pass": "backward"} if backward else {}), "case": name,
                      "impl": "torchvision" if tv else "b200", "layout": ("nhwc" if nhwc else "nchw") + ("->nhwc" if out_cl else ""), "dtype": "f16" if half else "f32",
                      "K": K, "out": list(ps), "alg_MB": round(alg / 1e6, 2), "us_median": round(med * 1e6, 2),
                      "us_best": round(best * 1e6, 2), "GBps_median": round(alg / med / 1e9, 1),
                      "frac_of_measured_peak": round(alg / med / 1e9 / PEAK, 3)}), flush=True)


if __name__ == "__main__":
    args = [a for a in sys.argv[1:] if not a.startswith("--")]
    flags = [a for a in sys.argv[1:] if a.startswith("--")]
    which = args or ["c1", "c2", "c3", "c5"]
    impls = (False,) if "--b200" in flags else (False, True)
    layouts = (False,) if "--nchw" in flags else (True,) if "--nhwc" in flags else (False, True)
    if "--backward" in flags:
        which = args or ["c1", "c2", "c3", "c5", "g64"]
        print(subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True).stdout.strip(), flush=True)
        shapes = {"c1": ("c1", 1, 20, 20, 640, 640, 8, 20), "c2": ("c2", 1, 40, 40, 1280, 1280, 64, 20),
                  "c3": ("c3", 256, 40, 40, 1280, 1280, 16, 10), "c5": ("c5x64", 64, 34, 60, 1088, 1920, 128, 10),
                  "g64": ("g64", 64, 40, 40, 1280, 1280, 64, 10)}
        for w in which:
            name, Bm, Hf, Wf, H_in, W_in, per_map, iters = shapes[w]
            for tv in impls:        # torchvision's gradient is NCHW only
                for nhwc in (layouts if not tv else (False,)):
                    case(name, Bm, Hf, Wf, H_in, W_in, per_map, nhwc=nhwc, tv=tv, iters=iters, backward=True)
            if "--half" in flags:
                for nhwc in layouts:
                    case(name, Bm, Hf, Wf, H_in, W_in, per_map, nhwc=nhwc, iters=iters, half=True, backward=True)
        sys.exit(0)
    for tv in impls:
        for nhwc in layouts:
            if "c1" in which:
                case("c1", 1, 20, 20, 640, 640, 8, nhwc=nhwc, tv=tv)
            if "c2" in which:
                case("c2", 1, 40, 40, 1280, 1280, 64, nhwc=nhwc, tv=tv)
            if "c3" in which:
                case("c3", 256, 40, 40, 1280, 1280, 16, nhwc=nhwc, tv=tv, iters=10)
                if nhwc and not tv:
                    case("c3", 256, 40, 40, 1280, 1280, 16, nhwc=True, iters=10, out_cl=True)
            if "c5" in which:
                case("c5x64", 64, 34, 60, 1088, 1920, 128, nhwc=nhwc, tv=tv, iters=10)
                if nhwc and not tv:
                    case("c5x64", 64, 34, 60, 1088, 1920, 128, nhwc=True, iters=10, out_cl=True)
            if "g64" in which:      # the bench.py stream group: 64 maps x 64 boxes per launch
                case("g64", 64, 40, 40, 1280, 1280, 64, nhwc=nhwc, tv=tv, iters=10)
                if not tv:
                    case("g64", 64, 40, 40, 1280, 1280, 64, nhwc=nhwc, iters=10, out_cl=True)
            if "g64h" in which and not tv:      # float16 storage
                case("g64", 64, 40, 40, 1280, 1280, 64, nhwc=nhwc, iters=10, half=True)
                case("c3", 256, 40, 40, 1280, 1280, 16, nhwc=nhwc, iters=10, half=True)
            if "c2_7" in which:
                case("c2_7x7", 1, 40, 40, 1280, 1280, 64, ps=(7, 7), nhwc=nhwc, tv=tv)
