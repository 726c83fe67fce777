#!/usr/bin/env python
"""Headline benchmark: tracked frames/sec of the per-frame hot path (BASELINE.json).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

The frame is BASELINE.json config 2 (the config the metric is quoted on): ROI Align of a
[1,512,40,40] map at 64 boxes -> [64,512,10,10], then the association step (predict, cost + gate,
assignment, update, births/purge) for 64 detections against ~64 tracks.  A GPU owns a GROUP of
--streams independent video streams (BASELINE.json north_star: "one stream group per GPU") and one
step advances every stream of the group by one frame with batched launches, so frames per step =
streams.  Synthetic inputs follow SURVEY.md section 8d.  Prints ONE JSON line (rank 0).

* value     : frames/s with every input already in HBM (device-resident maps, rois, detections),
              timed with CUDA events over exactly K steps, max over ranks.  Nothing else runs inside the
              timed region (the roofline probe is a separate pass); `step_ms` is the distribution of the
              per-step times inside it.
* e2e       : frames/s through the public Python API with HOST (pinned) buffers: per step the map,
              rois and detections are copied up and the match table is copied back.
* roofline  : ROI Align, algorithmic bytes / average launch duration measured with CUDA events on the
              launching stream in a separate pass right after the timed region (same buffers, nothing
              else on the GPU), against the measured copy bandwidth (MEASURED_PEAKS.json).
* cpu_baseline : the oracle port of the reference path (torchvision CPU roi_align +
              Tracking.update restated, single-threaded Python like the reference) on a bounded
              sample of the same frames, on this box's host cores.  The same leg checks a fresh
              device-side run of 40 frames, row by row, against that oracle.
* extra     : the other BASELINE configs, each a short device-timed run: c1 (single 640x640 stream), c3
              (256-map ROI extraction), c4 (512 x 512 association), c5 (64 1088x1920 streams), the
              single-stream latency mode, channels-last maps, the public API with device-resident maps.
--impl reference times the CPU path alone.  N > 1 (torchrun): one stream group per GPU (weak
scaling), result tables pushed into every peer's ring over NVLink peer memory (PeerResultGatherer, 16
frames at a time; NCCL all-gather if CUDA IPC is unavailable), value = total frames / max time; extra.c5_strong is BASELINE configs[4] as written: 64 c5
streams in total, 64/N per GPU (strong scaling).
"""
import argparse
import collections
import ctypes
import gc
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "tracked frames/sec at N=64 boxes; ROIAlign achieved HBM GB/s vs B200 peak"
C, PS = 512, 10
Shape = collections.namedtuple("Shape", "name HF WF H_IN W_IN NBOX desc")
WORKLOADS = {
    # BASELINE.json configs[0]: the reference's own CPU-runnable case (tracking.py shapes)
    "c1": Shape("c1", 20, 20, 640, 640, 8, "c1: 640x640 frame, map [1,512,20,20], 8 detections vs ~8 tracks, roi_align 10x10 + "
                                           "cost + gate + Kalman + assignment per frame"),
    # BASELINE.json configs[1]: the configuration the metric is quoted on (default)
    "c2": Shape("c2", 40, 40, 1280, 1280, 64, "c2: 1280x1280 frame, map [1,512,40,40], 64 detections vs ~64 tracks, roi_align 10x10 + "
                                              "cost + gate + Kalman + assignment per frame"),
    # BASELINE.json configs[4]: the streams of the multi-GPU configuration
    "c5": Shape("c5", 34, 60, 1088, 1920, 128, "c5: 1088x1920 frame, map [1,512,34,60], 128 detections vs ~128 tracks, roi_align "
                                               "10x10 + cost + gate + Kalman + assignment per frame"),
}
SETUP_FRAMES = 35          # history banks full (hist_max = 30) and Kalman dtypes in steady state


def roi_alg_bytes(sh, n_maps=1):
    """SURVEY.md section 8d: output written + every map read once + the roi records."""
    return n_maps * (sh.NBOX * C * PS * PS * 4 + C * sh.HF * sh.WF * 4 + sh.NBOX * 20)


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def make_frames(sh, seed, n_frames):
    """Detections of n_frames consecutive frames as dense arrays + the reference's obj dicts."""
    from alufe_b200 import synth
    scene = synth.Scene(seed, sh.NBOX, sh.H_IN, sh.W_IN)
    objs = [scene.step() for _ in range(n_frames)]
    boxes = np.array([o["bboxes"] for o in objs], dtype=np.float64)
    confs = np.array([o["confs"] for o in objs], dtype=np.float64)
    embs = np.array([np.stack(o["embs"]) for o in objs], dtype=np.float32)
    rois = np.concatenate([np.zeros((n_frames, sh.NBOX, 1)), boxes], axis=2).astype(np.float32)
    return objs, boxes, confs, embs, rois


class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons through NVML while the timed region runs."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.stop_flag, self.sm, self.reasons, self.max_mhz = index, False, [], set(), None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def sample(self):
        if self.nv is None:
            return
        nv = self.nv
        try:
            self.sm.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
            r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
            names = {"hw_slowdown": 0x8, "sw_power_cap": 0x4, "hw_thermal_slowdown": 0x40,
                     "sw_thermal_slowdown": 0x20, "hw_power_brake_slowdown": 0x80}
            for k, bit in names.items():
                if r & bit:
                    self.reasons.add(k)
        except Exception:
            pass

    def run(self):
        while not self.stop_flag:
            self.sample()
            time.sleep(0.01)

    def summary(self):
        med = float(np.median(self.sm)) if self.sm else None
        return {"sm_mhz": med, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(self.sm)}


def _cpu_worker(args):
    """One host process = one video stream through the reference path (module-level for spawn)."""
    seed, warm, max_frames, budget_s, workload = args
    sh = WORKLOADS[workload]
    import torch
    torch.set_num_threads(1)
    import alufe_b200  # noqa: F401
    from alufe_b200 import synth
    from oracle import tracker_ref, native
    try:
        from torchvision.ops import roi_align as tv_roi
    except Exception:                                              # noqa: BLE001
        tv_roi = None
    objs, *_ = make_frames(sh, seed, warm + max_frames)
    feat_cpu = synth.feature_map(seed, 1, C, sh.HF, sh.WF)
    f_t = torch.from_numpy(feat_cpu)
    ref = tracker_ref.TrackerRef(tracker_ref.SHIPPED_CONF)
    for obj in objs[:warm]:
        ref.update(obj)                       # banks fill and Kalman dtypes reach steady state
    n, t_roi, t_upd, t_start = 0, 0.0, 0.0, time.perf_counter()
    for obj in objs[warm:]:
        t0 = time.perf_counter()
        rois = np.array([[0.0] + list(b) for b in obj["bboxes"]], dtype=np.float32)
        if tv_roi is not None:
            tv_roi(f_t, torch.from_numpy(rois), (PS, PS), sh.HF / float(sh.H_IN), 2, True)
        else:
            native.roi_align(feat_cpu, rois, (PS, PS), sh.HF / float(sh.H_IN), 2, True)
        t1 = time.perf_counter()
        ref.update(obj)
        t2 = time.perf_counter()
        t_roi, t_upd, n = t_roi + (t1 - t0), t_upd + (t2 - t1), n + 1
        if t2 - t_start > budget_s:
            break
    return n, t_roi, t_upd, time.perf_counter() - t_start, ("torchvision" if tv_roi else "oracle C")


def cpu_group_fps(sh, warm, max_frames, budget_s, workers=None):
    """The reference path on the host cores: the reference is single-threaded Python per stream
    (torchvision's CPU roi_align does not scale with threads either, SURVEY.md 3.1), so independent
    streams are spread over one process per core.  Returns a cpu_baseline dict."""
    import multiprocessing as mp
    workers = workers or max(1, os.cpu_count() or 1)
    ctx = mp.get_context("spawn")
    with ctx.Pool(workers) as pool:
        out = pool.map(_cpu_worker, [(50000 + w, warm, max_frames, budget_s, sh.name) for w in range(workers)])
    fps = sum(n / wall for n, _, _, wall, _ in out)
    n_tot = sum(o[0] for o in out)
    ms_roi = 1e3 * sum(o[1] for o in out) / n_tot
    ms_upd = 1e3 * sum(o[2] for o in out) / n_tot
    return {"value": fps, "unit": "frames/s", "cores": workers, "kind": "port",
            "sample": ("%d independent " + sh.name + " streams, one host process each (%d logical CPUs), %d frames in total "
                       "after %d warm-up frames per stream: roi_align (%s CPU) %.1f ms + Tracking.update port %.1f ms per "
                       "frame per core; the association step is single-threaded Python as in the reference")
                      % (workers, os.cpu_count() or 0, n_tot, warm, out[0][4], ms_roi, ms_upd)}


_REAL_STDOUT = None


def quiet_stdout():
    """Libraries (NCCL) may print to stdout; the driver wants exactly one JSON line there.  Everything
    else is sent to stderr and emit() writes the line to the real stdout."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.dup(1)
        os.dup2(2, 1)


def emit(line):
    data = (json.dumps(line) + "\n").encode()
    sys.stdout.flush()
    os.write(_REAL_STDOUT if _REAL_STDOUT is not None else 1, data)


def run_reference(args):
    """--impl reference: the reference's CPU implementation of the path (oracle port; the
    reference is pure Python and its arithmetic lives in torchvision / filterpy / scipy), on all
    host cores, one stream per core, for the same per-frame workload as the GPU arm."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    sh = WORKLOADS[args.workload]
    # like the GPU arm: the workload is defined with full history banks (30 frames); warm-up steps the caller
    # did not ask for run as untimed set-up before the W warm-up steps
    setup = max(0, 30 - args.warmup)
    warm = setup + args.warmup
    frames = max(1, min(args.steps, 400))
    cpu = cpu_group_fps(sh, warm, frames, budget_s=120.0)
    fps = cpu["value"]
    line = {
        "impl": "reference", "metric": METRIC, "value": fps, "unit": "frames/s", "n_gpus": args.gpus, "steps": frames,
        "warmup": args.warmup, "setup_steps": setup, "ms_per_step": 1e3 * cpu["cores"] / fps, "higher_is_better": True,
        "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "%d independent streams (one per host core), each " % cpu["cores"] + sh.desc,
                   "frames_per_step": cpu["cores"]},
        "cpu_baseline": cpu,
        "e2e": {"value": fps, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    emit(line)


class StreamGroup:
    """S independent streams of one workload shape on one GPU with every input resident in HBM.

    One step = one frame of every stream: a single ROI Align launch over the S maps (K = NBOX*S ROIs,
    batch index = stream) on stream A, and one MultiStreamTracker step on stream B that waits for
    that frame's ROI launch (in the real pipeline the encoder sits between them), so ROI Align of
    frame t+1 overlaps the association of frame t."""

    def __init__(self, sh, S, n_frames, seed_base, dev, channels_last=False, with_roi=True, max_tracks=None):
        import torch
        import alufe_b200
        from alufe_b200 import _lib
        self.torch, self.lib, self._lib, self.S, self.F, self.dev, self.sh = torch, _lib.lib(), _lib, S, n_frames, dev, sh
        NB = sh.NBOX
        per = [make_frames(sh, 1000 * seed_base + s, n_frames) for s in range(S)]
        self.objs0 = per[0][0]
        self.boxes = np.stack([p[1] for p in per], axis=1)          # [F, S, NB, 4]
        self.confs = np.stack([p[2] for p in per], axis=1)
        self.embs = np.stack([p[3] for p in per], axis=1)
        rois = np.stack([p[4] for p in per], axis=1)                # [F, S, NB, 5]
        rois[..., 0] = np.arange(S, dtype=np.float32)[None, :, None]
        self.rois = rois.reshape(n_frames, S * NB, 5)
        self.d_boxes, self.d_confs = torch.from_numpy(self.boxes).to(dev), torch.from_numpy(self.confs).to(dev)
        self.d_embs, self.d_rois = torch.from_numpy(self.embs).to(dev), torch.from_numpy(self.rois).to(dev)
        self.d_ndet = torch.full((n_frames, S), NB, dtype=torch.int32, device=dev)
        self.d_frame = torch.arange(n_frames, dtype=torch.int32, device=dev)[:, None].repeat(1, S).contiguous()
        self.with_roi = with_roi
        self.map_b, self.out_b = S * C * sh.HF * sh.WF * 4, S * NB * C * PS * PS * 4
        self.roi_alg_bytes = roi_alg_bytes(sh, S)
        self.nhwc = 1 if channels_last else 0          # same values; only the memory order of each map differs
        if with_roi:
            # enough distinct maps / output buffers that nothing is served from the 126 MB L2
            self.nmap = max(2, -(-160 // max(1, self.map_b // 1000000)))
            self.nout = max(2, -(-260 // max(1, self.out_b // 1000000)))
            gen = torch.Generator(device=dev).manual_seed(1234 + seed_base)
            self.maps = torch.randn((self.nmap, S, sh.HF, sh.WF, C) if channels_last else (self.nmap, S, C, sh.HF, sh.WF),
                                    device=dev, generator=gen)
            self.outs = torch.empty((self.nout, S * NB, C, PS, PS), device=dev)
        self.trk = alufe_b200.MultiStreamTracker(S, alufe_b200.SHIPPED_CONF, max_tracks=max_tracks or max(256, 2 * NB),
                                                 max_dets=NB, device=dev)
        self.results = torch.zeros((n_frames, S, self.trk.stride), dtype=torch.int32, device=dev)
        # the association chain is short and latency-bound: it gets the high-priority stream so its CTAs are
        # scheduled ahead of the queued ROI Align tiles of the next frame
        self.sA, self.sB = torch.cuda.Stream(dev, priority=0), torch.cuda.Stream(dev, priority=-1)
        self.roi_done = [torch.cuda.Event() for _ in range(8)]
        self.ptr = {k: getattr(self, k).data_ptr() for k in
                    ("d_rois", "d_ndet", "d_boxes", "d_confs", "d_embs", "d_frame", "results")}
        if with_roi:
            self.ptr.update(maps=self.maps.data_ptr(), outs=self.outs.data_ptr())

    def roi(self, i):
        P, S, p, sh = ctypes.c_void_p, self.S, self.ptr, self.sh
        rc = self.lib.b200_roi_align_fwd_f32(P(p["maps"] + (i % self.nmap) * self.map_b), self.nhwc, S, C, sh.HF, sh.WF,
                                             P(p["d_rois"] + (i % self.F) * S * sh.NBOX * 20), S * sh.NBOX, PS, PS,
                                             sh.HF / float(sh.H_IN), 2, 1,
                                             P(p["outs"] + (i % self.nout) * self.out_b), P(self.sA.cuda_stream))
        if rc:
            self._lib.check(rc)

    def assoc(self, i):
        P, S, p, NB = ctypes.c_void_p, self.S, self.ptr, self.sh.NBOX
        rc = self.lib.b200_tracker_step(self.trk._h, P(p["d_ndet"] + 4 * i * S), P(p["d_boxes"] + i * S * NB * 32),
                                        P(p["d_confs"] + i * S * NB * 8), P(p["d_embs"] + i * S * NB * 512),
                                        P(p["d_frame"] + 4 * i * S), P(p["results"] + i * S * self.trk.stride * 4),
                                        P(self.sB.cuda_stream))
        if rc:
            self._lib.check(rc)

    def step(self, i):
        if self.with_roi:
            self.roi(i)
            ev = self.roi_done[i % len(self.roi_done)]
            ev.record(self.sA)
            self.sB.wait_event(ev)
        self.assoc(i)

    def run(self, first, count, after_step=None, start_after=None):
        """Runs `count` steps starting at frame `first`; returns (elapsed ms on the device, per-step ms).
        Per-step times come from one event per step recorded on the association stream (recording an event does
        not order the two streams, so the overlap of the pipeline is untouched)."""
        torch = self.torch
        main = torch.cuda.current_stream(self.dev)
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        marks = [torch.cuda.Event(enable_timing=True) for _ in range(count)]
        if start_after is not None:
            start_after()                     # e.g. a collective that lines the ranks up right before the first event
        gc.disable()                          # a collection inside the launch loop shows up as a millisecond step
        ev0.record(main)
        self.sA.wait_event(ev0)
        self.sB.wait_event(ev0)
        for k in range(count):
            self.step(first + k)
            marks[k].record(self.sB)
            if after_step is not None:
                after_step(first + k)
        main.wait_stream(self.sA)
        main.wait_stream(self.sB)
        return ev0, ev1, marks

    def finish(self, ev0, ev1, marks):
        torch = self.torch
        ev1.record(torch.cuda.current_stream(self.dev))
        gc.enable()
        torch.cuda.synchronize(self.dev)
        ends = [ev0.elapsed_time(m) for m in marks]
        return ev0.elapsed_time(ev1), [b - a for a, b in zip([0.0] + ends[:-1], ends)]

    def timed(self, first, count, **kw):
        return self.finish(*self.run(first, count, **kw))

    def probe_roi(self, n, first=0):
        """n ROI Align launches alone on their stream (nothing else on the GPU), CUDA events around each: the
        roofline measurement.  Map sets and output buffers keep rotating, so nothing is served from L2."""
        torch = self.torch
        torch.cuda.synchronize(self.dev)
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(n)]
        for k, (a, b) in enumerate(evs):
            a.record(self.sA)
            self.roi(first + k)
            b.record(self.sA)
        torch.cuda.synchronize(self.dev)
        return [a.elapsed_time(b) * 1e3 for a, b in evs]


def dist_summary(ms):
    """Distribution of the per-step times of a timed region (+ the first 64 of them in microseconds, in order: the first
    step carries the pipeline fill, a scheduling hiccup shows as one long step)."""
    a = np.asarray(ms, dtype=np.float64)
    return {"min": float(a.min()), "median": float(np.median(a)), "max": float(a.max()), "n": int(a.size),
            "first_us": [int(round(v * 1e3)) for v in a[:64]]}


DUMP_ROIS = 128          # 26 MB of ROI Align patches: a sample, since a step's whole output is 839 MB for 64 c2 streams


def dump_outputs(grp, i, out_dir):
    """Writes what step i of the stream group handed its caller to out_dir as .npy: the ROI Align patches of a fixed,
    seeded sample of the step's ROIs (float32 [DUMP_ROIS, 512, 10, 10], rows in the order of roi_align_rows) and the
    tracker's int32 result table [streams, stride], exactly, as float64.  The inputs are seeded, so two builds run with
    the same arguments can be compared output for output."""
    import torch
    os.makedirs(out_dir, exist_ok=True)
    n_roi = grp.S * grp.sh.NBOX
    rows = np.sort(np.random.default_rng(0).choice(n_roi, min(DUMP_ROIS, n_roi), replace=False))
    torch.cuda.synchronize(grp.dev)
    patches = grp.outs[i % grp.nout][torch.from_numpy(rows).to(grp.dev)]
    np.save(os.path.join(out_dir, "roi_align_patches.npy"), patches.cpu().numpy())
    np.save(os.path.join(out_dir, "roi_align_rows.npy"), rows.astype(np.float64))
    np.save(os.path.join(out_dir, "tracker_results.npy"), grp.results[i].cpu().numpy().astype(np.float64))


def oracle_check(dev, frames=40):
    """A fresh 2-stream device-side run (b200_tracker_step with device-resident inputs, the call the timed region
    makes) against the oracle tracker, every result row of every frame."""
    import torch
    from oracle import tracker_ref
    sh = WORKLOADS["c2"]
    g = StreamGroup(sh, 2, frames, 777, dev, with_roi=False)
    g.timed(0, frames)
    res = g.results.cpu().numpy()
    bad = 0
    for s in range(2):
        ref = tracker_ref.TrackerRef(tracker_ref.SHIPPED_CONF)
        objs = make_frames(sh, 1000 * 777 + s, frames)[0]
        for f, obj in enumerate(objs):
            want = ref.update(obj)
            got = g.trk.decode(res[f, s])
            if not (got[0] == want[0] and got[1] == want[1] and got[2] == want[2] and int(res[f, s, 5]) == 0):
                bad += 1
    del g
    torch.cuda.empty_cache()
    return {"frames_checked": 2 * frames, "mismatching_frames": bad}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=40)
    ap.add_argument("--streams", type=int, default=64, help="streams per GPU stepped together")
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--workload", choices=["c2", "c5"], default="c2",
                    help="per-stream frame shape: c2 (BASELINE configs[1], the headline) or c5 (configs[4])")
    ap.add_argument("--gather-every", type=int, default=16,
                    help="N > 1: all-gather the result tables every this many frames")
    ap.add_argument("--no-extra", action="store_true", help="skip the side measurements (other BASELINE configs)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last timed step computed to DIR/<name>.npy (rank 0)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the b200 path (--impl b200)")
    quiet_stdout()
    if args.impl == "reference":
        return run_reference(args)
    if args.warmup < 3:
        args.warmup = 3
    sh = WORKLOADS[args.workload]

    import torch
    import torch.distributed as dist
    import alufe_b200
    from alufe_b200 import _lib, dist as bdist

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product path has no CPU fallback")
    torch.cuda.set_device(local)
    # Run this rank's host side on the CPUs next to its GPU (NVML's ideal affinity): the e2e leg copies 212 MB per
    # step from pinned host memory, and pinned pages allocated on the far socket halve that copy rate.
    affinity0 = os.sched_getaffinity(0) if hasattr(os, "sched_getaffinity") else None
    near_cpus = None
    try:
        import pynvml
        pynvml.nvmlInit()
        pynvml.nvmlDeviceSetCpuAffinity(pynvml.nvmlDeviceGetHandleByIndex(local))
        near_cpus = len(os.sched_getaffinity(0))
    except Exception:                                               # noqa: BLE001
        pass
    dev = torch.device("cuda", local)
    if world > 1:
        bdist.init_process_group_small_footprint(dev)
    lib = _lib.lib()
    K, W, S = args.steps, args.warmup, args.streams
    peak, peak_src = measured_peaks()
    NB = sh.NBOX

    # ---- stream group of S streams on this GPU --------------------------------------------------------
    # The workload is defined with full history banks (hist_max = 30) and steady-state Kalman dtypes, which
    # takes 35 frames.  If the caller asks for fewer warm-up steps, the difference is run as untimed set-up
    # before the W warm-up steps, so the timed K steps always see the same workload.
    pre = max(0, SETUP_FRAMES - W)
    N_E2E, N_API = min(K, 60), 44                  # steps of the two public-API legs; they continue the same scenes in time
    n_total = pre + W + max(K, N_E2E + N_API)

    gather_kind = {}

    def make_gather(grp, n_streams_global, frames_total, boundaries):
        """The only inter-GPU traffic: the per-stream result tables, brought together for the consumer of tracking.py:329,
        GATHER_EVERY frames at a time (SURVEY.md section 8e: "optionally gather every K frames").  Product path:
        PeerResultGatherer -- every rank pushes its tables into every peer's ring over NVLink peer memory (one short
        kernel on a side stream behind an event on the association stream; nobody waits for another rank) and collects
        two gathers behind.  If CUDA IPC is not available on the box: ResultGatherer (one-CTA NCCL all-gather on a side
        stream).  Returns (after_step, flush, close)."""
        if world == 1:
            return None, (lambda: None), (lambda: None)
        G = max(1, args.gather_every)
        try:
            gat = bdist.PeerResultGatherer(n_streams_global, grp.trk.stride, G, dev)
            gather_kind["kind"] = "peer memory push over NVLink (b200_peer_gather_*), collected two gathers behind"
        except Exception as exc:                                    # noqa: BLE001
            gat = bdist.ResultGatherer(n_streams_global, grp.trk.stride, dev)
            gather_kind["kind"] = "NCCL all-gather, one-CTA kernels on a side stream (peer memory unavailable: %r)" % (exc,)
        peer = isinstance(gat, bdist.PeerResultGatherer)
        pending = []

        def collect_oldest():
            h = pending.pop(0)
            return gat.collect(h) if peer else gat.wait(h)

        def after_step(i):
            full = (i + 1) % G == 0
            if not (full or i == frames_total - 1 or (i + 1) in boundaries):   # also flush at the end of each run() call
                return
            i0 = (i // G) * G
            ev = torch.cuda.Event()
            ev.record(grp.sB)
            tables = grp.results[i0:i + 1]
            pending.append(gat.push_frames(tables, after=ev) if peer else gat.gather_frames(tables, async_op=True, after=ev))
            while len(pending) > 2:
                collect_oldest()

        def flush():
            while pending:
                collect_oldest()
            torch.cuda.current_stream(dev).wait_stream(gat.stream)

        def close():
            if peer:
                gat.close()
        return after_step, flush, close

    def lineup():
        """All ranks' first timing event lands right behind the same collective (start skew of microseconds)."""
        if world > 1:
            dist.all_reduce(torch.zeros(1, device=dev))

    grp = StreamGroup(sh, S, n_total, rank, dev)
    after_step, flush, close_gather = make_gather(grp, world * S, n_total, {pre + W})
    grp.timed(0, pre + W, after_step=after_step)
    flush()

    sampler = ClockSampler(local)
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    launches0 = lib.b200_launch_count()
    sampler.sample()
    sampler.start()
    ev = grp.run(pre + W, K, after_step=after_step, start_after=lineup)
    flush()                                    # the last gather completes inside the timed region
    elapsed_ms, step_ms = grp.finish(*ev)
    sampler.sample()
    sampler.stop_flag = True
    launches = lib.b200_launch_count() - launches0
    if world > 1:
        dist.barrier()
    t = torch.tensor([elapsed_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    elapsed_ms = float(t.item())
    close_gather()
    last = grp.results[pre + W + K - 1].cpu().numpy()
    assert (last[:, 5] == 0).all() and (last[:, 0] > 0).all(), "device path produced no matches"
    if args.dump_outputs and rank == 0:        # before the roofline probe, which writes into the same output buffers
        dump_outputs(grp, pre + W + K - 1, args.dump_outputs)

    # ---- roofline probe: ROI Align launches alone, after the timed region ---------------------------------
    roi_us = grp.probe_roi(16, first=pre + W)
    roi_us_avg = float(np.mean(roi_us))
    if world > 1:                              # every rank probes at the same time (what an N-GPU job looks like)
        tp = torch.tensor([roi_us_avg], dtype=torch.float64, device=dev)
        dist.all_reduce(tp, op=dist.ReduceOp.MAX)
        roi_us_max_ranks = float(tp.item())
    else:
        roi_us_max_ranks = roi_us_avg

    extra = {}
    # ---- BASELINE configs[4] as written: 64 c5 streams in total, 64 / N per GPU (strong scaling) ---------
    if not args.no_extra and 64 % world == 0:
        try:
            sh5, S5, K5 = WORKLOADS["c5"], 64 // world, min(max(K, 20), 60)
            n5 = SETUP_FRAMES + 5 + K5
            del grp.maps, grp.outs
            torch.cuda.empty_cache()
            g5 = StreamGroup(sh5, S5, n5, 300 + rank, dev)
            a5, f5, c5close = make_gather(g5, 64, n5, {SETUP_FRAMES + 5})
            g5.timed(0, SETUP_FRAMES + 5, after_step=a5)
            f5()
            if world > 1:
                dist.barrier()
            ev5 = g5.run(SETUP_FRAMES + 5, K5, after_step=a5, start_after=lineup)
            f5()
            ms5, step5 = g5.finish(*ev5)
            t5 = torch.tensor([ms5], dtype=torch.float64, device=dev)
            if world > 1:
                dist.all_reduce(t5, op=dist.ReduceOp.MAX)
            ms5 = float(t5.item())
            roi5 = g5.probe_roi(8, first=SETUP_FRAMES + 5)
            c5close()
            extra["c5_strong"] = {"value": 64 * K5 / (ms5 * 1e-3), "unit": "frames/s", "scaling": "strong",
                                  "streams_total": 64, "streams_per_gpu": S5, "steps": K5, "ms_per_step": ms5 / K5,
                                  "step_ms": dist_summary(step5), "roi_us_per_launch": float(np.mean(roi5)),
                                  "roi_frac_of_peak": g5.roi_alg_bytes / float(np.mean(roi5)) / 1e3 / peak,
                                  "workload": "64 streams in total, each " + sh5.desc}
            del g5
            torch.cuda.empty_cache()
        except Exception as exc:                                    # noqa: BLE001
            extra["c5_strong_error"] = repr(exc)

    # ---- end to end through the public API with host (pinned) buffers --------------------------------
    # capacity 512 like Tracking()'s default: with results collected two frames behind, the host-side bound on live tracks
    # (last known count + every detection of the pending frames) stays below it and step_async never has to drain
    ms2 = alufe_b200.MultiStreamTracker(S, alufe_b200.SHIPPED_CONF, max_tracks=max(512, 4 * NB), max_dets=NB, device=dev)
    NPIN = 2
    pin_maps = torch.randn((NPIN, S, C, sh.HF, sh.WF), generator=torch.Generator().manual_seed(99 + rank)).pin_memory()
    pin_rois = torch.from_numpy(grp.rois).pin_memory()
    feat_dev = [torch.empty((S, C, sh.HF, sh.WF), device=dev) for _ in range(2)]     # double-buffered upload target
    rois_dev = [torch.empty((S * NB, 5), device=dev) for _ in range(2)]
    n_det = np.full(S, NB, np.int32)
    # detections of every frame in page-locked host memory (where an encoder's device->host copy would land): the tracker
    # call uploads them by DMA from there
    pin_boxes = torch.from_numpy(grp.boxes).pin_memory()
    pin_confs = torch.from_numpy(grp.confs).pin_memory()
    pin_embs = torch.from_numpy(grp.embs).pin_memory()
    hb, hc, he = pin_boxes.numpy(), pin_confs.numpy(), pin_embs.numpy()
    n_e2e = N_E2E
    scale = sh.HF / float(sh.H_IN)
    copy_stream = torch.cuda.Stream(dev)
    uploaded = [torch.cuda.Event() for _ in range(2)]
    consumed = [torch.cuda.Event() for _ in range(2)]

    def upload(i):                                   # frame i's map and boxes, host (pinned) -> device
        b = i & 1
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(consumed[b])      # the ROI launch that read this buffer two frames ago
            feat_dev[b].copy_(pin_maps[i % NPIN], non_blocking=True)
            rois_dev[b].copy_(pin_rois[i % len(pin_rois)], non_blocking=True)
            uploaded[b].record(copy_stream)

    def e2e_step(i):
        """One frame of every stream through the public API.  The upload of frame i+1 is queued on a copy stream
        before the tracker call of frame i, as a caller feeding frames from the host would do."""
        b = i & 1
        main = torch.cuda.current_stream(dev)
        main.wait_event(uploaded[b])
        patches = alufe_b200.roi_align(feat_dev[b], rois_dev[b], (PS, PS), scale, 2, True)
        consumed[b].record(main)
        upload(i + 1)
        return patches, ms2.step_async(n_det, hb[i], hc[i], he[i], np.full(S, i, np.int32), pinned=True).result()

    for b in range(2):
        consumed[b].record(torch.cuda.current_stream(dev))
    upload(0)
    for i in range(pre + W):
        e2e_step(i)
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for k in range(n_e2e):
        _, res = e2e_step(pre + W + k)
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    assert (res[:, 0] > 0).all()
    # what this box's host link gives a plain pinned -> device copy of the same maps (e2e is bound by it)
    pa, pb = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    pa.record()
    for k in range(6):
        feat_dev[k & 1].copy_(pin_maps[k % NPIN], non_blocking=True)
    pb.record()
    torch.cuda.synchronize()
    pcie_probe_gbps = 6 * grp.map_b / (pa.elapsed_time(pb) * 1e-3) / 1e9
    t = torch.tensor([e2e_s], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_s = float(t.item())
    h2d = grp.map_b + S * NB * 20 + S * (8 + NB * (32 + 8 + 512))
    d2h = S * grp.trk.stride * 4
    # ---- the same public-API loop with the maps already on the device (how the reference's CUDA deployment calls
    # roi_align: the detector's map never leaves the GPU, only boxes / confidences / embeddings come from the host) ----
    if rank == 0 and not args.no_extra:
        try:
            sA = torch.cuda.Stream(dev, priority=0)
            sB = torch.cuda.Stream(dev, priority=-1)
            roi_ev = [torch.cuda.Event() for _ in range(4)]

            def api_step(i):
                """roi_align (stream A) + step_async (stream B, behind that frame's ROI Align, as the encoder would be) of
                frame i; the result of frame i - 1 is collected afterwards, as a consumer reading from a queue would
                (tracking.py:329).  Two user streams, so ROI Align of frame i + 1 overlaps the association of frame i."""
                j = pre + W + n_e2e + i            # the frames that follow the e2e leg's (same tracker, time moves on)
                with torch.cuda.stream(sA):
                    rois_dev[i & 1].copy_(pin_rois[j % len(pin_rois)], non_blocking=True)
                    patches = alufe_b200.roi_align(feat_dev[i & 1], rois_dev[i & 1], (PS, PS), scale, 2, True)
                    roi_ev[i & 3].record(sA)
                with torch.cuda.stream(sB):
                    sB.wait_event(roi_ev[i & 3])
                    h = ms2.step_async(n_det, hb[j], hc[j], he[j], np.full(S, j, np.int32), pinned=True)
                return patches, h
            sA.wait_stream(torch.cuda.current_stream(dev))
            sB.wait_stream(torch.cuda.current_stream(dev))
            LAG = 2                                # results are collected two frames behind the frame being queued
            queue = collections.deque()
            for k in range(4):
                queue.append(api_step(k)[1])
                if len(queue) > LAG:
                    queue.popleft().result()
            while queue:
                queue.popleft().result()
            torch.cuda.synchronize()
            n_api = 40
            t0 = time.perf_counter()
            for k in range(n_api):
                queue.append(api_step(4 + k)[1])
                if len(queue) > LAG:
                    res = queue.popleft().result()
            while queue:
                res = queue.popleft().result()
            torch.cuda.synchronize()
            dt = time.perf_counter() - t0
            extra["api_device_maps"] = {"value": S * n_api / dt, "unit": "frames/s", "ms_per_step": 1e3 * dt / n_api,
                                        "h2d_bytes_per_step": S * NB * 20 + S * (8 + NB * (32 + 8 + 512)),
                                        "note": "alufe_b200.roi_align + MultiStreamTracker.step_async(pinned=True) on two user streams (result of "
                                                "frame t collected after frame t + 2 is queued) with boxes / confidences / embeddings "
                                                "in pinned host memory and device-resident maps"}
        except Exception as exc:                                    # noqa: BLE001
            extra["api_device_maps_error"] = repr(exc)
    del pin_maps, feat_dev, ms2, pin_boxes, pin_confs, pin_embs, hb, hc, he
    torch.cuda.empty_cache()

    def side(name, fn):
        if rank == 0 and world == 1 and not args.no_extra:
            try:
                extra[name] = fn()
            except Exception as exc:                                # noqa: BLE001
                extra[name + "_error"] = repr(exc)
            torch.cuda.empty_cache()

    # ---- single-stream latency mode (one frame in flight; the shape the reference runs) --------------
    def single(shape):
        def fn():
            K1 = 300
            g1 = StreamGroup(shape, 1, SETUP_FRAMES + 5 + K1, 7000, dev)
            g1.timed(0, SETUP_FRAMES + 5)
            ms1, step1 = g1.timed(SETUP_FRAMES + 5, K1)
            roi1 = g1.probe_roi(32)
            return {"value": K1 / (ms1 * 1e-3), "unit": "frames/s", "ms_per_frame": ms1 / K1, "step_ms": dist_summary(step1),
                    "roi_us_per_launch": float(np.mean(roi1)), "workload": "one stream, " + shape.desc,
                    "roi_frac_of_peak": g1.roi_alg_bytes / float(np.mean(roi1)) / 1e3 / peak}
        return fn
    side("single_stream", single(sh))
    side("c1", single(WORKLOADS["c1"]))

    # ---- the same single-stream loop captured ONCE as a CUDA graph (SURVEY 8f-3): 150 consecutive frames, ROI Align on one
    # captured stream, the association step behind each frame's ROI launch on the other, replayed with one graph launch ----
    def single_graph():
        KG = 150
        g1 = StreamGroup(sh, 1, SETUP_FRAMES + 5 + KG, 7000, dev)
        g1.timed(0, SETUP_FRAMES + 5)                        # banks full, eagerly
        cap = torch.cuda.Stream(dev)
        cap.wait_stream(torch.cuda.current_stream(dev))
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph, stream=cap):
            g1.sA.wait_stream(cap)
            g1.sB.wait_stream(cap)
            g1.roi_done = [torch.cuda.Event() for _ in range(KG)]      # one event per frame inside the capture
            for k in range(KG):
                g1.step(SETUP_FRAMES + 5 + k)
            cap.wait_stream(g1.sA)
            cap.wait_stream(g1.sB)
        torch.cuda.synchronize(dev)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        with torch.cuda.stream(cap):
            a.record(cap)
            graph.replay()                                   # ONE launch: 150 frames of ROI Align + association
            b.record(cap)
        torch.cuda.synchronize(dev)
        ms = a.elapsed_time(b)
        last = g1.results[SETUP_FRAMES + 5 + KG - 1].cpu().numpy()
        assert int(last[0, 5]) == 0 and int(last[0, 0]) > 0
        return {"value": KG / (ms * 1e-3), "unit": "frames/s", "ms_per_frame": ms / KG, "frames_in_graph": KG,
                "matches_last_frame": int(last[0, 0]),
                "workload": "one stream, " + sh.desc + "; 150 frames captured once with torch.cuda.graph, one replay timed"}
    side("single_stream_graph", single_graph)

    # ---- the same stream group fed channels-last maps (what a channels_last detector would hand over) ----
    def channels_last():
        Kc = min(K, 100)
        gc = StreamGroup(sh, S, SETUP_FRAMES + 5 + Kc, 9000, dev, channels_last=True)
        gc.timed(0, SETUP_FRAMES + 5)
        msc, stepc = gc.timed(SETUP_FRAMES + 5, Kc)
        roic = gc.probe_roi(16)
        return {"value": S * Kc / (msc * 1e-3), "unit": "frames/s", "ms_per_step": msc / Kc, "step_ms": dist_summary(stepc),
                "roi_us_per_launch": float(np.mean(roic)),
                "roi_frac_of_peak": gc.roi_alg_bytes / float(np.mean(roic)) / 1e3 / peak,
                "kernel": "roi_prep_kernel + roi_align_pipe_kernel<10,10,NHWC>"}
    side("channels_last_maps", channels_last)

    # ---- BASELINE configs[2]: training-style batched extraction, 256 maps x 16 boxes -> [4096,512,10,10] ----
    def c3_roi():
        Bm, per = 256, 16
        from alufe_b200 import synth
        rng = np.random.default_rng(0)
        boxes = np.concatenate([synth.random_boxes(rng, per, 1280, 1280) for _ in range(Bm)])
        rois = np.concatenate([np.repeat(np.arange(Bm), per)[:, None].astype(np.float64), boxes], 1).astype(np.float32)
        r = torch.from_numpy(rois).to(dev)
        feat = torch.randn((Bm, C, 40, 40), device=dev)
        out = None
        evs = []
        for k in range(13):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            out = alufe_b200.roi_align(feat, r, (PS, PS), 40 / 1280.0, 2, True)
            b.record()
            evs.append((a, b))
        torch.cuda.synchronize()
        us = float(np.median([a.elapsed_time(b) for a, b in evs[3:]])) * 1e3
        alg = Bm * per * C * PS * PS * 4 + Bm * C * 40 * 40 * 4 + Bm * per * 20
        touched = None
        tp = os.path.join(ROOT, "profiles", "roi_traffic.json")
        if os.path.exists(tp):
            touched = json.load(open(tp)).get("dram_bytes_per_launch_c3")
        d = {"us_per_launch": us, "rois": Bm * per, "out_shape": list(out.shape), "alg_bytes": alg,
             "frac_of_peak_algorithmic": alg / us / 1e3 / peak,
             "note": "inputs (839 MB of maps) and output (839 MB) are each larger than L2; the algorithmic figure counts "
                     "every map byte once although only the sectors under the boxes are read"}
        if touched:
            d["dram_bytes_measured"] = touched
            d["frac_of_peak_dram_traffic"] = touched / us / 1e3 / peak
        return d
    side("c3_roi", c3_roi)

    # ---- BASELINE configs[3]: dense crowd, 512 detections x ~512 tracks, association only ---------------
    def c4_assoc():
        sh4 = Shape("c4", 40, 40, 1280, 1280, 512, "c4: 512 detections vs ~512 tracks, cost + gate + Kalman + assignment")
        K4 = 30
        g4 = StreamGroup(sh4, 1, SETUP_FRAMES + K4, 4000, dev, with_roi=False, max_tracks=1088)
        g4.timed(0, SETUP_FRAMES)
        ms4, step4 = g4.timed(SETUP_FRAMES, K4)
        last4 = g4.results[SETUP_FRAMES + K4 - 1].cpu().numpy()
        d = {"ms_per_frame": ms4 / K4, "step_ms": dist_summary(step4), "matches_last_frame": int(last4[0, 0]),
             "live_tracks": int(last4[0, 3]), "workload": sh4.desc}
        # the dense bank contraction of north_star kernel 2 as an operator: 512 tracks x 30 rows x 128 against 512 detections
        from alufe_b200 import cost as cost_ops
        bank = torch.nn.functional.normalize(torch.randn((512, 30, 128), device=dev), dim=2)
        lens = torch.full((512,), 30, dtype=torch.int32, device=dev)
        det = torch.nn.functional.normalize(torch.randn((512, 128), device=dev), dim=1)
        evs = []
        spacer = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
        for k in range(13):
            spacer.zero_()                      # flushes L2 and gives the host a head start: the events then time the
            spacer.zero_()                      # GPU work of the call, not how fast Python can enqueue it on an idle GPU
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            cost_ops.app_cost_topk(bank, lens, det, topk=5)
            b.record()
            evs.append((a, b))
        torch.cuda.synchronize()
        del spacer
        us = float(np.median([a.elapsed_time(b) for a, b in evs[3:]])) * 1e3
        d["dense_app_cost_us"] = us
        d["dense_app_cost_kernel"] = "tcgen05: bf16 three-way split, six products, TMEM accumulators (app_tc_walk_kernel)"
        d["dense_app_cost_tflops"] = 2.0 * 512 * 30 * 512 * 128 / us / 1e6
        return d
    side("c4_assoc", c4_assoc)

    # ---- CPU baseline on this box's host cores (rank 0, N == 1 only) ---------------------------------
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        if affinity0 is not None:
            os.sched_setaffinity(0, affinity0)                       # the CPU baseline uses every host core
        cpu = cpu_group_fps(sh, warm=30, max_frames=60, budget_s=12.0)
        try:
            extra["oracle_check"] = oracle_check(dev)
        except Exception as exc:                                    # noqa: BLE001
            extra["oracle_check_error"] = repr(exc)

    if rank == 0:
        traffic = None
        tp = os.path.join(ROOT, "profiles", "roi_traffic.json")
        if os.path.exists(tp) and args.workload == "c2":
            traffic = json.load(open(tp)).get("dram_bytes_per_launch_%d_streams" % S)
        frames = world * S * K
        line = {
            "metric": METRIC, "value": frames / (elapsed_ms * 1e-3), "unit": "frames/s", "n_gpus": world, "steps": K,
            "warmup": W, "setup_steps": pre, "ms_per_step": elapsed_ms / K, "step_ms": dist_summary(step_ms),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": "%d independent streams per GPU, each " % S + sh.desc, "streams_per_gpu": S,
                       "frames_per_step": S, "roi_out": [PS, PS], "layout": "nchw",
                       "l2": "inputs larger than L2: each step reads %d maps (%.0f MB) and writes %.0f MB; %d map sets and %d "
                             "output buffers rotate" % (S, grp.map_b / 1e6, grp.out_b / 1e6, grp.nmap, grp.nout),
                       "pipeline": "ROI Align of frame t+1 (stream A) overlaps the association of frame t (stream B)",
                       "gather": ("result tables of all ranks brought together every %d frames: %s; the last gather completes "
                                  "inside the timed region" % (max(1, args.gather_every), gather_kind.get("kind")))
                       if world > 1 else "single GPU: none",
                       "state_dtype": "f64 Kalman/assignment duals, f32 ROI/cost"},
            "clocks": sampler.summary(),
            "e2e": {"value": world * S * n_e2e / e2e_s, "unit": "frames/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "steps": n_e2e, "api": "alufe_b200.roi_align + MultiStreamTracker.step_async(pinned=True).result() (pinned host buffers)",
                    "h2d_gbps": h2d * n_e2e / e2e_s / 1e9, "pcie_probe_gbps": pcie_probe_gbps,
                    "host_cpus_near_gpu": near_cpus},
            "gpu_launches": int(launches),
            "roofline": {"kernel": "roi_prep_kernel + roi_align_tma_kernel<10,10,float> (one ROI Align launch, NCHW maps)",
                         "bound": "hbm", "achieved": grp.roi_alg_bytes / roi_us_avg / 1e3, "peak": peak, "unit": "GB/s",
                         "frac": grp.roi_alg_bytes / roi_us_avg / 1e3 / peak, "traffic": traffic,
                         "alg_bytes_per_launch": grp.roi_alg_bytes, "us_per_launch": roi_us_avg,
                         "us_per_launch_slowest_rank": roi_us_max_ranks, "launches_timed": len(roi_us),
                         "peak_source": peak_src,
                         "note": "separate pass after the timed region: %d ROI Align launches on the same rotating buffers, "
                                 "bracketed by CUDA events on their stream, nothing else running on the GPU" % len(roi_us)},
            "cpu_baseline": cpu,
            "extra": extra,
        }
        emit(line)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
