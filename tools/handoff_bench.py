"""Cost of the detector / encoder -> tracker hand-off (MultiStreamTracker.step_detections, Tracking.update_tensors).
Seeded inputs, warm-up first, CUDA events (device legs) or a host clock around synchronised work (host legs).  Writes one
JSON line per measurement, each with the device name and power limit read in the same run.

  group   64 config-2 streams (bench.py's stream group: 64 x 64 detections, max_tracks 256), detector rows [4096, 6] and
          embeddings [4096, 128] on the device, in stream-major order: the torch preparation a caller writes today
          (stable sort by stream, bincount, scatter into the padded float64 / float32 layout) + step_device, against
          step_detections, and step_device alone on inputs padded before the timed region; the three arms step their
          own handles through the same frames, alternating frame by frame, and their result tables are compared.
          pack_kernel + finish_kernel alone come from a torch.profiler run of their own.  float32 and float16 inputs.
  single  one config-2 stream: Tracking.update fed from .cpu().tolist() lists (the reference's hand-off,
          tracking.py:315-324) against Tracking.update_tensors, wall time per frame including the synchronise.
  graph   one config-2 stream as a CUDA graph: box prep -> ROI Align (map [1,512,40,40], 64 boxes, 10 x 10) -> a matmul
          standing in for the encoder -> step_detections; replay time per frame (the copy of the detector rows into the
          graph's input buffer is outside the timed window).

usage: python tools/handoff_bench.py [--out profiles/r04_handoff_bench.jsonl] [--frames N]"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import alufe_b200  # noqa: E402
from alufe_b200 import MultiStreamTracker, Tracking, SHIPPED_CONF, synth  # noqa: E402

SETUP = 35                   # history banks full (hist_max = 30) and Kalman dtypes in steady state, as in bench.py


def device_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader,nounits", "-i", "0"],
                       capture_output=True, text=True).stdout.strip().split(",")
    return {"device": torch.cuda.get_device_name(0), "power_limit_w": float(q[1]) if len(q) > 1 else None}


def frames_c2(S, F, seed):
    """F frames of S config-2 streams: rows [F, S*64, 6] (x1,y1,x2,y2,conf,cls) float32, embeddings [F, S*64, 128]."""
    Hf, Wf, H, W, n = synth.CONFIGS["c2"]
    scenes = [synth.Scene(seed + s, n, H, W) for s in range(S)]
    dets = np.zeros((F, S * n, 6), np.float32)
    embs = np.zeros((F, S * n, 128), np.float32)
    for f in range(F):
        for s, sc in enumerate(scenes):
            o = sc.step()
            dets[f, s * n:(s + 1) * n, :4] = o["bboxes"]
            dets[f, s * n:(s + 1) * n, 4] = o["confs"]
            embs[f, s * n:(s + 1) * n] = np.stack(o["embs"])
    return dets, embs


class TorchPrep:
    """What a caller has to write in front of step_device today: compact each stream's rows in input order into the
    padded [S, max_dets] float64 / float32 layout (buffers allocated once)."""

    def __init__(self, S, MD, dev):
        self.S, self.MD = S, MD
        self.boxes = torch.zeros((S * MD, 4), dtype=torch.float64, device=dev)
        self.confs = torch.zeros((S * MD,), dtype=torch.float64, device=dev)
        self.embs = torch.zeros((S * MD, 128), dtype=torch.float32, device=dev)
        self.ar = torch.arange(1 << 16, device=dev)

    def __call__(self, dets, embs, sidx):
        K = sidx.shape[0]
        key, perm = torch.sort(sidx, stable=True)
        counts = torch.bincount(sidx, minlength=self.S)
        starts = torch.cumsum(counts, 0) - counts
        flat = key.long() * self.MD + (self.ar[:K] - starts[key.long()])
        self.boxes[flat] = dets[perm, :4].double()
        self.confs[flat] = dets[perm, 4].double()
        self.embs[flat] = embs[perm].float()
        return (counts.int(), self.boxes.view(self.S, self.MD, 4), self.confs.view(self.S, self.MD),
                self.embs.view(self.S, self.MD, 128))


def group(info, out, frames, half):
    S, MD, dev = 64, 64, torch.device("cuda", 0)
    F = SETUP + frames
    dets_np, embs_np = frames_c2(S, F, 500)
    dt = torch.float16 if half else torch.float32
    dets = torch.from_numpy(dets_np).to(dev, dt)
    embs = torch.from_numpy(embs_np).to(dev, dt)
    K = S * synth.CONFIGS["c2"][4]
    sidx = torch.arange(S, dtype=torch.int32, device=dev).repeat_interleave(K // S)
    fid = torch.arange(F, dtype=torch.int32, device=dev)[:, None].repeat(1, S).contiguous()
    a = MultiStreamTracker(S, SHIPPED_CONF, max_tracks=256, max_dets=MD, device=dev)
    b = MultiStreamTracker(S, SHIPPED_CONF, max_tracks=256, max_dets=MD, device=dev)
    c = MultiStreamTracker(S, SHIPPED_CONF, max_tracks=256, max_dets=MD, device=dev)
    prep = TorchPrep(S, MD, dev)
    res_a = torch.zeros((S, a.stride), dtype=torch.int32, device=dev)
    res_b = torch.zeros_like(res_a)
    res_c = torch.zeros_like(res_a)
    tod = torch.zeros(K, dtype=torch.int32, device=dev)
    # step_device alone: the rows are stream-major with max_dets per stream, so the padded layout is a reshape, made
    # before the timed region
    pad = dets.view(F, S, MD, 6)
    c_boxes, c_confs = pad[..., :4].double().contiguous(), pad[..., 4].double().contiguous()
    c_embs = embs.view(F, S, MD, 128).float().contiguous()
    c_ndet = torch.full((S,), MD, dtype=torch.int32, device=dev)

    def arm_a(f):
        n_det, bx, cf, em = prep(dets[f], embs[f], sidx)
        a.step_device(n_det, bx, cf, em, fid[f], res_a)

    def arm_b(f):
        b.step_detections(dets[f, :, :4], dets[f, :, 4], embs[f], fid[f], sidx, result=res_b, track_of_det=tod)

    def arm_c(f):
        c.step_device(c_ndet, c_boxes[f], c_confs[f], c_embs[f], fid[f], res_c)

    for f in range(SETUP):
        arm_a(f)
        arm_b(f)
        arm_c(f)
    torch.cuda.synchronize()
    ev = [[torch.cuda.Event(enable_timing=True) for _ in range(6)] for _ in range(frames)]
    same = True
    for i in range(frames):
        f = SETUP + i
        ev[i][0].record(); arm_a(f); ev[i][1].record()
        ev[i][2].record(); arm_b(f); ev[i][3].record()
        ev[i][4].record(); arm_c(f); ev[i][5].record()
        if i % 16 == 15:
            torch.cuda.synchronize()
            same = same and torch.equal(res_a, res_b) and torch.equal(res_a, res_c)
    torch.cuda.synchronize()
    same = same and torch.equal(res_a, res_b) and torch.equal(res_a, res_c)
    ta = np.array([e[0].elapsed_time(e[1]) * 1e3 for e in ev])
    tb = np.array([e[2].elapsed_time(e[3]) * 1e3 for e in ev])
    tc = np.array([e[4].elapsed_time(e[5]) * 1e3 for e in ev])
    # pack_kernel + finish_kernel alone: kernel durations from a profiler run of their own (after the timed legs)
    from torch.profiler import profile, ProfilerActivity
    n_prof = 20
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for i in range(n_prof):
            arm_b(SETUP + i % frames)
        torch.cuda.synchronize()
    kern = {}
    for e in prof.events():
        if e.device_type == torch.autograd.DeviceType.CUDA:
            for name in ("pack_kernel", "finish_kernel"):
                if name in e.name:
                    kern.setdefault(name, []).append(e.time_range.elapsed_us())
    line = dict(info, leg="group", dtype="f16" if half else "f32", streams=S, K=K, max_dets=MD, frames=frames,
                torch_prep_plus_step_device_us_median=round(float(np.median(ta)), 2),
                step_detections_us_median=round(float(np.median(tb)), 2),
                step_device_alone_us_median=round(float(np.median(tc)), 2),
                step_detections_minus_step_device_us_median=round(float(np.median(tb - tc)), 2),
                torch_prep_plus_step_device_us_p10_p90=[round(float(np.percentile(ta, q)), 2) for q in (10, 90)],
                step_detections_us_p10_p90=[round(float(np.percentile(tb, q)), 2) for q in (10, 90)],
                results_equal=bool(same),
                pack_kernel_us_median=round(float(np.median(kern.get("pack_kernel", [np.nan]))), 2),
                finish_kernel_us_median=round(float(np.median(kern.get("finish_kernel", [np.nan]))), 2),
                packed_bytes_per_step=K * (4 * 8 + 8 + 128 * 4 + 4) + S * 8,
                timing="CUDA events around each arm, three arms alternating frame by frame on their own handles; kernel "
                       "times: torch.profiler, %d steps" % n_prof)
    out.write(json.dumps(line) + "\n")
    print(json.dumps(line), flush=True)


def single(info, out, frames):
    dev = torch.device("cuda", 0)
    Hf, Wf, H, W, n = synth.CONFIGS["c2"]
    F = SETUP + frames
    dets_np, embs_np = frames_c2(1, F, 700)
    dets = torch.from_numpy(dets_np).to(dev)
    embs = torch.from_numpy(embs_np).to(dev)
    a = Tracking(conf=SHIPPED_CONF, max_tracks=256, max_dets=128, device=dev)
    b = Tracking(conf=SHIPPED_CONF, max_tracks=256, max_dets=128, device=dev)

    def arm_a(f):                       # tracking.py:315-324: everything to the host, lists rebuilt
        d, e = dets[f], embs[f]
        obj = {"bboxes": d[:, :4].cpu().tolist(), "confs": d[:, 4].cpu().tolist(), "embs": list(e.cpu().numpy()),
               "input_hw": (H, W), "frame_id": f}
        return a.update(obj)

    def arm_b(f):
        d = dets[f]
        return b.update_tensors(d[:, :4], d[:, 4], embs[f], f)

    for f in range(SETUP):
        assert arm_a(f) == arm_b(f)
    ta, tb, same = [], [], True
    for i in range(frames):
        f = SETUP + i
        torch.cuda.synchronize()
        t0 = time.perf_counter(); ra = arm_a(f); torch.cuda.synchronize(); t1 = time.perf_counter()
        rb = arm_b(f); torch.cuda.synchronize(); t2 = time.perf_counter()
        ta.append((t1 - t0) * 1e6)
        tb.append((t2 - t1) * 1e6)
        same = same and ra == rb
    line = dict(info, leg="single", dtype="f32", streams=1, K=n, frames=frames,
                update_from_lists_us_median=round(float(np.median(ta)), 2),
                update_tensors_us_median=round(float(np.median(tb)), 2),
                update_from_lists_us_p10_p90=[round(float(np.percentile(ta, q)), 2) for q in (10, 90)],
                update_tensors_us_p10_p90=[round(float(np.percentile(tb, q)), 2) for q in (10, 90)],
                results_equal=bool(same),
                timing="host clock around each call and a device synchronise, arms alternating frame by frame")
    out.write(json.dumps(line) + "\n")
    print(json.dumps(line), flush=True)


def graph(info, out, frames):
    dev = torch.device("cuda", 0)
    Hf, Wf, H, W, n = synth.CONFIGS["c2"]
    F = SETUP + frames
    dets_np, _ = frames_c2(1, F, 900)
    ms = MultiStreamTracker(1, SHIPPED_CONF, max_tracks=256, max_dets=n, device=dev)
    feat = torch.from_numpy(synth.feature_map(3, 1, 512, Hf, Wf)).to(dev)
    proj = torch.randn((512 * 100, 128), device=dev, generator=torch.Generator(device=dev).manual_seed(0)) * 0.01
    dets = torch.zeros((n, 6), device=dev)
    frame = torch.zeros(1, dtype=torch.int32, device=dev)
    active = torch.zeros(1, dtype=torch.int32, device=dev)       # warm-up: stream idle
    result = torch.zeros((1, ms.stride), dtype=torch.int32, device=dev)
    tod = torch.zeros(n, dtype=torch.int32, device=dev)

    def seq():
        patches = alufe_b200.roi_align_from_input_boxes(feat, dets, (H, W), out_size=(10, 10))
        emb = patches.reshape(n, -1) @ proj
        ms.step_detections(dets[:, :4], dets[:, 4], emb, frame, active=active, result=result, track_of_det=tod)

    side = torch.cuda.Stream(dev)
    side.wait_stream(torch.cuda.current_stream(dev))
    with torch.cuda.stream(side):
        seq()
    torch.cuda.current_stream(dev).wait_stream(side)
    torch.cuda.synchronize()
    active.fill_(1)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        seq()
    t = []
    for f in range(F):
        dets.copy_(torch.from_numpy(dets_np[f]))
        frame.fill_(f)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); g.replay(); e1.record()
        torch.cuda.synchronize()
        if f >= SETUP:
            t.append(e0.elapsed_time(e1) * 1e3)
    ok = int(result[0, 5].item()) == 0
    line = dict(info, leg="graph", dtype="f32", streams=1, K=n, frames=frames,
                replay_us_median=round(float(np.median(t)), 2),
                replay_us_p10_p90=[round(float(np.percentile(t, q)), 2) for q in (10, 90)], status_ok=ok,
                sequence="box prep + ROI Align [1,512,40,40] -> [64,512,10,10] + matmul [64,51200]x[51200,128] + "
                         "step_detections (pack, step, finish)",
                timing="CUDA events around each replay")
    out.write(json.dumps(line) + "\n")
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r04_handoff_bench.jsonl"))
    ap.add_argument("--frames", type=int, default=200)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("handoff_bench: needs a CUDA device")
    info = device_info()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "a") as out:
        group(info, out, args.frames, half=False)
        group(info, out, args.frames, half=True)
        single(info, out, args.frames)
        graph(info, out, args.frames)


if __name__ == "__main__":
    main()
