"""Cost of moving tracker state on the device (b200_tracker_export_device / b200_tracker_import_device, state_dict,
load_state_dict, grow, reset of one stream).  Writes one JSON line per measurement, each with the device name and power
limit read in the same run.

  kernels  a 64-stream handle of 256 slots at hist_max 30, filled to 256 live tracks per stream by loading a synthetic
           valid image (BYTES_PER_TRACK x 16 384 tracks = 270 MB, more than the 126 MB of L2): export and import of all
           64 rows timed with CUDA events around each launch; GB/s from 2 x live tracks x BYTES_PER_TRACK (every byte
           read once and written once), as a fraction of tools/bw_probe.py's copy_rw_GBps measured in the same run.
  grow     256 -> 512 slots, wall clock to a synchronise: grow() (image export, handle creation, import, each also timed
           on its own) against the per-stream host loop grow() used to run (export -> create -> import_state), re-implemented
           here; median of several runs, each on a freshly loaded handle, the two paths alternating.
  stream   reset(streams=[k]) and moving one stream between two handles (state_dict([k]) -> load_state_dict(.., [j])),
           wall clock to a synchronise.

usage: python tools/tracker_state_bench.py [--out profiles/r05_tracker_state_bench.jsonl]"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import alufe_b200  # noqa: E402,F401
from alufe_b200 import MultiStreamTracker, SHIPPED_CONF, _lib  # noqa: E402

S, CAP, H = 64, 256, SHIPPED_CONF["hist_max"]
# ids, stage, bank_len, miss, age (4+1+4+4+4) + x (64) + P (512) + ema (512) + last_bbox (32) + last_conf, last_cost (16)
# + the bank (hist_max x 512)
BYTES_PER_TRACK = 17 + 64 + 512 + 512 + 32 + 16 + H * 512


def device_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader,nounits", "-i", "0"],
                       capture_output=True, text=True).stdout.strip().split(",")
    return {"device": torch.cuda.get_device_name(0), "power_limit_w": float(q[1]) if len(q) > 1 else None}


def synthetic_image(ms, n_live):
    """A valid image: n_live tracks per stream, ids 0..n_live-1, full banks, random values."""
    g = torch.Generator(device="cuda").manual_seed(5)
    sd = ms._new_image(S, CAP)
    sd["n_live"].fill_(n_live)
    sd["next_id"].fill_(n_live + 7)
    sd["ids"][:, :n_live] = torch.arange(n_live, dtype=torch.int32, device="cuda")
    for k in ("x", "P", "last_bbox", "last_conf", "last_cost"):
        sd[k][:, :n_live] = torch.rand(sd[k][:, :n_live].shape, generator=g, device="cuda", dtype=torch.float64)
    for k in ("ema", "bank"):
        sd[k][:, :n_live] = torch.rand(sd[k][:, :n_live].shape, generator=g, device="cuda")
    sd["stage"][:, :n_live] = 2
    sd["bank_len"][:, :n_live] = H
    sd["age"][:, :n_live] = 40
    return sd


def event_times(fn, n):
    for _ in range(3):
        fn()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(n)]
    for a, b in ev:
        a.record()
        fn()
        b.record()
    torch.cuda.synchronize()
    return [a.elapsed_time(b) * 1e3 for a, b in ev]         # us


def wall(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) * 1e6                 # us


def stats(xs):
    return {"median": round(float(np.median(xs)), 2), "p10_p90": [round(float(np.percentile(xs, q)), 2) for q in (10, 90)]}


def bw_probe():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "bw_probe.py")], capture_output=True, text=True,
                         check=True).stdout
    return json.loads(out.strip().splitlines()[-1])


def loaded_handle(sd):
    ms = MultiStreamTracker(S, SHIPPED_CONF, max_tracks=CAP, max_dets=64)
    ms.load_state_dict(sd)
    return ms


def kernels(sd, info, bw, launches):
    ms = loaded_handle(sd)
    img = ms._new_image(S, CAP)
    im_out, im_in = ms._c_image(img), ms._c_image(sd)
    status = torch.empty(S, dtype=torch.int32, device="cuda")
    lib, st = _lib.lib(), _lib.stream_ptr()
    exp = event_times(lambda: _lib.check(lib.b200_tracker_export_device(ms._h, None, ctypes.byref(im_out), None, st)),
                      launches)
    imp = event_times(lambda: _lib.check(lib.b200_tracker_import_device(ms._h, None, ctypes.byref(im_in),
                                                                         _lib.ptr(status), st)), launches)
    torch.cuda.synchronize()
    assert (status == 0).all()
    same = all(torch.equal(img[k], sd[k]) for k in img)          # export of what was imported gives the image back
    nbytes = 2 * S * CAP * BYTES_PER_TRACK
    rows = []
    for name, ts in (("export_device", exp), ("import_device", imp)):
        med = float(np.median(ts))
        gbps = nbytes / (med * 1e-6) / 1e9
        rows.append(dict(info, leg="kernels", call=name, streams=S, live_tracks=S * CAP, hist_max=H,
                         bytes_per_track=BYTES_PER_TRACK, bytes_moved=nbytes, launches=launches, us=stats(ts),
                         GBps_at_median=round(gbps, 1), copy_rw_GBps=round(bw["copy_rw_GBps"], 1),
                         fraction_of_copy_rw=round(gbps / bw["copy_rw_GBps"], 3),
                         ideal_us_at_copy_rw=round(nbytes / (bw["copy_rw_GBps"] * 1e9) * 1e6, 1),
                         round_trip_equal=bool(same),
                         timing="CUDA events around each launch; image and handle state 270 MB each, larger than L2"))
    ms.close()
    return rows


def old_grow(ms, max_tracks):
    """grow() as it was: a synchronous export of every stream to host arrays, a new handle, an import of every stream."""
    snaps = [ms.export(s) for s in range(ms.S)]
    old = ms._h
    ms._create(max_tracks, ms.max_dets)
    _lib.lib().b200_tracker_destroy(old)
    for s, snap in enumerate(snaps):
        ms.import_state(s, snap)


def grow(sd, info, runs):
    new, parts, old = [], {"state_dict": [], "create": [], "import": []}, []
    for _ in range(runs):
        ms = loaded_handle(sd)
        new.append(wall(lambda: ms.grow(max_tracks=2 * CAP)))
        ms.close()
        ms = loaded_handle(sd)                             # the same path, one part at a time
        box = {}
        parts["state_dict"].append(wall(lambda: box.update(img=ms.state_dict())))
        h_old = ms._h
        parts["create"].append(wall(lambda: ms._create(2 * CAP, ms.max_dets)))
        parts["import"].append(wall(lambda: ms._import(box["img"], None)))
        _lib.lib().b200_tracker_destroy(h_old)
        ms.close()
        del box
        ms = loaded_handle(sd)
        old.append(wall(lambda: old_grow(ms, 2 * CAP)))
        ms.close()
    return [dict(info, leg="grow", streams=S, live_tracks=S * CAP, slots=[CAP, 2 * CAP], runs=runs,
                 grow_us=stats(new), host_loop_us=stats(old), parts_us={k: stats(v) for k, v in parts.items()},
                 timing="host clock to a device synchronise; new path and host loop alternating, fresh handle each run")]


def stream_ops(sd, info, runs):
    a, b = loaded_handle(sd), loaded_handle(sd)
    reset = [wall(lambda: a.reset(streams=[k % S])) for k in range(runs)]
    move = [wall(lambda: b.load_state_dict(a.state_dict([(k + 1) % S]), streams=[k % S])) for k in range(runs)]
    a.close()
    b.close()
    return [dict(info, leg="stream", streams=S, live_tracks_per_stream=CAP, runs=runs, reset_one_stream_us=stats(reset),
                 move_one_stream_us=stats(move),
                 timing="host clock to a device synchronise; move = state_dict([k]) on one handle + load_state_dict into "
                        "another (which reads the status back)")]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r05_tracker_state_bench.jsonl"))
    ap.add_argument("--launches", type=int, default=40)
    ap.add_argument("--runs", type=int, default=5)
    args = ap.parse_args()
    info = device_info()
    bw = bw_probe()
    ms = MultiStreamTracker(S, SHIPPED_CONF, max_tracks=CAP, max_dets=64)
    sd = synthetic_image(ms, CAP)
    ms.close()
    rows = kernels(sd, info, bw, args.launches) + grow(sd, info, args.runs) + stream_ops(sd, info, 4 * args.runs)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "a") as out:
        for r in rows:
            line = json.dumps(r)
            print(line)
            out.write(line + "\n")


if __name__ == "__main__":
    main()
