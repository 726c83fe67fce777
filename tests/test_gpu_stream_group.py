"""The tracker step at the scale bench.py times it, against the oracle tracker: 64-stream c2 and c5 groups on the
three-launch chain (front_kernel, back_kernel<false>, update_kernel) with ROI Align of the next frame beside it, the
front kernel's row split at every CTA count per stream it can take, update_kernel's grid-stride loop past its first pass,
and the fused chains at their capacity limit (max_tracks 512, max_dets 256, hist_max 32).

The oracle (oracle.tracker_ref) is plain numpy and slow at these sizes, so each test runs a few distinct scenes and
replicates them over its streams (stream s shows scene s % k, so neighbouring streams differ).  TrackerRef runs once per
distinct scene, in a pool of spawned worker processes, on the same obj dicts the device gets; a stream's expected output
is the output TrackerRef computed for its scene.  Nothing about a stream's output is assumed."""
import ctypes
import multiprocessing as mp
import os
import re
import types

import numpy as np
import pytest

from conftest import assert_close
from oracle import native, tracker_ref

pytestmark = pytest.mark.gpu


def _oracle_run(cfg, frames):
    """Oracle worker: TrackerRef over one scene's frames (obj dicts; None = the scene's streams are idle that step).
    Returns, per frame, (update() tuple or None, live tracks, next id) after it, and the final TrackerRef."""
    ref = tracker_ref.TrackerRef(cfg)
    out = []
    for obj in frames:
        want = None if obj is None else ref.update(obj)
        out.append((want, len(ref.tracks), ref.next_id))
    return out, ref


# The oracle pool's workers import this module to find _oracle_run: they get numpy and the oracle, never torch or the
# package, so no worker touches the GPU.
if mp.parent_process() is None:
    import torch
    import alufe_b200  # noqa: F401
    from alufe_b200 import MultiStreamTracker, SHIPPED_CONF, synth, _lib
    from alufe_b200.tracking import R_NMATCH, R_NLIVE, R_NEXT, R_STATUS, R_M1, R_M2
    from test_gpu_tracker import _oracle_state, _compare_state
    from test_gpu_tracker_state import _row

FRONT_WARPS = 4                 # warps per front_kernel CTA (B200_TRK_FRONT_WARPS)


@pytest.fixture(scope="module")
def oracle_pool():
    with mp.get_context("spawn").Pool(min(8, os.cpu_count() or 1)) as pool:
        yield pool


def _scene_frames(seed, n, H, W, F, idle=(), empty=(), f32=False, **dynamics):
    """F steps of one scene: obj dicts with frame_id = the step, None where the scene's streams are idle (the scene
    does not advance); an empty frame has no detections.  f32: boxes and confidences rounded to float32, the values a
    detector emits."""
    sc = synth.Scene(seed, n, H, W, **dynamics)
    out = []
    for f in range(F):
        if f in idle:
            out.append(None)
            continue
        obj = sc.step()
        obj["frame_id"] = f
        if f in empty:
            obj["embs"], obj["bboxes"], obj["confs"] = [], [], []
        if f32:
            obj["bboxes"] = np.asarray(obj["bboxes"], np.float32).astype(np.float64).reshape(-1, 4).tolist()
            obj["confs"] = np.asarray(obj["confs"], np.float32).astype(np.float64).tolist()
        out.append(obj)
    return out


def _pad(scenes, MD):
    """Frames of k scenes -> step_device's arrays [F, k, ...]: n_det (-1 = idle), boxes, confs, embs padded to MD."""
    F, k = len(scenes[0]), len(scenes)
    n_det = np.full((F, k), -1, np.int32)
    boxes, confs, embs = np.zeros((F, k, MD, 4)), np.zeros((F, k, MD)), np.zeros((F, k, MD, 128), np.float32)
    for j, frames in enumerate(scenes):
        for f, obj in enumerate(frames):
            if obj is None:
                continue
            m = len(obj["bboxes"])
            assert m <= MD, "scene %d frame %d: %d detections for max_dets %d" % (j, f, m, MD)
            n_det[f, j] = m
            if m:
                boxes[f, j, :m], confs[f, j, :m], embs[f, j, :m] = obj["bboxes"], obj["confs"], np.stack(obj["embs"])
    return n_det, boxes, confs, embs


def _check_step(ms, res, want, what):
    """res: one step's result table; want: {stream: (update() tuple or None, live tracks, next id)} from the oracle."""
    for s, (w, n_live, next_id) in want.items():
        row = res[s]
        assert int(row[R_STATUS]) == 0, (what, s)
        assert (int(row[R_NLIVE]), int(row[R_NEXT])) == (n_live, next_id), (what, s)
        assert ms.decode(row) == (([], [], []) if w is None else tuple(w)), (what, s)


def _check_state(sd, s, ref, what):
    """Row s of a state_dict (host tensors) against the oracle tracker, within _compare_state's tolerances."""
    row = _row(sd, s)
    ids, st = _oracle_state(ref)
    _compare_state(types.SimpleNamespace(snapshot=lambda: row), ids, st, what)
    assert row["next_id"] == ref.next_id, what


def _host(sd):
    return {k: v.cpu() for k, v in sd.items()}


def _same_state(a, b, what):
    """Two state_dicts, bit for bit (NaN last costs included)."""
    for k in a:
        assert a[k].shape == b[k].shape and a[k].numpy().tobytes() == b[k].numpy().tobytes(), (what, k)


def _launches(fn):
    lib = _lib.lib()
    c0 = lib.b200_launch_count()
    fn()
    return lib.b200_launch_count() - c0


def _front_split():
    """(SMs, front_kernel CTAs per SM, CTAs the device holds at once), as b200_tracker_create gets them from the
    occupancy calculator: per SM from front_kernel's register count in the build's ptxas log (registers are allocated
    per warp in units of 256, 64 K of them per SM); 2 if the log is missing."""
    sms = torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count
    per_sm = 2
    log = os.path.join(_lib.CSRC, "build", "tracker.ptxas.log")
    if os.path.exists(log):
        with open(log) as fh:
            m = re.search(r"entry function '\w*front_kernel\w*'.*?Used (\d+) registers", fh.read(), re.S)
        if m:
            per_warp = -(-int(m.group(1)) * 32 // 256) * 256
            per_sm = max(1, min(65536 // (per_warp * FRONT_WARPS), 2048 // (32 * FRONT_WARPS)))
    return sms, per_sm, sms * per_sm


def _front_G(resident, S, MT):
    """CTAs per stream of front_kernel (b200_tracker_step): fill the device once, at most one CTA per four rows."""
    return min(max(resident // S, 1), -(-MT // 4))


def test_c2_group_as_the_bench_runs_it(oracle_pool):
    """bench.py's StreamGroup: 64 c2 streams, max_tracks 256, max_dets 64, the default (three-launch) schedule on a
    high-priority stream behind each frame's ROI Align, which runs on a normal-priority stream, so ROI Align of frame
    f + 1 overlaps the association of frame f.  40 frames (the 30-row banks wrap) with drops, churn, idle and empty
    frames: every result row and the final state of every stream against the oracle, replicas bit-identical, and a
    sample of each of three frames' ROI Align outputs against the oracle's ROI Align."""
    S, k, F, MT, MD, C, PS = 64, 8, 40, 256, 64, 512, 10
    Hf, Wf, H, W, n = synth.CONFIGS["c2"]
    cfg = dict(SHIPPED_CONF)
    scenes = [_scene_frames(300 + j, n, H, W, F, drop=0.1, churn=0.1, churn_every=8,
                            idle={f for f in range(F) if (f + 3 * j) % 11 == 4},
                            empty={f for f in range(F) if (f + 5 * j) % 13 == 6}) for j in range(k)]
    jobs = [oracle_pool.apply_async(_oracle_run, (cfg, frames)) for frames in scenes]
    pick = np.arange(S) % k
    n_det, boxes, confs, embs = (a[:, pick] for a in _pad(scenes, MD))
    rois = np.concatenate([np.broadcast_to(np.repeat(np.arange(S), MD)[None, :, None], (F, S * MD, 1)),
                           boxes.reshape(F, S * MD, 4)], axis=2).astype(np.float32)
    dev = torch.device("cuda", torch.cuda.current_device())
    d = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)  # noqa: E731
    d_n, d_b, d_c, d_e, d_rois = d(n_det), d(boxes), d(confs), d(embs), d(rois)
    d_f = torch.arange(F, dtype=torch.int32, device=dev)[:, None].repeat(1, S).contiguous()
    feat = torch.randn((S, C, Hf, Wf), device=dev, generator=torch.Generator(device=dev).manual_seed(3))
    outs = torch.empty((2, S * MD, C, PS, PS), device=dev)         # ROI Align output, rotating like the bench's
    sample_frames = (1, F // 2, F - 1)
    rng = np.random.default_rng(11)
    rows = {f: np.sort(rng.choice(S * MD, 64, replace=False)) for f in sample_frames}
    d_rows = {f: d(r) for f, r in rows.items()}
    ms = MultiStreamTracker(S, cfg, max_tracks=MT, max_dets=MD)
    results = torch.zeros((F, S, ms.stride), dtype=torch.int32, device=dev)
    lib, P = _lib.lib(), _lib.ptr
    sA, sB = torch.cuda.Stream(dev, priority=0), torch.cuda.Stream(dev, priority=-1)
    roi_done = [torch.cuda.Event() for _ in range(F)]
    sA.wait_stream(torch.cuda.current_stream(dev))
    sB.wait_stream(torch.cuda.current_stream(dev))
    samples, launches = {}, []
    for f in range(F):
        _lib.check(lib.b200_roi_align_fwd_f32(P(feat), 0, S, C, Hf, Wf, P(d_rois[f]), S * MD, PS, PS, Hf / float(H), 2, 1,
                                              P(outs[f % 2]), ctypes.c_void_p(sA.cuda_stream)))
        if f in rows:                                              # before ROI Align of frame f + 2 reuses the buffer
            with torch.cuda.stream(sA):
                samples[f] = outs[f % 2].index_select(0, d_rows[f])
        roi_done[f].record(sA)
        sB.wait_event(roi_done[f])
        with torch.cuda.stream(sB):
            launches.append(_launches(lambda: ms.step_device(d_n[f], d_b[f], d_c[f], d_e[f], d_f[f], results[f])))
    torch.cuda.synchronize(dev)
    assert launches == [3] * F                                     # front_kernel, back_kernel<false>, update_kernel
    res = results.cpu().numpy()
    sd = _host(ms.state_dict())
    assert np.array_equal(res, res[:, pick]), "replicas of a scene differ in their result rows"
    for key, v in sd.items():
        b = v.numpy().reshape(S, -1).view(np.uint8)
        assert np.array_equal(b, b[pick]), "replicas of a scene differ in state_dict()[%r]" % key
    want = [j.get() for j in jobs]
    for f in range(F):
        _check_step(ms, res[f], {s: want[pick[s]][0][f] for s in range(S)}, "frame %d" % f)
    for s in range(S):
        _check_state(sd, s, want[pick[s]][1], "stream %d" % s)
    maps = feat.cpu().numpy()
    for f in sample_frames:
        ref = native.roi_align(maps, rois[f][rows[f]], (PS, PS), Hf / float(H), 2, True)
        assert_close(samples[f].cpu().numpy(), ref, rtol=1e-5, atol=2e-6, what="ROI Align frame %d" % f)


def _packed(n_det, boxes, confs, embs, rng):
    """One step of every stream as a detector and an encoder emit it: float32 rows [K, 6] (x1, y1, x2, y2, conf, cls)
    and embeddings [K, 128], the streams interleaved in a random order, each stream's detections in their own order."""
    counts = np.maximum(n_det, 0)
    sidx = rng.permutation(np.repeat(np.arange(len(n_det), dtype=np.int32), counts))
    dets, e = np.zeros((len(sidx), 6), np.float32), np.zeros((len(sidx), 128), np.float32)
    for s, m in enumerate(counts):
        at = np.nonzero(sidx == s)[0]
        dets[at, :4], dets[at, 4], e[at] = boxes[s, :m], confs[s, :m], embs[s, :m]
    return dets, e, sidx


def test_c5_group_update_queue_schedules_and_handoff(oracle_pool, monkeypatch):
    """64 c5 streams of ~122 detections: one step queues ~7 800 matches, so update_kernel's grid-stride loop runs a
    second pass.  The same inputs go through the default (three-launch) chain, the two-launch chain, the six-kernel
    chain and step_detections (one shuffled [K, 6] tensor with stream indices).  The first three chains share
    front_kernel, assign_body and update_entries: bit-identical results and state.  Then the default handle's state is
    loaded into a fresh handle and both run on, bit-identically."""
    S, k, F, F2, MT, MD = 64, 8, 12, 2, 256, 128
    Hf, Wf, H, W, n = synth.CONFIGS["c5"]
    cfg = dict(SHIPPED_CONF, lost_reid_after=3, max_age=10)
    scenes = [_scene_frames(400 + j, n, H, W, F + F2, f32=True, drop=0.05) for j in range(k)]
    jobs = [oracle_pool.apply_async(_oracle_run, (cfg, frames)) for frames in scenes]
    pick = np.arange(S) % k
    n_det, boxes, confs, embs = (a[:, pick] for a in _pad(scenes, MD))
    dev = torch.device("cuda", torch.cuda.current_device())
    d = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)  # noqa: E731
    d_n, d_b, d_c, d_e = d(n_det), d(boxes), d(confs), d(embs)
    d_f = torch.arange(F + F2, dtype=torch.int32, device=dev)[:, None].repeat(1, S).contiguous()
    handles, schedule = {}, {"chain3": None, "chain2": "2", "chain6": "6", "packed": None}
    for name, chain in schedule.items():
        if chain is None:
            monkeypatch.delenv("B200TRACK_CHAIN", raising=False)
        else:
            monkeypatch.setenv("B200TRACK_CHAIN", chain)
        handles[name] = MultiStreamTracker(S, cfg, max_tracks=MT, max_dets=MD)
    monkeypatch.delenv("B200TRACK_CHAIN", raising=False)
    stride = handles["chain3"].stride
    results = {name: torch.zeros((F + F2, S, stride), dtype=torch.int32, device=dev) for name in list(handles) + ["loaded"]}
    launches = {name: [] for name in results}
    rng = np.random.default_rng(8)
    K = []
    for f in range(F + F2):
        if f == F:
            handles["loaded"] = MultiStreamTracker(S, cfg, max_tracks=MT, max_dets=MD)
            handles["loaded"].load_state_dict(handles["chain3"].state_dict())
        dets, e, sidx = _packed(n_det[f], boxes[f], confs[f], embs[f], rng)
        K.append(len(sidx))
        dd = d(dets)
        for name, ms in handles.items():
            if name == "packed":
                step = lambda: ms.step_detections(dd[:, :4], dd[:, 4], d(e), d_f[f], d(sidx), result=results[name][f])  # noqa
            else:
                step = lambda: ms.step_device(d_n[f], d_b[f], d_c[f], d_e[f], d_f[f], results[name][f])  # noqa: E731
            launches[name].append(_launches(step))
    torch.cuda.synchronize(dev)
    # pack_kernel + the three-launch chain + finish_kernel for step_detections
    assert {name: set(v) for name, v in launches.items()} == {"chain3": {3}, "chain2": {2}, "chain6": {6}, "packed": {5},
                                                              "loaded": {3}}
    assert min(K) > 7000
    res = {name: r.cpu().numpy() for name, r in results.items()}
    sd = {name: _host(ms.state_dict()) for name, ms in handles.items()}
    for name in ("chain2", "packed"):
        assert np.array_equal(res[name], res["chain3"]), name
        _same_state(sd[name], sd["chain3"], name)
    assert np.array_equal(res["loaded"][F:], res["chain3"][F:])
    _same_state(sd["loaded"], sd["chain3"], "loaded")
    want = [j.get() for j in jobs]
    for name in ("chain3", "chain6"):
        for f in range(F + F2):
            _check_step(handles[name], res[name][f], {s: want[pick[s]][0][f] for s in range(S)}, "%s frame %d" % (name, f))
        for s in range(S):
            _check_state(sd[name], s, want[pick[s]][1], "%s stream %d" % (name, s))
    # a second pass of update_kernel: 4 entries x 4 warps per CTA, 2 CTAs per SM
    sms = torch.cuda.get_device_properties(dev).multi_processor_count
    most = int(res["chain3"][:, :, R_NMATCH].sum(axis=1).max())
    assert most > 16 * 2 * sms, (most, sms)
    print("c5 group: SMs %d, most matches in one step %d (update_kernel pass: %d), K %d..%d"
          % (sms, most, 32 * sms, min(K), max(K)))


def test_front_row_split_and_fused_capacity_edge(oracle_pool, monkeypatch):
    """max_tracks 512, max_dets 256, hist_max 32 -- the largest handle the fused chains take -- with three crowded scenes
    (~230 detections against up to ~440 tracks, long-lost ReID rows) on streams 0, S // 2 and S - 1 of handles whose
    stream counts S make front_kernel run G = 128 (one to four rows per CTA), 8, 4, 2 and 1 CTAs per stream; every
    other stream is idle.  Chains 2 and 3 at every S, chain 6 and a 513-track handle (six-kernel chain by capacity)
    beside them: the same results as the oracle, the same state bit for bit across S and across chains 2 / 3."""
    MT, MD, F = 512, 256, 10
    cfg = dict(SHIPPED_CONF, hist_max=32, lost_reid_after=2, max_age=8)
    scenes = [_scene_frames(700 + j, 300, 1280, 1280, F, drop=0.25, churn=0.1, churn_every=4) for j in range(3)]
    jobs = [oracle_pool.apply_async(_oracle_run, (cfg, frames)) for frames in scenes]
    dev = torch.device("cuda", torch.cuda.current_device())
    n_det, boxes, confs, embs = (torch.from_numpy(a).to(dev) for a in _pad(scenes, MD))
    sms, per_sm, resident = _front_split()
    gs = [-(-MT // 4), 8, 4, 2, 1]
    streams = [resident // g for g in gs]
    assert [_front_G(resident, S, MT) for S in streams] == gs, (resident, streams)
    print("front_kernel: SMs %d, CTAs per SM %d, S %s -> G %s" % (sms, per_sm, streams, gs))

    def run(S, chain, max_tracks=MT):
        if chain is None:
            monkeypatch.delenv("B200TRACK_CHAIN", raising=False)
        else:
            monkeypatch.setenv("B200TRACK_CHAIN", chain)
        ms = MultiStreamTracker(S, cfg, max_tracks=max_tracks, max_dets=MD)
        monkeypatch.delenv("B200TRACK_CHAIN", raising=False)
        where = list(dict.fromkeys([0, S // 2, S - 1]))            # stream of scene j (S = 2 holds two of them)
        at = torch.tensor(where, device=dev)
        m = len(where)
        nd = torch.full((S,), -1, dtype=torch.int32, device=dev)
        bx = torch.zeros((S, MD, 4), dtype=torch.float64, device=dev)
        cf = torch.zeros((S, MD), dtype=torch.float64, device=dev)
        em = torch.zeros((S, MD, 128), dtype=torch.float32, device=dev)
        results = torch.zeros((F, S, ms.stride), dtype=torch.int32, device=dev)
        launches = []
        for f in range(F):
            nd[at], bx[at], cf[at], em[at] = n_det[f, :m], boxes[f, :m], confs[f, :m], embs[f, :m]
            fr = torch.full((S,), f, dtype=torch.int32, device=dev)
            launches.append(_launches(lambda: ms.step_device(nd, bx, cf, em, fr, results[f])))
        sd = _host(ms.state_dict(streams=where))
        torch.cuda.synchronize(dev)
        res = results.cpu().numpy()
        out = types.SimpleNamespace(ms=ms, where=where, res=res, sd=sd, launches=launches, S=S, chain=chain)
        ms.close()
        return out

    runs = []
    for S in streams:
        runs += [run(S, "2"), run(S, "3")]
    runs += [run(streams[0], "6"), run(streams[0], None, MT + 1)]
    want = [j.get() for j in jobs]
    first = {}                                                     # scene -> state row of the first run that had it
    for r in runs:
        what = "S %d chain %s max_tracks %d" % (r.S, r.chain, r.ms.max_tracks)
        assert set(r.launches) == {int(r.chain or 6)}, what
        assert (r.res[:, :, R_STATUS] == 0).all(), what
        idle = np.setdiff1d(np.arange(r.S), r.where)
        assert (r.res[:, idle, :8] == 0).all(), what                # idle all along: no tracks, next id 0, status 0
        for f in range(F):
            _check_step(r.ms, r.res[f], {s: want[j][0][f] for j, s in enumerate(r.where)}, "%s frame %d" % (what, f))
        for j in range(len(r.where)):
            row = {key: v[j:j + 1] for key, v in r.sd.items()}
            if r.chain == "6" or r.ms.max_tracks != MT:
                _check_state(r.sd, j, want[j][1], "%s scene %d" % (what, j))
            elif j not in first:
                _check_state(r.sd, j, want[j][1], "%s scene %d" % (what, j))
                first[j] = row
            else:
                _same_state(row, first[j], "%s scene %d" % (what, j))
    assert sorted(first) == [0, 1, 2]
    # coverage, from the result headers of the G = 1 run (every run saw the same inputs)
    g1 = next(r for r in runs if r.S == streams[-1] and r.chain == "3")
    m1, m2 = g1.res[:, g1.where, R_M1], g1.res[:, g1.where, R_M2]
    nd = n_det.cpu().numpy()[:, :len(g1.where)]
    assert ((m1 > 256) & (nd < m1)).any(), "no stage-1 matrix with more than 256 track rows and fewer detections"
    assert (m2 > 0).any(), "no long-lost (ReID) rows"
    assert (m1 + m2 > 128).any(), "no stream with more rows than one front_kernel CTA has threads"
    print("fused capacity edge: largest M1 %d, largest M1 + M2 %d" % (m1.max(), (m1 + m2).max()))
