"""MultiStreamTracker.step_detections / b200_tracker_step_packed (detector rows + encoder embeddings in their own layout
-> the tracker step) and Tracking.update_tensors: bit-identical to step_device fed the same values compacted on the host,
equal to the oracle tracker, every layout and edge case of the hand-off, and inside a captured CUDA graph."""
import numpy as np
import pytest
import torch

from conftest import assert_close
from oracle import tracker_ref

pytestmark = pytest.mark.gpu

import alufe_b200  # noqa: E402,F401
from alufe_b200 import MultiStreamTracker, Tracking, SHIPPED_CONF, roi, synth  # noqa: E402
from alufe_b200 import _lib  # noqa: E402
from alufe_b200.tracking import R_NMATCH, R_NLIVE, R_NEXT, R_STATUS  # noqa: E402

CFG = dict(SHIPPED_CONF, lost_reid_after=5, max_age=15)
STATE_KEYS = ("ids", "x", "P", "stage", "ema", "bank", "bank_len", "miss", "age", "last_bbox", "last_conf", "last_cost")


def _frame(objs, rng, half=False, junk=0):
    """One frame of every stream (obj, or None = no frame) as a detector and an encoder emit it: rows [K, 6] =
    (x1, y1, x2, y2, conf, cls) and embeddings [K, 128] in float32 (or float16), interleaved across streams in a random
    order, plus `junk` rows whose stream index is outside [0, S).  Returns (dets, embs, stream_index, rows of each
    stream in input order)."""
    dt = np.float16 if half else np.float32
    parts = [(s, j) for s, o in enumerate(objs) if o is not None for j in range(len(o["bboxes"]))]
    parts += [(bad, 0) for bad in rng.choice([-1, len(objs), 1 << 20], junk)]
    order = rng.permutation(len(parts)) if parts else np.zeros(0, np.int64)
    K = len(parts)
    dets = np.zeros((K, 6), dt)
    embs = np.zeros((K, 128), dt)
    sidx = np.zeros(K, np.int32)
    rows = [[] for _ in objs]
    for k, p in enumerate(order):
        s, j = parts[p]
        sidx[k] = s
        if 0 <= s < len(objs):
            o = objs[s]
            dets[k, :4], dets[k, 4], dets[k, 5] = o["bboxes"][j], o["confs"][j], 0
            embs[k] = o["embs"][j]
            rows[s].append(k)
        else:
            dets[k] = rng.uniform(0, 500, 6)
            embs[k] = rng.standard_normal(128)
    return dets, embs, sidx, rows


def _oracle_obj(dets, embs, rows, f, hw):
    """What the oracle gets for one stream: the emitted (rounded) values, in the stream's input order."""
    return {"bboxes": dets[rows, :4].astype(np.float64).tolist(), "confs": dets[rows, 4].astype(np.float64).tolist(),
            "embs": [embs[k].astype(np.float32) for k in rows], "input_hw": hw, "frame_id": f}


def _dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _check_track_of_det(ms, table, tod, rows):
    """track_of_det[k] = the track id of the match of det_idx j of stream s, where k is that detection's input row."""
    want = np.full(len(tod), -1, np.int64)
    for s, r in enumerate(rows):
        for tid, j in ms.decode(table[s])[0]:
            want[r[j]] = tid
    assert tod.tolist() == want.tolist()


def _scenes(S, seed):
    """10 .. 47 identities per stream: within the max_dets (48 / 64) of the handles below at any S."""
    return [synth.Scene(seed + s, 10 + (7 * s) % 38, 1088, 1920, drop=0.15, churn=0.15, churn_every=7) for s in range(S)]


@pytest.mark.parametrize("S,chain", [(4, None), (16, None), (4, "6")])
def test_packed_step_is_bit_identical_to_step_device(S, chain, monkeypatch):
    """S = 4 runs the two-launch step, S = 16 the three-launch one, B200TRACK_CHAIN=6 the six-kernel chain.  A second
    handle gets the same values compacted on the host in input order through step_device: every result table and every
    exported state is equal bit for bit (same kernels, same values)."""
    if chain is not None:
        monkeypatch.setenv("B200TRACK_CHAIN", chain)
    F, MD, hw = 36, 64, (1088, 1920)
    packed = MultiStreamTracker(S, CFG, max_tracks=192, max_dets=MD)
    padded = MultiStreamTracker(S, CFG, max_tracks=192, max_dets=MD)
    scenes = _scenes(S, 40)
    rng = np.random.default_rng(S)
    res_a = torch.zeros((F, S, packed.stride), dtype=torch.int32, device="cuda")
    res_b = torch.zeros_like(res_a)
    for f in range(F):
        objs = []
        for s in range(S):
            if (f + 2 * s) % 9 == 4:
                objs.append(None)                                  # stream idle this step
                continue
            o = scenes[s].step()
            if (f + s) % 13 == 6:
                o["embs"], o["bboxes"], o["confs"] = [], [], []    # empty frame
            objs.append(o)
        dets, embs, sidx, rows = _frame(objs, rng)
        active = np.array([o is not None for o in objs], np.int32)
        frame = torch.full((S,), f, dtype=torch.int32, device="cuda")
        d = _dev(dets)
        _, tod = packed.step_detections(d[:, :4], d[:, 4], _dev(embs), frame, _dev(sidx), active=_dev(active),
                                        result=res_a[f])
        n_det = np.where(active == 1, [len(r) for r in rows], -1).astype(np.int32)
        boxes, confs, e = np.zeros((S, MD, 4)), np.zeros((S, MD)), np.zeros((S, MD, 128), np.float32)
        for s, r in enumerate(rows):
            boxes[s, :len(r)], confs[s, :len(r)], e[s, :len(r)] = dets[r, :4], dets[r, 4], embs[r]
        padded.step_device(_dev(n_det), _dev(boxes), _dev(confs), _dev(e), frame, res_b[f])
        _check_track_of_det(packed, res_a[f].cpu().numpy(), tod.cpu().numpy(), rows)
        if f in (17, F - 1):
            for s in range(S):
                a, b = packed.export(s), padded.export(s)
                assert a["next_id"] == b["next_id"]
                for k in STATE_KEYS:
                    assert np.array_equal(a[k], b[k], equal_nan=True), (f, s, k)
    assert torch.equal(res_a, res_b)
    assert (res_a[:, :, R_STATUS] == 0).all()


@pytest.mark.parametrize("half,rows_layout", [(False, True), (False, False), (True, True)])
def test_packed_step_vs_oracle(half, rows_layout):
    """The oracle is fed the values the detector emitted (float32- or float16-rounded) in each stream's input order;
    boxes and confidences come as views of the detector's [K, 6] rows or as separate contiguous tensors."""
    S, F, MD, hw = 3, 30, 48, (1088, 1920)
    ms = MultiStreamTracker(S, CFG, max_tracks=128, max_dets=MD)
    refs = [tracker_ref.TrackerRef(CFG) for _ in range(S)]
    scenes = _scenes(S, 70)
    rng = np.random.default_rng(5)
    for f in range(F):
        objs = [sc.step() for sc in scenes]
        dets, embs, sidx, rows = _frame(objs, rng, half=half)
        d = _dev(dets)
        boxes, confs = (d[:, :4], d[:, 4]) if rows_layout else (d[:, :4].contiguous(), d[:, 4].contiguous())
        table, tod = ms.step_detections(boxes, confs, _dev(embs), torch.full((S,), f, dtype=torch.int32, device="cuda"),
                                        _dev(sidx))
        table = table.cpu().numpy()
        want_tod = np.full(len(sidx), -1)
        for s in range(S):
            want = refs[s].update(_oracle_obj(dets, embs, rows[s], f, hw))
            assert ms.decode(table[s]) == tuple(want), (f, s)
            for tid, j in want[0]:
                want_tod[rows[s][j]] = tid
        assert tod.cpu().numpy().tolist() == want_tod.tolist(), f
    for s in range(S):
        assert ms.export(s)["ids"].tolist() == sorted(refs[s].tracks)


def _idle_row(row, n_live, next_id, status=0):
    assert row[:8].tolist() == [0, 0, 0, n_live, next_id, status, 0, 0]


def test_packed_step_edge_cases():
    """K = 0 (misses advance, no predict), rows with a stream index outside [0, S) (ignored, -1), active = 0 (idle row,
    state untouched), a stream with max_dets + 1 detections (ECAPACITY, state untouched, the others step normally),
    stream_index = None on a one-stream handle."""
    S, MD, hw = 3, 24, (1088, 1920)
    ms = MultiStreamTracker(S, CFG, max_tracks=96, max_dets=MD)
    refs = [tracker_ref.TrackerRef(CFG) for _ in range(S)]
    scenes = [synth.Scene(90 + s, 12 + 3 * s, 1088, 1920, drop=0.1) for s in range(S)]
    rng = np.random.default_rng(9)

    def state(s):
        return ms.export(s)

    def same_state(a, b):
        assert a["next_id"] == b["next_id"] and all(np.array_equal(a[k], b[k], equal_nan=True) for k in STATE_KEYS)

    for f in range(12):
        objs = [sc.step() for sc in scenes]
        if f == 6:
            objs = [dict(o, embs=[], bboxes=[], confs=[]) for o in objs]        # K = 0 below
        active = np.ones(S, np.int32)
        if f == 4:
            active[1] = 0
        if f == 8:                                                               # stream 2 over capacity
            o = objs[2]
            extra = MD + 1 - len(o["bboxes"])
            eb = synth.random_boxes(rng, extra, 1088, 1920)
            o["bboxes"] = o["bboxes"] + eb.tolist()
            o["confs"] = o["confs"] + [0.9] * extra
            o["embs"] = o["embs"] + [rng.standard_normal(128).astype(np.float32) for _ in range(extra)]
        dets, embs, sidx, rows = _frame(objs, rng, junk=0 if f == 6 else 3)
        if f == 6:
            assert len(dets) == 0
        before = [state(s) for s in range(S)] if f in (4, 8) else None
        d = _dev(dets).reshape(-1, 6)
        table, tod = ms.step_detections(d[:, :4], d[:, 4], _dev(embs).reshape(-1, 128),
                                        torch.full((S,), f, dtype=torch.int32, device="cuda"), _dev(sidx),
                                        active=_dev(active))
        table, tod = table.cpu().numpy(), tod.cpu().numpy()
        want_tod = np.full(len(sidx), -1)
        for s in range(S):
            if f == 4 and s == 1:
                _idle_row(table[s], len(refs[s].tracks), refs[s].next_id)
                same_state(state(s), before[s])
                continue
            if f == 8 and s == 2:
                _idle_row(table[s], len(refs[s].tracks), refs[s].next_id, _lib.ECAPACITY)
                same_state(state(s), before[s])
                continue
            want = refs[s].update(_oracle_obj(dets, embs, rows[s], f, hw))
            assert ms.decode(table[s]) == tuple(want), (f, s)
            assert int(table[s, R_STATUS]) == 0
            for tid, j in want[0]:
                want_tod[rows[s][j]] = tid
        assert tod.tolist() == want_tod.tolist(), f
        assert all(tod[k] == -1 for k in range(len(sidx)) if not 0 <= sidx[k] < S)
        if f == 6:                                  # empty frame: every track missed, Kalman state not predicted
            for s in range(S):
                ids, snap = sorted(refs[s].tracks), state(s)
                assert snap["miss"].tolist() == [refs[s].tracks[i].miss_count for i in ids]
                assert_close(snap["x"], np.array([refs[s].tracks[i].kf.x.reshape(-1) for i in ids]).reshape(-1, 8),
                             what="x after the empty frame")
    for s in range(S):
        ids = sorted(refs[s].tracks)
        snap = state(s)
        assert snap["ids"].tolist() == ids and snap["next_id"] == refs[s].next_id
        assert snap["miss"].tolist() == [refs[s].tracks[i].miss_count for i in ids]

    one = MultiStreamTracker(1, CFG, max_tracks=64, max_dets=16)
    ref = tracker_ref.TrackerRef(CFG)
    sc = synth.Scene(7, 9, 720, 1280)
    for f in range(6):
        dets, embs, sidx, rows = _frame([sc.step()], rng)
        d = _dev(dets)
        table, tod = one.step_detections(d[:, :4], d[:, 4], _dev(embs), torch.full((1,), f, dtype=torch.int32, device="cuda"))
        want = ref.update(_oracle_obj(dets, embs, rows[0], f, (720, 1280)))
        assert one.decode(table[0].cpu().numpy()) == tuple(want)
        _check_track_of_det(one, table.cpu().numpy(), tod.cpu().numpy(), rows)


def test_step_detections_argument_errors():
    ms = MultiStreamTracker(2, CFG, max_tracks=32, max_dets=8)
    K = 4
    d = torch.zeros((K, 6), device="cuda")
    e = torch.zeros((K, 128), device="cuda")
    fr = torch.zeros(2, dtype=torch.int32, device="cuda")
    with pytest.raises(TypeError):
        ms.step_detections(d[:, :4].double(), d[:, 4].double(), e, fr)
    with pytest.raises(TypeError):
        ms.step_detections(d[:, :4], d[:, 4].half(), e, fr)
    with pytest.raises(TypeError):
        ms.step_detections(d[:, :4], d[:, 4], e.t().contiguous().t(), fr)
    with pytest.raises(TypeError):
        ms.step_detections(d[:, :4], d[:, 4], e, fr, torch.zeros(K, dtype=torch.int64, device="cuda"))
    with pytest.raises(ValueError):
        ms.step_detections(d[:, :3], d[:, 4], e, fr)
    with pytest.raises(ValueError):
        ms.step_detections(d[:, :4], d[:3, 4], e, fr)
    with pytest.raises(ValueError):
        ms.step_detections(d[:, :4], d[:, 4], e[:, :64], fr)
    with pytest.raises(ValueError):
        ms.step_detections(d[:, :4], d[:, 4], e, fr[:1])
    lib = _lib.lib()
    rc = lib.b200_tracker_step_packed(ms._h, K, _lib.ptr(d), 4, _lib.ptr(d), 6, 7, _lib.ptr(e), 0, None, None,
                                      _lib.ptr(fr), None, None, None)
    assert rc == _lib.EINVAL and b"det_dtype" in lib.b200_last_error()
    rc = lib.b200_tracker_step_packed(ms._h, K, _lib.ptr(d), 3, _lib.ptr(d), 6, 0, _lib.ptr(e), 0, None, None,
                                      _lib.ptr(fr), None, None, None)
    assert rc == _lib.EINVAL and b"box_stride" in lib.b200_last_error()
    rc = lib.b200_tracker_step_packed(ms._h, -1, None, 4, None, 1, 0, None, 0, None, None, _lib.ptr(fr), None, None, None)
    assert rc == _lib.EINVAL and b"K" in lib.b200_last_error()


@pytest.mark.parametrize("half,max_tracks,max_dets", [(False, 512, 256), (False, 32, 16), (True, 32, 16)])
def test_update_tensors_equals_update(half, max_tracks, max_dets):
    """Tracking.update_tensors from device tensors returns exactly Tracking.update's tuple for the same (emitted)
    values; a handle of max_dets = 16 against 64-detection c2 frames grows on the way."""
    Hf, Wf, H_in, W_in, n = synth.CONFIGS["c2"]
    a = Tracking(conf=SHIPPED_CONF, max_tracks=max_tracks, max_dets=max_dets)
    b = Tracking(conf=SHIPPED_CONF, max_tracks=512, max_dets=256)
    scene = synth.Scene(11, n, H_in, W_in, drop=0.1, churn=0.1, churn_every=8)
    rng = np.random.default_rng(2)
    for f in range(30):
        obj = scene.step()
        if f == 12:
            obj["embs"], obj["bboxes"], obj["confs"] = [], [], []
        dets, embs, _, rows = _frame([obj], rng, half=half)
        d = _dev(dets).reshape(-1, 6)
        got = a.update_tensors(d[:, :4], d[:, 4], _dev(embs).reshape(-1, 128), f)
        assert got == b.update(_oracle_obj(dets, embs, rows[0], f, (H_in, W_in))), f
    assert a._ms.max_dets >= n and (max_tracks == 512 or a._ms.max_tracks > max_tracks)
    sa, sb = a.snapshot(), b.snapshot()
    assert sa["next_id"] == sb["next_id"] and all(np.array_equal(sa[k], sb[k], equal_nan=True) for k in STATE_KEYS)
    with pytest.raises(ValueError):
        a.update_tensors(d[:, :4], d[:-1, 4], _dev(embs), 99)
    with pytest.raises(ValueError):
        a.update_tensors(d[:, :4], d[:, 4], _dev(embs)[:, :64], 99)


def test_handoff_replays_as_cuda_graph():
    """Detector rows -> box prep + ROI Align over S maps -> a matmul standing in for the encoder -> step_detections,
    captured once; per frame only the detector rows and the frame ids are copied in (the stream indices are static)."""
    Hf, Wf, H_in, W_in, n = synth.CONFIGS["c2"]
    S, C, MD = 2, 128, 64
    dev = torch.device("cuda", 0)
    ms = MultiStreamTracker(S, SHIPPED_CONF, max_tracks=192, max_dets=MD, device=dev)
    refs = [tracker_ref.TrackerRef(SHIPPED_CONF) for _ in range(S)]
    scenes = [synth.Scene(30 + s, n, H_in, W_in) for s in range(S)]            # no drops: K is fixed at S * n
    K = S * n
    rng = np.random.default_rng(4)
    sidx_np = rng.permutation(np.repeat(np.arange(S, dtype=np.int32), n))
    rows = [np.nonzero(sidx_np == s)[0].tolist() for s in range(S)]
    feat = torch.from_numpy(synth.feature_map(2, S, C, Hf, Wf)).to(dev)
    proj = torch.randn((C * 100, 128), device=dev, generator=torch.Generator(device=dev).manual_seed(0)) * 0.01
    dets = torch.zeros((K, 6), device=dev)
    sidx = torch.from_numpy(sidx_np).to(dev)
    frame = torch.zeros(S, dtype=torch.int32, device=dev)
    active = torch.zeros(S, dtype=torch.int32, device=dev)            # warm-up: every stream idle, state untouched
    result = torch.zeros((S, ms.stride), dtype=torch.int32, device=dev)
    tod = torch.zeros(K, dtype=torch.int32, device=dev)

    def frame_sequence():
        patches = roi.roi_align_from_input_boxes(feat, dets, (H_in, W_in), out_size=(10, 10), batch_index=sidx)
        emb = patches.reshape(K, -1) @ proj                                   # "encoder" (card.py:24-41)
        ms.step_detections(dets[:, :4], dets[:, 4], emb, frame, sidx, active=active, result=result, track_of_det=tod)
        return emb

    side = torch.cuda.Stream(dev)
    side.wait_stream(torch.cuda.current_stream(dev))
    with torch.cuda.stream(side):
        frame_sequence()
    torch.cuda.current_stream(dev).wait_stream(side)
    torch.cuda.synchronize(dev)
    assert all(len(ms.export(s)["ids"]) == 0 for s in range(S))
    active.fill_(1)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        emb = frame_sequence()
    n_matched = 0
    for f in range(12):
        objs = [sc.step() for sc in scenes]
        d = np.zeros((K, 6), np.float32)
        for s in range(S):
            d[rows[s], :4], d[rows[s], 4] = objs[s]["bboxes"], objs[s]["confs"]
        dets.copy_(torch.from_numpy(d))
        frame.fill_(f)
        graph.replay()
        torch.cuda.synchronize(dev)
        e = emb.cpu().numpy()
        table = result.cpu().numpy()
        want_tod = np.full(K, -1)
        for s in range(S):
            want = refs[s].update(_oracle_obj(d, e, rows[s], f, (H_in, W_in)))
            assert ms.decode(table[s]) == tuple(want), (f, s)
            for tid, j in want[0]:
                want_tod[rows[s][j]] = tid
        assert tod.cpu().numpy().tolist() == want_tod.tolist(), f
        n_matched += int((want_tod >= 0).sum())
    assert n_matched > 0
