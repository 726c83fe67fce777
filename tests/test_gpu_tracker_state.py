"""GPU: the tracker state as a device-side image (state_dict / load_state_dict, per-stream reset, device-side growth).

Scenes with drops, churn, ReID rows and purges run for more frames than hist_max, so bank rings have wrapped before an
image is taken.  Every comparison between two handles is bit for bit."""
import ctypes
import io

import numpy as np
import pytest
import torch

from oracle import tracker_ref

pytestmark = pytest.mark.gpu

import alufe_b200  # noqa: E402,F401
from alufe_b200 import MultiStreamTracker, SHIPPED_CONF, Tracking, synth  # noqa: E402
from alufe_b200 import _lib  # noqa: E402

CFG = dict(SHIPPED_CONF, hist_max=5, lost_reid_after=3, max_age=8)
MD = 32


def _streams(S, seed, n_frames):
    """Per stream, a list of frames: an obj dict, or None when the stream is idle that step."""
    out = []
    for s in range(S):
        sc = synth.Scene(seed + s, 6 + 3 * s, 1088, 1920, drop=0.25, churn=0.2, churn_every=5)
        out.append([None if (f + s) % 9 == 4 else sc.step() for f in range(n_frames)])
    return out


def _arrays(objs, f):
    S = len(objs)
    n_det = np.full(S, -1, np.int32)
    boxes, confs, embs = np.zeros((S, MD, 4)), np.zeros((S, MD)), np.zeros((S, MD, 128), np.float32)
    for s, obj in enumerate(objs):
        if obj is None:
            continue
        n = n_det[s] = len(obj["bboxes"])
        if n:
            boxes[s, :n], confs[s, :n], embs[s, :n] = obj["bboxes"], obj["confs"], np.stack(obj["embs"])
    return n_det, boxes, confs, embs, np.full(S, f, np.int32)


def _step(ms, frames, f):
    """Steps ms on frame f of every stream; returns the decoded rows plus each row's header."""
    res = ms.step(*_arrays([fr[f] for fr in frames], f))
    return [(ms.decode(r), r[:8].tolist()) for r in res]


def _same(a, b, what=""):
    assert a["next_id"] == b["next_id"], what
    for k in a:
        if k != "next_id":
            assert a[k].dtype == b[k].dtype and a[k].shape == b[k].shape and a[k].tobytes() == b[k].tobytes(), (what, k)


def _exports(ms):
    return [ms.export(s) for s in range(ms.S)]


def _row(sd, r):
    """Row r of an image in export()'s form (host arrays cut at n_live)."""
    n = int(sd["n_live"][r])
    out = {k: v[r, :n].cpu().numpy() for k, v in sd.items() if k not in ("n_live", "next_id")}
    out["next_id"] = int(sd["next_id"][r])
    return out


def _c_call(ms, fn, sd, streams=None, status=None):
    im = ms._c_image(sd)
    return getattr(_lib.lib(), fn)(ms._h, _lib.ptr(streams), ctypes.byref(im), _lib.ptr(status),
                                   _lib.stream_ptr(ms.device))


@pytest.mark.parametrize("chain", ["2", "3", "6"])
def test_state_dict_equals_export_and_loads_bit_identically(chain, monkeypatch):
    monkeypatch.setenv("B200TRACK_CHAIN", chain)
    S, MT = 6, 96
    frames = _streams(S, 40, 32)
    src = MultiStreamTracker(S, CFG, max_tracks=MT, max_dets=MD)
    for f in range(20):
        _step(src, frames, f)
    sd = src.state_dict()
    torch.cuda.synchronize()
    n = sd["n_live"].cpu().numpy()
    assert n.min() > 0
    for s, e in enumerate(_exports(src)):
        _same(_row(sd, s), e, "stream %d" % s)
        for k, v in sd.items():
            if k not in ("n_live", "next_id"):
                assert not v[s, n[s]:].any(), (k, s)                 # slots past n_live stay zero
    small = int(n.max()) + MD
    assert small < MT
    loaded = []
    for cap in (2 * MT, small):
        dst = MultiStreamTracker(S, CFG, max_tracks=cap, max_dets=MD)
        dst.load_state_dict(sd)
        assert dst.max_tracks == cap and (dst.n_live == n).all()
        for s, (a, b) in enumerate(zip(_exports(dst), _exports(src))):
            _same(a, b, "loaded stream %d" % s)
        loaded.append(dst)
    for f in range(20, 32):
        want = _step(src, frames, f)
        for dst in loaded:
            assert _step(dst, frames, f) == want, "frame %d, max_tracks %d" % (f, dst.max_tracks)
    for dst in loaded:
        for s, (a, b) in enumerate(zip(_exports(dst), _exports(src))):
            _same(a, b, "stream %d after 12 frames" % s)


def test_grow_matches_the_host_round_trip_and_the_oracle():
    S, MT = 4, 40
    frames = _streams(S, 50, 30)
    a = MultiStreamTracker(S, CFG, max_tracks=MT, max_dets=MD)
    b = MultiStreamTracker(S, CFG, max_tracks=MT, max_dets=MD)
    refs = [tracker_ref.TrackerRef(CFG) for _ in range(S)]

    def step_all(f):
        got_a, got_b = _step(a, frames, f), _step(b, frames, f)
        assert got_a == got_b, "frame %d" % f
        for s in range(S):
            if frames[s][f] is not None:
                want = refs[s].update(frames[s][f])
                assert got_a[s][0] == (want[0], want[1], want[2]), (f, s)
                assert got_a[s][1][3] == len(refs[s].tracks) and got_a[s][1][4] == refs[s].next_id

    for f in range(15):
        step_all(f)
    n_live, stale = a.n_live.copy(), a._n_live_stale
    a.grow(max_tracks=2 * MT)
    assert a.max_tracks == 2 * MT and (a.n_live == n_live).all() and a._n_live_stale == stale
    snaps = [b.export(s) for s in range(S)]              # the host round trip grow() used to make
    old = b._h
    b._create(2 * MT, MD)
    _lib.lib().b200_tracker_destroy(old)
    for s, snap in enumerate(snaps):
        b.import_state(s, snap)
    for s, (x, y) in enumerate(zip(_exports(a), _exports(b))):
        _same(x, y, "grown stream %d" % s)
    for f in range(15, 30):
        step_all(f)
    for s, (x, y) in enumerate(zip(_exports(a), _exports(b))):
        _same(x, y, "stream %d" % s)


def test_import_state_loads_like_load_state_dict_and_refuses_malformed_snapshots():
    """import_state (host arrays, b200_tracker_import) goes through the device import: a valid snapshot lands exactly as
    load_state_dict of the same row does, and a snapshot the row check rejects raises and leaves the stream as it was."""
    S, H = 3, CFG["hist_max"]
    frames = _streams(S, 170, 30)
    src = MultiStreamTracker(S, CFG, max_tracks=64, max_dets=MD)
    a = MultiStreamTracker(S, CFG, max_tracks=64, max_dets=MD)
    b = MultiStreamTracker(S, CFG, max_tracks=64, max_dets=MD)
    for f in range(20):
        _step(src, frames, f)
        if f < 8:
            _step(a, frames, f)
            _step(b, frames, f)
    snap = src.export(2)
    assert len(snap["ids"]) >= 2 and (snap["bank_len"] == H).any()      # 20 frames at hist_max 5: full, wrapped rings
    a.import_state(1, snap)
    b.load_state_dict(src.state_dict([2]), streams=[1])
    assert a.n_live[1] == b.n_live[1] == len(snap["ids"])
    _same(a.export(1), snap, "imported")
    for s, (x, y) in enumerate(zip(_exports(a), _exports(b))):
        _same(x, y, "stream %d" % s)
    moved = [frames[0], frames[2], frames[1]]
    for f in range(20, 30):
        got_a, want = _step(a, moved, f), _step(src, frames, f)
        assert got_a == _step(b, moved, f) and got_a[1] == want[2], "frame %d" % f

    before, n_before = a.export(0), int(a.n_live[0])

    def bad(**edit):
        out = {k: (v.copy() if isinstance(v, np.ndarray) else v) for k, v in snap.items()}
        for k, (i, v) in edit.items():
            out[k][i] = v
        return out

    ids, next_id = snap["ids"], snap["next_id"]
    cases = {"unsorted ids": bad(ids=(slice(0, 2), ids[1::-1])), "negative id": bad(ids=(0, -1)),
             "id not below next_id": bad(ids=(-1, next_id)), "bank_len above hist_max": bad(bank_len=(0, H + 1)),
             "negative bank_len": bad(bank_len=(0, -1)), "stage above 2": bad(stage=(1, 3))}
    for what, snap_bad in cases.items():
        with pytest.raises(ValueError, match="malformed state"):
            a.import_state(0, snap_bad)
        _same(a.export(0), before, what)
        assert a.n_live[0] == n_before, what

    empty = MultiStreamTracker(1, CFG, max_tracks=8, max_dets=MD).export(0)     # no tracks: a one-slot image
    empty["next_id"] = 7
    a.import_state(2, empty)
    _same(a.export(2), empty, "empty")
    assert a.n_live[2] == 0


def test_grow_keeps_the_old_handle_when_creation_fails():
    ms = MultiStreamTracker(2, CFG, max_tracks=16, max_dets=MD)
    frames = _streams(2, 70, 8)
    for f in range(8):
        _step(ms, frames, f)
    before, h, mt = _exports(ms), ms._h.value, ms.max_tracks
    with pytest.raises(ValueError):
        ms.grow(max_tracks=100000)                      # beyond tracker_create's limit
    assert ms._h.value == h and ms.max_tracks == mt
    for x, y in zip(_exports(ms), before):
        _same(x, y)


def test_move_one_stream_between_handles():
    frames_a, frames_b = _streams(4, 80, 30), _streams(3, 90, 30)
    A = MultiStreamTracker(4, CFG, max_tracks=64, max_dets=MD)
    B = MultiStreamTracker(3, CFG, max_tracks=48, max_dets=MD)
    for f in range(18):
        _step(A, frames_a, f)
        _step(B, frames_b, f)
    B.load_state_dict(A.state_dict([3]), streams=[0])
    _same(B.export(0), A.export(3), "moved")
    assert B.n_live[0] == A.n_live_now()[3]
    C = MultiStreamTracker(3, CFG, max_tracks=48, max_dets=MD)    # B's other streams, never touched by the move
    for f in range(18):
        _step(C, frames_b, f)
    for s in (1, 2):
        _same(B.export(s), C.export(s), "untouched stream %d" % s)
    moved = [frames_a[3]] + frames_b[1:]
    for f in range(18, 30):
        got_a, got_b, got_c = _step(A, frames_a, f), _step(B, moved, f), _step(C, frames_b, f)
        assert got_b[0] == got_a[3] and got_b[1:] == got_c[1:], "frame %d" % f
    _same(B.export(0), A.export(3))


def test_reset_some_streams_vs_oracle():
    S = 5
    frames = _streams(S, 100, 30)
    ms = MultiStreamTracker(S, CFG, max_tracks=64, max_dets=MD)
    refs = [tracker_ref.TrackerRef(CFG) for _ in range(S)]

    def step_all(f):
        got = _step(ms, frames, f)
        for s in range(S):
            if frames[s][f] is not None:
                want = refs[s].update(frames[s][f])
                assert got[s][0] == (want[0], want[1], want[2]), (f, s)
                assert got[s][1][3] == len(refs[s].tracks) and got[s][1][4] == refs[s].next_id

    for f in range(15):
        step_all(f)
    before = _exports(ms)
    ms.reset(streams=[1, 3])
    after = _exports(ms)
    for s in range(S):
        if s in (1, 3):
            assert len(after[s]["ids"]) == 0 and after[s]["next_id"] == 0 and ms.n_live[s] == 0
        else:
            _same(after[s], before[s], "stream %d" % s)
    refs[1], refs[3] = tracker_ref.TrackerRef(CFG), tracker_ref.TrackerRef(CFG)
    for f in range(15, 30):
        step_all(f)
    with pytest.raises(ValueError):
        ms.reset(streams=[2, 2])
    with pytest.raises(ValueError):
        ms.reset(streams=[S])


def test_capacity_on_load():
    frames = _streams(4, 110, 12)[3:]                            # a scene of 15 objects
    src = MultiStreamTracker(1, CFG, max_tracks=64, max_dets=MD)
    for f in range(12):
        _step(src, frames, f)
    sd = src.state_dict()
    n = int(sd["n_live"][0])
    assert n > 8
    fixed = MultiStreamTracker(1, CFG, max_tracks=8, max_dets=MD, auto_grow=False)
    _step(fixed, _streams(1, 120, 2), 0)
    before = fixed.export(0)
    with pytest.raises(_lib.B200Error):
        fixed.load_state_dict(sd)
    assert fixed.max_tracks == 8
    _same(fixed.export(0), before, "unchanged")
    grows = MultiStreamTracker(1, CFG, max_tracks=8, max_dets=MD)
    grows.load_state_dict(sd)
    assert grows.max_tracks >= n
    _same(grows.export(0), src.export(0), "grown on load")


def test_malformed_rows_are_skipped_and_reported():
    S = 8
    frames = _streams(S, 130, 14)
    src = MultiStreamTracker(S, CFG, max_tracks=64, max_dets=MD)
    dst = MultiStreamTracker(S, CFG, max_tracks=64, max_dets=MD)
    for f in range(14):
        _step(src, frames, f)
        if f < 7:
            _step(dst, frames, f)
    sd = src.state_dict()
    torch.cuda.synchronize()
    assert int(sd["n_live"].min()) >= 2
    before = _exports(dst)
    sd["ids"][1, :2] = sd["ids"][1, :2].flip(0)                  # unsorted ids
    sd["bank_len"][2, 0] = CFG["hist_max"] + 1
    sd["stage"][3, 1] = 3
    sd["n_live"][4] = -1
    sd["n_live"][6] = sd["ids"].shape[1] + 1                     # more than cap
    streams = torch.tensor([0, 1, 2, 3, 4, 5, 6, 99], dtype=torch.int32, device="cuda")
    status = torch.full((S,), 7, dtype=torch.int32, device="cuda")
    assert _c_call(dst, "b200_tracker_import_device", sd, streams, status) == _lib.OK
    E, C = _lib.EINVAL, _lib.ECAPACITY
    assert status.cpu().tolist() == [0, E, E, E, E, 0, C, E]
    after = _exports(dst)
    for s in range(S):
        if s in (0, 5):
            _same(after[s], src.export(s), "applied %d" % s)
        else:
            _same(after[s], before[s], "skipped %d" % s)
    # export: a row whose stream has more live tracks than the image's cap, and an out-of-range stream
    small = src._new_image(2, 1)
    st = torch.full((2,), 7, dtype=torch.int32, device="cuda")
    assert _c_call(src, "b200_tracker_export_device", small, torch.tensor([0, -1], dtype=torch.int32, device="cuda"),
                   st) == _lib.OK
    assert st.cpu().tolist() == [C, E] and not any(v.any() for v in small.values())
    # host-side errors against a live handle
    other = src._new_image(S, 4)
    other["bank"] = torch.zeros((S, 4, CFG["hist_max"] + 1, 128), device="cuda")
    assert _c_call(dst, "b200_tracker_import_device", other) == _lib.EINVAL
    assert b"hist_max" in _lib.lib().b200_last_error()
    assert _c_call(dst, "b200_tracker_export_device", src._new_image(S - 1, 4)) == _lib.EINVAL
    assert b"n_rows == n_streams" in _lib.lib().b200_last_error()
    with pytest.raises(ValueError):
        dst.load_state_dict(other)
    with pytest.raises(ValueError):
        dst.load_state_dict(src.state_dict([0, 1]), streams=[3, 3])
    with pytest.raises(ValueError):
        dst.state_dict([S])


def test_torch_save_round_trip():
    S = 3
    frames = _streams(S, 140, 22)
    a = MultiStreamTracker(S, CFG, max_tracks=64, max_dets=MD)
    for f in range(14):
        _step(a, frames, f)
    buf = io.BytesIO()
    torch.save({k: v.cpu() for k, v in a.state_dict().items()}, buf)
    buf.seek(0)
    b = MultiStreamTracker(S, CFG, max_tracks=64, max_dets=MD)
    b.load_state_dict(torch.load(buf))
    for s, (x, y) in enumerate(zip(_exports(a), _exports(b))):
        _same(x, y, "restored %d" % s)
    for f in range(14, 22):
        assert _step(a, frames, f) == _step(b, frames, f), "frame %d" % f
    for x, y in zip(_exports(a), _exports(b)):
        _same(x, y)


def test_state_dict_replays_as_cuda_graph():
    S = 4
    frames = _streams(S, 150, 20)
    ms = MultiStreamTracker(S, CFG, max_tracks=64, max_dets=MD)
    for f in range(8):
        _step(ms, frames, f)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        ms.state_dict()                                  # warm-up outside the capture
    torch.cuda.current_stream().wait_stream(side)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        sd = ms.state_dict()
    for f in range(8, 20):
        _step(ms, frames, f)
    g.replay()
    torch.cuda.synchronize()
    for s, e in enumerate(_exports(ms)):
        _same(_row(sd, s), e, "replayed %d" % s)


def test_tracking_state_dict_continues_like_the_oracle():
    ref = tracker_ref.TrackerRef(CFG)
    trk = Tracking(conf=CFG, max_tracks=32, max_dets=16)
    scene = synth.Scene(160, 22, 1280, 1280, drop=0.2, churn=0.2, churn_every=6)
    for f in range(15):
        obj = scene.step()
        assert trk.update(obj) == ref.update(obj), "frame %d" % f
    trk.tracks                                          # fills the snapshot cache that loading must drop
    sd = trk.state_dict()
    fresh = Tracking(conf=CFG, max_tracks=8, max_dets=4)
    fresh.load_state_dict(sd)
    assert fresh._ms.max_tracks >= 8 and sorted(fresh.tracks) == sorted(ref.tracks) and fresh.next_id == ref.next_id
    trk.load_state_dict(sd)                             # loading into itself changes nothing
    for f in range(15, 30):
        obj = scene.step()
        want = ref.update(obj)
        assert fresh.update(obj) == want and trk.update(obj) == want, "frame %d" % f
    assert sorted(fresh.tracks) == sorted(ref.tracks) and fresh.next_id == ref.next_id
