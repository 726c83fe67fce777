"""GPU parity of the fused, GPU-resident tracker (Tracking.update) against the golden traces of
the live reference and against the oracle tracker on larger synthetic scenes."""
import numpy as np
import torch
import pytest

from conftest import assert_close, load_golden
from oracle import tracker_ref

pytestmark = pytest.mark.gpu

import alufe_b200  # noqa: E402,F401
from alufe_b200 import Tracking, MultiStreamTracker, SHIPPED_CONF, synth  # noqa: E402
from alufe_b200 import _lib  # noqa: E402


def _compare_state(trk, want_ids, want, what):
    """want: dict with x, P, ema, bank (list per track), miss, age, last_bbox."""
    s = trk.snapshot()
    assert s["ids"].tolist() == list(want_ids), what
    assert_close(s["x"], want["x"], rtol=1e-5, atol=1e-6, what=what + " x")
    assert_close(s["P"], want["P"], rtol=1e-5, atol=1e-5, what=what + " P")
    assert_close(s["ema"], want["ema"], rtol=1e-5, atol=1e-6, what=what + " ema")
    assert s["miss"].tolist() == list(want["miss"]), what
    assert s["age"].tolist() == list(want["age"]), what
    assert_close(s["last_bbox"], want["last_bbox"], rtol=1e-5, atol=1e-5, what=what + " last_bbox")
    assert s["bank_len"].tolist() == [len(b) for b in want["bank"]], what
    for r, b in enumerate(want["bank"]):
        if len(b):
            assert_close(s["bank"][r, :len(b)], np.stack(b), rtol=1e-5, atol=1e-6, what=what + " bank")


@pytest.mark.parametrize("name", ["c1_steady", "churn"])
def test_tracker_vs_golden_reference_trace(name):
    g = load_golden("tracker_" + name)
    cfg = dict(SHIPPED_CONF)
    for k in g.files:
        if k.startswith("cfg_"):
            cfg[k[4:]] = int(g[k]) if k[4:] in ("lost_reid_after", "max_age", "hist_max") else float(g[k])
    trk = Tracking(conf=cfg, max_tracks=64, max_dets=32)
    for f in range(int(g["n_frames"])):
        p = "f%03d_" % f
        obj = {"embs": [e for e in g[p + "embs"]], "bboxes": g[p + "boxes"].tolist(), "confs": g[p + "confs"].tolist(),
               "input_hw": (int(g["H"]), int(g["W"])), "frame_id": f}
        m, ut, ud = trk.update(obj)
        assert np.array_equal(np.array(m, dtype=np.int64).reshape(-1, 2), g[p + "matches"]), p
        assert ut == g[p + "unmatched_tracks"].tolist(), p
        assert ud == g[p + "unmatched_dets"].tolist(), p
        if p + "st_ids" in g:
            n = g[p + "st_bank_len"]
            want = dict(x=g[p + "st_x"], P=g[p + "st_P"], ema=g[p + "st_ema"], miss=g[p + "st_miss"].tolist(),
                        age=g[p + "st_age"].tolist(), last_bbox=g[p + "st_last_bbox"],
                        bank=[list(g[p + "st_bank"][r, :n[r]]) for r in range(len(n))])
            _compare_state(trk, g[p + "st_ids"].tolist(), want, p)
            assert trk.next_id == int(g[p + "st_next_id"])
            s = trk.snapshot()
            assert (s["stage"] == g[p + "st_x_is64"].astype(int) + g[p + "st_P_is64"].astype(int)).all()


def _oracle_state(ref):
    ids = sorted(ref.tracks)
    T = [ref.tracks[i] for i in ids]
    return ids, dict(x=np.array([t.kf.x.reshape(-1) for t in T], dtype=np.float64).reshape(-1, 8),
                     P=np.array([t.kf.P for t in T], dtype=np.float64).reshape(-1, 8, 8),
                     ema=np.array([t.ema for t in T], dtype=np.float32).reshape(-1, 128),
                     miss=[t.miss_count for t in T], age=[t.age for t in T],
                     last_bbox=np.array([t.last_bbox for t in T], dtype=np.float64).reshape(-1, 4),
                     bank=[t.bank for t in T])


@pytest.mark.parametrize("case", [
    dict(n=64, H=1280, W=1280, frames=45, scene={}, conf={}),                                   # BASELINE config 2
    dict(n=40, H=1280, W=1280, frames=70, scene=dict(drop=0.3, churn=0.15, churn_every=9),
         conf=dict(lost_reid_after=4, max_age=12, hist_max=8), empty=(20, 21, 50)),
    dict(n=128, H=1088, W=1920, frames=12, scene=dict(drop=0.1), conf={}),                      # config 5 stream
    dict(n=24, H=640, W=640, frames=40, scene=dict(drop=0.5, churn=0.3, churn_every=5),
         conf=dict(lost_reid_after=2, max_age=6, hist_max=3, emb_top_k=2, conf_update_min=0.7)),
    # banks deeper than 32 rows use the L2-resident variant of the stage-1 cost kernel
    dict(n=20, H=640, W=640, frames=52, scene=dict(drop=0.15, churn=0.1, churn_every=11),
         conf=dict(hist_max=44, emb_top_k=7, lost_reid_after=6, max_age=20)),
    # a crowd: 256 detections per frame, births and misses every frame (BASELINE config 4 is 512)
    dict(n=256, H=1280, W=1280, frames=5, scene=dict(drop=0.08), conf={}),
    # BASELINE config 4 as a tracker: ~512 detections x ~512+ tracks with drops and churn, so births, misses, ReID
    # rows and contested assignment rows all go through the 8-warp register solver fed by the cost kernel's row
    # summaries (the path only shapes above 256 columns take)
    dict(n=512, H=1280, W=1280, frames=12, scene=dict(drop=0.1, churn=0.1, churn_every=4),
         conf=dict(lost_reid_after=3, max_age=8), every=3),
])
@pytest.mark.parametrize("chain", ["2", "3", "6"])
def test_tracker_vs_oracle(case, chain, monkeypatch):
    """All device paths of the step: the two-launch chain (few streams), the three-launch chain (stream groups) -- both
    for handles of at most 512 tracks x 256 detections -- and the six-kernel chain that larger handles use (each forced
    with B200TRACK_CHAIN)."""
    cfg = dict(SHIPPED_CONF, **case["conf"])
    if chain != "6" and case["n"] > 128:
        pytest.skip("crowds need more than 512 track slots: six-kernel chain only")
    monkeypatch.setenv("B200TRACK_CHAIN", chain)
    ref = tracker_ref.TrackerRef(cfg)
    big = case["n"] > 128
    trk = Tracking(conf=cfg, max_tracks=max(768, 3 * case["n"]) if big else 512, max_dets=max(192, case["n"]))
    scene = synth.Scene(7, case["n"], case["H"], case["W"], **case["scene"])
    saw_reid = 0
    for f in range(case["frames"]):
        obj = scene.step()
        if f in case.get("empty", ()):
            obj["embs"], obj["bboxes"], obj["confs"] = [], [], []
        trace = {}
        want = ref.update(obj, trace=trace)
        saw_reid += int("C_reid" in trace)
        got = trk.update(obj)
        assert got[0] == want[0] and got[1] == want[1] and got[2] == want[2], "frame %d" % f
        if f % case.get("every", 6) == case.get("every", 6) - 1 or f == case["frames"] - 1:
            ids, st = _oracle_state(ref)
            _compare_state(trk, ids, st, "frame %d" % f)
            assert trk.next_id == ref.next_id
    if case["conf"].get("lost_reid_after", 50) < 10:
        assert saw_reid > 0


def test_tracker_queries_and_errors():
    cfg = dict(SHIPPED_CONF)
    ref = tracker_ref.TrackerRef(cfg)
    trk = Tracking(conf=cfg, max_tracks=64, max_dets=32)
    scene = synth.Scene(3, 12, 640, 640)
    for _ in range(8):
        obj = scene.step()
        ref.update(obj)
        trk.update(obj)
    obj = scene.step()
    ids = sorted(ref.tracks)
    want = ref.stage1_cost(ids, obj["embs"], obj["bboxes"], obj["confs"], obj["input_hw"])
    ref.predict_all()   # reference computes costs after predict; emulate on the oracle copy only for C_app
    got = trk.cal_cost(row_to_tid=ids, det_embs=obj["embs"], det_boxes=obj["bboxes"], det_confs=obj["confs"],
                       input_hw=obj["input_hw"])
    for k in ("C_total", "C_app", "C_bbox", "C_conf"):
        assert_close(got[k].cpu().numpy(), want[k], rtol=1e-5, atol=2e-6, what=k)
    tv = trk.tracks[ids[0]]
    assert tv.track_id == ids[0] and tv.encoder_feat.shape == (128,) and len(tv.feat_historical) == 8
    C = np.zeros((len(ids), len(obj["bboxes"])), np.float32)
    out = trk.apply_kalman_gating(C, ids, obj["bboxes"], maha_thr=9.49)
    assert out is C and (C == 1e9).any() and (C == 0).any()
    with pytest.raises(ValueError):
        trk.update({"embs": [], "bboxes": [], "confs": [], "frame_id": 1})
    with pytest.raises(ValueError):
        trk.update({"embs": [], "bboxes": [], "confs": [], "input_hw": (1, 1)})
    with pytest.raises(ValueError):
        trk.update({"embs": [np.zeros(128)], "bboxes": [], "confs": [], "input_hw": (1, 1), "frame_id": 1})
    with pytest.raises(ValueError):
        trk.update({"embs": [np.zeros(64, np.float32)], "bboxes": [[0, 0, 1, 1]], "confs": [0.9], "input_hw": (1, 1),
                    "frame_id": 1})
    with pytest.raises(KeyError):
        import os, tempfile, yaml
        d = tempfile.mkdtemp()
        with open(os.path.join(d, "c.yaml"), "w") as fh:
            yaml.safe_dump({"model": {}}, fh)
        Tracking(os.path.join(d, "c.yaml"))
    small = Tracking(conf=cfg, max_tracks=16, max_dets=16, auto_grow=False)
    sc = synth.Scene(0, 12, 640, 640)
    small.update(sc.step())
    with pytest.raises(_lib.B200Error):
        small.update(synth.Scene(1, 12, 640, 640).step())     # 12 live + 12 new could exceed 16


@pytest.mark.parametrize("n", [12, 300])
def test_tracker_nan_embedding_raises_like_scipy(n):
    """A NaN embedding on a detection that passes the gate puts NaN into the cost matrix; the reference dies in
    scipy's linear_sum_assignment with ValueError (hung.py:28).  n = 12 takes the staged validation pass, n = 300
    the row summaries written by the cost kernel."""
    cfg = dict(SHIPPED_CONF)
    ref = tracker_ref.TrackerRef(cfg)
    trk = Tracking(conf=cfg, max_tracks=2 * n + 64, max_dets=n)
    scene = synth.Scene(5, n, 1280, 1280)
    for _ in range(4):
        obj = scene.step()
        assert trk.update(obj) == ref.update(obj)
    obj = scene.step()
    obj["embs"][n // 2] = np.full(128, np.nan, np.float32)
    with pytest.raises(ValueError):
        ref.update(obj)
    with pytest.raises(ValueError):
        trk.update(obj)
    # The reference raises inside stage 1's hungarian_assign, after predict_all and before any update / miss /
    # birth / purge (mainTracking.py:475-516): the failed step leaves "predict only" behind, and a caller that
    # catches the error and carries on sees the same tracker as the reference's caller would.
    ids, st = _oracle_state(ref)
    _compare_state(trk, ids, st, "after the failed step")
    assert trk.next_id == ref.next_id
    for _ in range(3):
        obj = scene.step()
        assert trk.update(obj) == ref.update(obj)
    ids, st = _oracle_state(ref)
    _compare_state(trk, ids, st, "three frames after the failed step")


def test_tracker_grows_like_the_unbounded_reference():
    """Start far too small: every capacity is outgrown mid-sequence and the outputs still match the oracle."""
    cfg = dict(SHIPPED_CONF, lost_reid_after=4, max_age=10)
    ref = tracker_ref.TrackerRef(cfg)
    trk = Tracking(conf=cfg, max_tracks=8, max_dets=4)
    scene = synth.Scene(5, 30, 1280, 1280, drop=0.2, churn=0.2, churn_every=6)
    for f in range(30):
        obj = scene.step()
        want = ref.update(obj)
        got = trk.update(obj)
        assert got[0] == want[0] and got[1] == want[1] and got[2] == want[2], "frame %d" % f
    assert trk._ms.max_tracks >= len(ref.tracks) and trk._ms.max_dets >= 30
    ids, st = _oracle_state(ref)
    _compare_state(trk, ids, st, "after growth")
    assert trk.next_id == ref.next_id


@pytest.mark.parametrize("chain", ["default", "2", "3", "6"])
def test_multistream_equals_independent_trackers(chain, monkeypatch):
    if chain != "default":
        monkeypatch.setenv("B200TRACK_CHAIN", chain)
    cfg = dict(SHIPPED_CONF, lost_reid_after=5, max_age=15)
    S, MD = 5, 48
    ms = MultiStreamTracker(S, cfg, max_tracks=128, max_dets=MD)
    singles = [tracker_ref.TrackerRef(cfg) for _ in range(S)]
    scenes = [synth.Scene(10 + s, 10 + 6 * s, 1088, 1920, drop=0.2, churn=0.2, churn_every=8) for s in range(S)]
    for f in range(40):
        n_det = np.zeros(S, np.int32)
        boxes = np.zeros((S, MD, 4))
        confs = np.zeros((S, MD))
        embs = np.zeros((S, MD, 128), np.float32)
        want = []
        for s in range(S):
            if (f + s) % 7 == 3:                     # this stream has no frame this step
                n_det[s] = -1
                want.append(None)
                continue
            obj = scenes[s].step()
            if (f + s) % 11 == 5:
                obj["embs"], obj["bboxes"], obj["confs"] = [], [], []
            n = len(obj["bboxes"])
            n_det[s] = n
            if n:
                boxes[s, :n] = obj["bboxes"]
                confs[s, :n] = obj["confs"]
                embs[s, :n] = np.stack(obj["embs"])
            want.append(singles[s].update(obj))
        res = ms.step(n_det, boxes, confs, embs, np.full(S, f))
        for s in range(S):
            got = ms.decode(res[s])
            if want[s] is None:
                assert got == ([], [], [])
            else:
                assert got[0] == want[s][0] and got[1] == want[s][1] and got[2] == want[s][2], (f, s)
            assert int(res[s, 3]) == len(singles[s].tracks) and int(res[s, 4]) == singles[s].next_id


def test_tracker_methods_one_by_one_vs_oracle():
    """predict_all / update_matched / mark_missed / create_new_tracks / purge_dead (mainTracking.py:340-448) driven by hand
    in the order Tracking.update uses them, state compared with the oracle after EVERY call; costs and assignments come
    from the oracle so that only the methods under test touch the device state."""
    from oracle.lsap_ref import hungarian_assign
    cfg = dict(SHIPPED_CONF, lost_reid_after=3, max_age=6, hist_max=5)
    ref = tracker_ref.TrackerRef(cfg)
    trk = Tracking(conf=cfg, max_tracks=12, max_dets=8)            # small on purpose: create_new_tracks has to grow it
    scene = synth.Scene(21, 14, 640, 640, drop=0.25, churn=0.2, churn_every=4)

    def same(what):
        ids, st = _oracle_state(ref)
        _compare_state(trk, ids, st, what)
        assert trk.next_id == ref.next_id, what

    for f in range(24):
        obj = scene.step()
        embs, boxes, confs = obj["embs"], obj["bboxes"], obj["confs"]
        N = len(boxes)
        ref.predict_all()
        trk.predict_all()
        same("predict_all %d" % f)
        main = sorted(t for t, tr in ref.tracks.items() if tr.miss_count <= cfg["lost_reid_after"])
        reid = sorted(t for t, tr in ref.tracks.items() if tr.miss_count > cfg["lost_reid_after"])
        free = list(range(N))
        if main and N:
            C = np.array(ref.stage1_cost(main, embs, boxes, confs, obj["input_hw"])["C_total"], dtype=np.float32)
            C = ref.gate(C, main, boxes, cfg["maha_thr"])
            m1, ur, free = hungarian_assign(C, cost_max=cfg["cost_max"])
            ref.absorb(m1, main, embs, boxes, confs, f, C, cost_update_max=cfg["cost_update_max"], maha_thr=cfg["maha_thr"])
            trk.update_matched(m1, main, embs, boxes, confs, f, C, ema_alpha=cfg["ema_alpha"],
                               conf_update_min=cfg["conf_update_min"], cost_update_max=cfg["cost_update_max"],
                               maha_thr=cfg["maha_thr"])
            same("update_matched %d" % f)
            lost = [main[r] for r in ur]
            ref.mark_missed(lost)
            trk.mark_missed(lost + [10 ** 6])                      # an id that is not live is skipped (:350-351)
            same("mark_missed %d" % f)
        if reid and free:
            e_u, b_u, c_u = [embs[j] for j in free], [boxes[j] for j in free], [confs[j] for j in free]
            C2 = np.array(ref.app_cost(reid, e_u), dtype=np.float32)
            m2, ur2, ud2 = hungarian_assign(C2, cost_max=cfg["reid_only_cost_max"])
            ref.absorb(m2, reid, e_u, b_u, c_u, f, C2, cost_update_max=cfg["reid_only_cost_max"], maha_thr=1e18)
            trk.update_matched(m2, reid, e_u, b_u, c_u, f, C2, ema_alpha=cfg["ema_alpha"],
                               conf_update_min=cfg["conf_update_min"], cost_update_max=cfg["reid_only_cost_max"], maha_thr=1e18)
            same("update_matched (reid) %d" % f)
            ref.mark_missed([reid[r] for r in ur2])
            trk.mark_missed([reid[r] for r in ur2])
            free = [free[j] for j in ud2]
        elif reid:
            ref.mark_missed(reid)
            trk.mark_missed(reid)
        ref.spawn(free, embs, boxes, confs, f)
        trk.create_new_tracks(free, embs, boxes, confs, f)
        same("create_new_tracks %d" % f)
        ref.purge_dead()
        trk.purge_dead()
        same("purge_dead %d" % f)
    assert ref.next_id > 20 and trk._ms.max_tracks > 12
    with pytest.raises(KeyError):
        trk.update_matched([(0, 0)], [10 ** 6], [obj["embs"][0]], [obj["bboxes"][0]], [0.9], 99, np.zeros((1, 1), np.float32))
    # the hand-driven tracker and a fused update() agree on the next frame
    obj = scene.step()
    assert trk.update(obj) == tuple(ref.update(obj))


def test_step_device_vs_oracle():
    """MultiStreamTracker.step_device / b200_tracker_step with DEVICE-resident inputs (the path bench.py times):
    every result row of every frame and the exported state against one oracle tracker per stream, 36 frames with
    drops, churn, empty and idle frames; interleaved with a second handle of a different capacity (the assignment
    kernels' shared-memory opt-in is per function, not per handle)."""
    cfg = dict(SHIPPED_CONF, lost_reid_after=5, max_age=15)
    S, MD, F = 4, 64, 36
    ms = MultiStreamTracker(S, cfg, max_tracks=192, max_dets=MD)
    big = Tracking(conf=cfg, max_tracks=512, max_dets=256)          # ~200 KB of assignment smem; created after `ms`...
    small = Tracking(conf=cfg, max_tracks=32, max_dets=16)          # ...and a small one created last
    refs = [tracker_ref.TrackerRef(cfg) for _ in range(S)]
    ref_big, ref_small = tracker_ref.TrackerRef(cfg), tracker_ref.TrackerRef(cfg)
    scenes = [synth.Scene(40 + s, 20 + 12 * s, 1088, 1920, drop=0.15, churn=0.15, churn_every=7) for s in range(S)]
    sc_big, sc_small = synth.Scene(90, 200, 1280, 1280, drop=0.05), synth.Scene(91, 6, 640, 640)
    n_det = np.zeros((F, S), np.int32)
    boxes = np.zeros((F, S, MD, 4))
    confs = np.zeros((F, S, MD))
    embs = np.zeros((F, S, MD, 128), np.float32)
    want = [[None] * S for _ in range(F)]
    for f in range(F):
        for s in range(S):
            if (f + 2 * s) % 9 == 4:
                n_det[f, s] = -1
                continue
            obj = scenes[s].step()
            if (f + s) % 13 == 6:
                obj["embs"], obj["bboxes"], obj["confs"] = [], [], []
            n = len(obj["bboxes"])
            n_det[f, s] = n
            if n:
                boxes[f, s, :n], confs[f, s, :n], embs[f, s, :n] = obj["bboxes"], obj["confs"], np.stack(obj["embs"])
            want[f][s] = refs[s].update(obj)
    import torch
    d = lambda a: torch.from_numpy(a).cuda()  # noqa: E731
    d_n, d_b, d_c, d_e = d(n_det), d(boxes), d(confs), d(embs)
    d_f = torch.arange(F, dtype=torch.int32, device="cuda")[:, None].repeat(1, S).contiguous()
    results = torch.zeros((F, S, ms.stride), dtype=torch.int32, device="cuda")
    for f in range(F):
        ms.step_device(d_n[f], d_b[f], d_c[f], d_e[f], d_f[f], results[f])
        if f % 6 == 0:                                              # other handles step in between
            o = sc_big.step()
            assert big.update(o) == tuple(ref_big.update(o)), "big %d" % f
            o = sc_small.step()
            assert small.update(o) == tuple(ref_small.update(o)), "small %d" % f
    res = results.cpu().numpy()
    for f in range(F):
        for s in range(S):
            got = ms.decode(res[f, s])
            assert int(res[f, s, 5]) == 0
            if want[f][s] is None:
                assert got == ([], [], []), (f, s)
            else:
                assert got[0] == want[f][s][0] and got[1] == want[f][s][1] and got[2] == want[f][s][2], (f, s)
    for s in range(S):
        ids, st = _oracle_state(refs[s])
        snap = ms.export(s)
        assert snap["ids"].tolist() == ids and snap["next_id"] == refs[s].next_id
        assert_close(snap["x"], st["x"], rtol=1e-5, atol=1e-6, what="x")
        assert_close(snap["P"], st["P"], rtol=1e-5, atol=1e-5, what="P")
        assert_close(snap["ema"], st["ema"], rtol=1e-5, atol=1e-6, what="ema")
        assert snap["miss"].tolist() == st["miss"] and snap["age"].tolist() == st["age"]
    # a host step after device steps sees the right live count (n_live is re-read, not stale)
    assert ms.n_live_now().tolist() == [len(r.tracks) for r in refs]


@pytest.mark.parametrize("path", ["step_device", "create_new_tracks"])
def test_host_step_grows_after_device_side_births(path):
    """Tracks created by device-side calls (step_device, create_new_tracks) are not in the host's live count.  A host step
    whose births do not fit beside them must grow the handle first, not drop them: two groups of 8 detections fill a
    16-track handle, then a host step brings 8 more, far from every track, and must match the unbounded oracle."""
    cfg = dict(SHIPPED_CONF)
    rng = np.random.default_rng(3)
    objs = []
    for g in range(3):                              # 400 px between groups: the Mahalanobis gate rejects every pair
        e = rng.standard_normal((8, 128)).astype(np.float32)
        e /= np.linalg.norm(e, axis=1, keepdims=True)
        objs.append({"embs": list(e), "bboxes": [[100.0 + 150 * j, 100.0 + 400 * g, 140.0 + 150 * j, 140.0 + 400 * g]
                                                  for j in range(8)],
                     "confs": [0.9] * 8, "input_hw": (1280, 1280), "frame_id": g})
    ref = tracker_ref.TrackerRef(cfg)
    trk = Tracking(conf=cfg, max_tracks=16, max_dets=8)
    if path == "step_device":
        ms = trk._ms
        d = lambda a, dt: torch.tensor(np.asarray(a), dtype=dt, device="cuda")  # noqa: E731
        for o in objs[:2]:
            ref.update(o)
            ms.step_device(d([8], torch.int32), d([o["bboxes"]], torch.float64), d([o["confs"]], torch.float64),
                           d([np.stack(o["embs"])], torch.float32), d([o["frame_id"]], torch.int32))
        res = ms.step([8], [objs[2]["bboxes"]], [objs[2]["confs"]], [np.stack(objs[2]["embs"])], [2])
        got = ms.decode(res[0])
    else:
        for o in objs[:2]:
            ref.spawn(range(8), o["embs"], o["bboxes"], o["confs"], o["frame_id"])
            trk.create_new_tracks(range(8), o["embs"], o["bboxes"], o["confs"], o["frame_id"])
        got = trk.update(objs[2])
    want = ref.update(objs[2])
    assert len(ref.tracks) == 24 and trk._ms.max_tracks >= 24
    assert got[0] == want[0] and got[1] == want[1] and got[2] == want[2]
    ids, st = _oracle_state(ref)
    _compare_state(trk, ids, st, path)
    assert trk.next_id == ref.next_id


def test_step_async_matches_step_and_defers_errors():
    """MultiStreamTracker.step_async: up to four steps queued ahead of their results; every result equals the oracle's,
    results come back in order, a NaN frame raises at .result() of THAT step only and the stream carries on."""
    cfg = dict(SHIPPED_CONF, lost_reid_after=5, max_age=15)
    S, MD, F = 3, 32, 30
    ms = MultiStreamTracker(S, cfg, max_tracks=96, max_dets=MD)
    refs = [tracker_ref.TrackerRef(cfg) for _ in range(S)]
    scenes = [synth.Scene(60 + s, 12 + 5 * s, 720, 1280, drop=0.15, churn=0.15, churn_every=6) for s in range(S)]
    frames, want = [], []
    for f in range(F):
        n_det = np.zeros(S, np.int32)
        boxes, confs, embs = np.zeros((S, MD, 4)), np.zeros((S, MD)), np.zeros((S, MD, 128), np.float32)
        w = []
        for s in range(S):
            obj = scenes[s].step()
            n = len(obj["bboxes"])
            n_det[s] = n
            boxes[s, :n], confs[s, :n], embs[s, :n] = obj["bboxes"], obj["confs"], np.stack(obj["embs"])
            if f == 20 and s == 1:
                embs[s, 0] = np.nan                       # scipy raises for this stream at this frame ...
                obj = dict(obj, embs=[np.full(128, np.nan, np.float32)] + obj["embs"][1:])
                with pytest.raises(ValueError):
                    refs[s].update(obj)
                w.append(None)
            else:
                w.append(refs[s].update(obj))
        frames.append((n_det, boxes, confs, embs))
        want.append(w)
    handles = []
    for f in range(F):
        handles.append(ms.step_async(*frames[f], np.full(S, f)))
        if len(handles) == 4:                             # the ring is full: collect the oldest
            _check_async(ms, handles.pop(0), want[f - 3], f - 3)
    ms.drain()
    roomy = MultiStreamTracker(1, cfg, max_tracks=256, max_dets=4)          # capacity never forces a drain here
    one = (np.array([1], np.int32), np.array([[[10., 10., 50., 80.]] + [[0.] * 4] * 3]), np.array([[0.9, 0, 0, 0]]),
           np.ones((1, 4, 128), np.float32))
    kept = [roomy.step_async(*one, [k]) for k in range(4)]
    with pytest.raises(_lib.B200Error):
        roomy.step_async(*one, [4])                                          # a fifth pending step
    assert [int(h.result()[0, 3]) for h in kept] == [1, 1, 1, 1]             # one live track throughout
    base = F - len(handles)
    for k, h in enumerate(handles):
        _check_async(ms, h, want[base + k], base + k)


def test_step_async_pinned_arrays_are_read_in_place():
    """step_async(pinned=True): page-locked detection arrays are uploaded by DMA from where they are (no staging copy);
    same results as the oracle, pageable arrays are refused."""
    cfg = dict(SHIPPED_CONF)
    S, MD, F = 2, 24, 12
    ms = MultiStreamTracker(S, cfg, max_tracks=64, max_dets=MD)
    refs = [tracker_ref.TrackerRef(cfg) for _ in range(S)]
    scenes = [synth.Scene(80 + s, 10 + 9 * s, 720, 1280, drop=0.1) for s in range(S)]
    pb = torch.zeros((F, S, MD, 4), dtype=torch.float64).pin_memory()
    pc = torch.zeros((F, S, MD), dtype=torch.float64).pin_memory()
    pe = torch.zeros((F, S, MD, 128), dtype=torch.float32).pin_memory()
    nd = np.zeros((F, S), np.int32)
    want = []
    for f in range(F):
        w = []
        for s in range(S):
            obj = scenes[s].step()
            n = len(obj["bboxes"])
            nd[f, s] = n
            pb[f, s, :n] = torch.tensor(obj["bboxes"], dtype=torch.float64)
            pc[f, s, :n] = torch.tensor(obj["confs"], dtype=torch.float64)
            pe[f, s, :n] = torch.from_numpy(np.stack(obj["embs"]))
            w.append(refs[s].update(obj))
        want.append(w)
    prev = None
    for f in range(F):
        h = ms.step_async(nd[f], pb[f], pc[f].numpy(), pe[f], np.full(S, f), pinned=True)
        if prev is not None:
            _check_async(ms, prev[0], want[prev[1]], prev[1])
        prev = (h, f)
    _check_async(ms, prev[0], want[prev[1]], prev[1])
    with pytest.raises(ValueError):
        ms.step_async(nd[0], np.zeros((S, MD, 4)), np.zeros((S, MD)), np.zeros((S, MD, 128), np.float32), np.full(S, 99),
                      pinned=True)
    with pytest.raises(TypeError):
        ms.step_async(nd[0], np.zeros((S, MD, 4), np.float32), pc[0], pe[0], np.full(S, 99), pinned=True)


def _check_async(ms, handle, want, f):
    if any(w is None for w in want):
        with pytest.raises(ValueError):
            handle.result()
        res = handle.table                                # ... and the other streams' rows are still there
    else:
        res = handle.result()
    for s, w in enumerate(want):
        if w is None:
            assert int(res[s, 5]) != 0
            continue
        got = ms.decode(res[s])
        assert got[0] == w[0] and got[1] == w[1] and got[2] == w[2], (f, s)


@pytest.mark.parametrize("seed,chain", [(k, None) for k in range(10)] + [(k, "3") for k in range(10, 16)] + [(16, "6"), (17, "6")])
def test_tracker_fuzz_vs_oracle(seed, chain, monkeypatch):
    """Randomised differential test: random hyper-parameters (including degenerate ones: one-row banks,
    top-1, immediate purge, ReID stage almost always on), random scene dynamics, empty and idle frames."""
    if chain is not None:
        monkeypatch.setenv("B200TRACK_CHAIN", chain)
    rng = np.random.default_rng(1000 + seed)
    cfg = dict(SHIPPED_CONF,
               hist_max=int(rng.choice([1, 2, 5, 30, 33, 64])), emb_top_k=int(rng.choice([1, 3, 5, 9])),
               max_age=int(rng.choice([0, 1, 5, 40])), lost_reid_after=int(rng.choice([0, 1, 3, 50])),
               init_conf_min=float(rng.choice([0.0, 0.5, 0.7])), conf_update_min=float(rng.choice([0.0, 0.55, 0.8])),
               cost_max=float(rng.choice([50.0, 1.0, 0.3])), cost_update_max=float(rng.choice([30.0, 0.5])),
               maha_thr=float(rng.choice([9.49, 2.0, 1e6])), reid_only_cost_max=float(rng.choice([0.4, 0.05, 2.0])),
               ema_alpha=float(rng.choice([0.9, 0.5, 0.0])), w_bbox=float(rng.choice([0.3, 0.0, 2.0])))
    n = int(rng.integers(1, 40))
    scene = synth.Scene(int(rng.integers(1 << 30)), n, 720, 1280, drop=float(rng.choice([0.0, 0.2, 0.6])),
                        churn=float(rng.choice([0.0, 0.3])), churn_every=int(rng.integers(2, 9)),
                        noise=float(rng.choice([0.05, 0.5])))
    ref = tracker_ref.TrackerRef(cfg)
    trk = Tracking(conf=cfg, max_tracks=16, max_dets=8)            # also exercises growth
    for f in range(36):
        obj = scene.step()
        if rng.uniform() < 0.08:
            obj["embs"], obj["bboxes"], obj["confs"] = [], [], []
        want = ref.update(obj)
        got = trk.update(obj)
        assert got[0] == want[0] and got[1] == want[1] and got[2] == want[2], "seed %d frame %d cfg %s" % (seed, f, cfg)
    ids, st = _oracle_state(ref)
    _compare_state(trk, ids, st, "seed %d" % seed)
    assert trk.next_id == ref.next_id
