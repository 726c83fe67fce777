"""Generates tests/golden/*.npz by running the UNMODIFIED reference (build container only).

    python tests/golden/make_golden.py

Needs /root/reference mounted (it is imported, never copied).  The third-party ops the
reference calls are the versions installed in this image (torchvision 0.26.0, scipy
1.18.1, numpy 2.3.5); filterpy is replaced by oracle/filterpy_shim.py (SURVEY.md 8c).
Fixtures hold inputs AND outputs so the GPU box needs neither the reference nor a
bit-stable RNG.
"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

from oracle import reference_loader  # noqa: E402
import alufe_b200  # noqa: E402,F401
from alufe_b200 import synth  # noqa: E402

OUT = os.path.dirname(os.path.abspath(__file__))


def dump_state(trk):
    """Flatten the reference tracker's state dict into arrays."""
    ids = sorted(trk.tracks.keys())
    st = {"ids": np.array(ids, dtype=np.int64), "next_id": np.int64(trk.next_id)}
    st["x"] = np.array([trk.tracks[i].kf.x.reshape(-1).astype(np.float64) for i in ids]).reshape(-1, 8)
    st["P"] = np.array([trk.tracks[i].kf.P.astype(np.float64) for i in ids]).reshape(-1, 8, 8)
    st["x_is64"] = np.array([trk.tracks[i].kf.x.dtype == np.float64 for i in ids])
    st["P_is64"] = np.array([trk.tracks[i].kf.P.dtype == np.float64 for i in ids])
    st["ema"] = np.array([trk.tracks[i].memory.encoder_feat for i in ids], dtype=np.float32).reshape(-1, 128)
    st["bank_len"] = np.array([len(trk.tracks[i].memory.feat_historical) for i in ids], dtype=np.int64)
    hist = max([len(trk.tracks[i].memory.feat_historical) for i in ids], default=0)
    bank = np.zeros((len(ids), hist, 128), dtype=np.float32)
    for r, i in enumerate(ids):
        fh = trk.tracks[i].memory.feat_historical
        if fh:
            bank[r, :len(fh)] = np.stack(fh)
    st["bank"] = bank
    st["miss"] = np.array([trk.tracks[i].miss_count for i in ids], dtype=np.int64)
    st["age"] = np.array([trk.tracks[i].age for i in ids], dtype=np.int64)
    st["last_bbox"] = np.array([trk.tracks[i].memory.last_bbox for i in ids], dtype=np.float64).reshape(-1, 4)
    st["last_conf"] = np.array([trk.tracks[i].memory.last_conf for i in ids], dtype=np.float64)
    st["last_cost"] = np.array([np.nan if trk.tracks[i].memory.last_match_cost is None
                                else trk.tracks[i].memory.last_match_cost for i in ids], dtype=np.float64)
    return st


def run_tracker_case(name, seed, n, H, W, frames, overrides, scene_kw, empty_frames=()):
    ref = reference_loader.load()
    trk = reference_loader.new_tracking()
    for k, v in overrides.items():
        assert hasattr(trk, k), k
        setattr(trk, k, v)
    seen = []
    orig = ref.mainTracking.hungarian_assign

    def spy(C, cost_max=1e9):
        seen.append(np.array(C, dtype=np.float32).copy())
        return orig(C, cost_max=cost_max)

    ref.mainTracking.hungarian_assign = spy
    scene = synth.Scene(seed, n, H, W, **scene_kw)
    out = {"n_frames": np.int64(frames), "H": np.int64(H), "W": np.int64(W)}
    for k, v in overrides.items():
        out["cfg_" + k] = np.float64(v)
    try:
        for f in range(frames):
            obj = scene.step()
            if f in empty_frames:
                obj["embs"], obj["bboxes"], obj["confs"] = [], [], []
            seen.clear()
            m, ut, ud = trk.update(obj)
            p = "f%03d_" % f
            out[p + "embs"] = np.array(obj["embs"], dtype=np.float32).reshape(-1, 128)
            out[p + "boxes"] = np.array(obj["bboxes"], dtype=np.float64).reshape(-1, 4)
            out[p + "confs"] = np.array(obj["confs"], dtype=np.float64)
            out[p + "matches"] = np.array(m, dtype=np.int64).reshape(-1, 2)
            out[p + "unmatched_tracks"] = np.array(ut, dtype=np.int64)
            out[p + "unmatched_dets"] = np.array(ud, dtype=np.int64)
            for s, C in enumerate(seen):
                out[p + "C%d" % s] = C
            if f % 5 == 4 or f == frames - 1:
                for k, v in dump_state(trk).items():
                    out[p + "st_" + k] = v
    finally:
        ref.mainTracking.hungarian_assign = orig
    np.savez_compressed(os.path.join(OUT, "tracker_%s.npz" % name), **out)
    print("tracker_%s: %d frames, %d live tracks, next_id %d" % (name, frames, len(trk.tracks), trk.next_id))


def run_cost_cases():
    ref = reference_loader.load()
    rng = np.random.default_rng(11)
    out = {}
    for idx, (M, N) in enumerate([(5, 7), (8, 8), (1, 3), (13, 2)]):
        bp = synth.random_boxes(rng, M, 640, 640)
        bc = synth.random_boxes(rng, N, 640, 640)
        if idx == 0:
            bp[0] = [10.0, 10.0, 10.2, 10.3]        # sub-pixel -> w,h clamp to 1
            bc[1] = [50.0, 60.0, 40.0, 50.0]        # inverted -> clamp
        cp = rng.uniform(0.0, 1.0, M)
        cq = rng.uniform(0.0, 1.0, N)
        if idx == 0:
            cp[1] = 0.0                             # eps clamp
        Capp = rng.uniform(0, 2, (M, N)).astype(np.float32)
        import torch
        r = ref.costCard.cal_cost(C_app=torch.from_numpy(Capp), boxes_prev=bp.tolist(),
                                  boxes_cur=bc.tolist(), input_hw=(640, 640),
                                  conf_prev=cp.tolist(), conf_cur=cq.tolist(),
                                  assign=[(i % N) if i % 3 else -1 for i in range(M)])
        p = "k%d_" % idx
        out[p + "bp"], out[p + "bc"], out[p + "cp"], out[p + "cq"], out[p + "Capp"] = bp, bc, cp, cq, Capp
        for key in ("C_total", "C_bbox", "C_center", "C_scale", "C_conf"):
            out[p + key] = r[key].numpy()
        out[p + "total_cost"] = np.float64(r["total_cost"])
    np.savez_compressed(os.path.join(OUT, "cost.npz"), **out)
    print("cost: ok")


def run_kalman_cases():
    ref = reference_loader.load()
    KF = ref.KalmanFilter
    rng = np.random.default_rng(5)
    out = {}
    for idx in range(4):
        box = synth.random_boxes(rng, 1, 640, 640)[0]
        kf = KF.init_kf_from_bbox(box.tolist())
        p = "t%d_" % idx
        out[p + "box0"] = box
        zs, xs, Ps, d2pre, d2post, did_upd = [], [], [], [], [], []
        for step in range(12):
            kf.predict()
            box = box + rng.normal(0, 2.0, 4)
            upd = not (idx == 1 and step in (3, 4, 5))      # a gap: predicts without updates
            d2pre.append(KF.gating_distance_maha(kf, box.tolist()))
            if upd:
                kf.update(KF.bbox_xyxy_to_z(box.tolist()))
            d2post.append(KF.gating_distance_maha(kf, box.tolist()))
            zs.append(box.copy())
            xs.append(kf.x.reshape(-1).astype(np.float64))
            Ps.append(kf.P.astype(np.float64))
            did_upd.append(upd)
        out[p + "boxes"] = np.array(zs)
        out[p + "x"] = np.array(xs)
        out[p + "P"] = np.array(Ps)
        out[p + "d2pre"] = np.array(d2pre)
        out[p + "d2post"] = np.array(d2post)
        out[p + "upd"] = np.array(did_upd)
        out[p + "pred_bbox"] = np.array(KF.x_to_bbox_xyxy(kf.x.reshape(-1)))
    np.savez_compressed(os.path.join(OUT, "kalman.npz"), **out)
    print("kalman: ok")


def run_lsap_cases():
    ref = reference_loader.load()
    rng = np.random.default_rng(3)
    out = {}
    cases = [(8, 8, 0.0), (64, 64, 0.0), (64, 64, 0.9), (20, 33, 0.5), (33, 20, 0.5), (128, 128, 0.95),
             (7, 1, 0.0), (1, 9, 0.0)]
    for idx, (m, n, g) in enumerate(cases):
        C = synth.lsap_matrix(rng, m, n, g)
        mt, ut, ud = ref.hung.hungarian_assign(C, cost_max=50.0)
        p = "m%d_" % idx
        out[p + "C"] = C
        out[p + "matches"] = np.array(mt, dtype=np.int64).reshape(-1, 2)
        out[p + "ut"] = np.array(ut, dtype=np.int64)
        out[p + "ud"] = np.array(ud, dtype=np.int64)
    # ties: integer and constant matrices (scipy's tie-break rules)
    for idx, C in enumerate([np.zeros((6, 6), np.float32), rng.integers(0, 4, (12, 12)).astype(np.float32),
                             rng.integers(0, 3, (9, 14)).astype(np.float32),
                             rng.integers(0, 3, (14, 9)).astype(np.float32)]):
        from scipy.optimize import linear_sum_assignment
        r, c = linear_sum_assignment(C)
        out["tie%d_C" % idx] = C
        out["tie%d_rows" % idx] = r
        out["tie%d_cols" % idx] = c
    np.savez_compressed(os.path.join(OUT, "lsap.npz"), **out)
    print("lsap: ok")


def run_roi_cases():
    import torch
    from torchvision.ops import roi_align
    out = {}
    feat = synth.feature_map(0, 2, 16, 20, 20)
    boxes = np.concatenate([synth.random_boxes(np.random.default_rng(1), 10, 640, 640),
                            synth.edge_case_boxes(640, 640)])
    rois = np.concatenate([(np.arange(len(boxes)) % 2)[:, None].astype(np.float64), boxes], axis=1).astype(np.float32)
    out["feat"], out["rois"] = feat, rois
    for tag, (ps, sr, al) in {"a": ((10, 10), 2, True), "b": ((7, 7), 2, True), "c": ((7, 7), -1, False),
                              "d": ((3, 5), 3, True)}.items():
        y = roi_align(torch.from_numpy(feat), torch.from_numpy(rois), ps, 20 / 640.0, sr, al)
        out["out_" + tag] = y.numpy()
        out["arg_" + tag] = np.array([ps[0], ps[1], sr, int(al)], dtype=np.int64)
    np.savez_compressed(os.path.join(OUT, "roi.npz"), **out)
    print("roi: ok")


def run_roi_wrapper_cases():
    """The reference's own ROI call conventions, called unbound (both methods ignore ``self``):
    MainInfer.roi_align_from_input_boxes (tracking.py:193-221) and PreProcess._preprocess_roi
    (trainingCard.py:24-79), on square and non-square maps, with inverted / out-of-image / sub-pixel boxes."""
    import torch
    w = reference_loader.load_roi_wrappers()
    out = {}
    for tag, (C, Hf, Wf, H_in, W_in) in {"sq": (32, 20, 20, 640, 640), "wide": (24, 34, 60, 1088, 1920)}.items():
        feat = synth.feature_map(3, 1, C, Hf, Wf)
        boxes = np.concatenate([synth.random_boxes(np.random.default_rng(4), 9, H_in, W_in),
                                synth.edge_case_boxes(H_in, W_in)]).astype(np.float64)
        out[tag + "_feat"], out[tag + "_boxes"] = feat, boxes
        out[tag + "_hw"] = np.array([H_in, W_in], dtype=np.int64)
        f = torch.from_numpy(feat)
        for ps in ((7, 7), (10, 10)):
            y = w.roi_align_from_input_boxes(None, f, boxes.tolist(), (H_in, W_in), out_size=ps)
            out["%s_r1_%d" % (tag, ps[0])] = y.numpy()
        y = w.roi_align_from_input_boxes(None, f, boxes.tolist(), (H_in, W_in))          # default 7x7
        assert np.array_equal(y.numpy(), out[tag + "_r1_7"])
        out[tag + "_r2_10"] = w.preprocess_roi(None, f, torch.from_numpy(boxes), (H_in, W_in)).numpy()
        out[tag + "_r2_7_nomin"] = w.preprocess_roi(None, f, torch.from_numpy(boxes), (H_in, W_in), output_size=(7, 7),
                                                    sampling_ratio=2, aligned=True, enforce_min_size=0.0).numpy()
    # the two conventions agree bit for bit on most ROIs: three preprocess_roi outputs keep only the rows where they
    # differ, which brings the file under 1 MB (tests/conftest.py::load_roi_wrappers_golden restores them)
    for key, base in (("sq_r2_7_nomin", "sq_r1_7"), ("wide_r2_7_nomin", "wide_r1_7"), ("wide_r2_10", "wide_r1_10")):
        rows = np.array([i for i in range(len(out[key])) if not np.array_equal(out[key][i], out[base][i])], dtype=np.int64)
        out[key] = out[key][rows]
        out[key + "_rows"], out[key + "_base"] = rows, np.array(base)
    np.savez_compressed(os.path.join(OUT, "roi_wrappers.npz"), **out)
    print("roi_wrappers: ok")


LIVE_TUNABLES = ("hist_max", "emb_top_k", "max_age", "lost_reid_after", "init_conf_min", "conf_update_min", "cost_max",
                 "cost_update_max", "maha_thr", "reid_only_cost_max", "ema_alpha", "w_bbox")


def tracker_fuzz_case(seed):
    """Randomised tracker case `seed`: hyper-parameter overrides and 18 frames of a scene with misses, births, empty
    frames and the ReID-only stage, all drawn from seeded generators."""
    rng = np.random.default_rng(500 + seed)
    over = dict(hist_max=int(rng.choice([1, 3, 30])), emb_top_k=int(rng.choice([1, 5])),
                max_age=int(rng.choice([1, 6, 40])), lost_reid_after=int(rng.choice([0, 2, 50])),
                init_conf_min=float(rng.choice([0.0, 0.5, 0.7])), conf_update_min=float(rng.choice([0.0, 0.55, 0.8])),
                cost_max=float(rng.choice([50.0, 1.0])), cost_update_max=float(rng.choice([30.0, 0.5])),
                maha_thr=float(rng.choice([9.49, 2.0, 1e6])), reid_only_cost_max=float(rng.choice([0.4, 2.0])),
                ema_alpha=float(rng.choice([0.9, 0.5])), w_bbox=float(rng.choice([0.3, 2.0])))
    n = int(rng.integers(2, 14))
    scene = synth.Scene(int(rng.integers(1 << 30)), n, 720, 1280, drop=float(rng.choice([0.0, 0.3])),
                        churn=float(rng.choice([0.0, 0.3])), churn_every=int(rng.integers(2, 7)))
    frames = []
    for _ in range(18):
        obj = scene.step()
        if rng.uniform() < 0.1:
            obj["embs"], obj["bboxes"], obj["confs"] = [], [], []
        frames.append(obj)
    return over, frames


def cost_fuzz_cases():
    """Ten randomised cal_cost inputs (1..19 x 1..19) and hungarian_assign matrices, from a seeded generator."""
    rng = np.random.default_rng(77)
    for _ in range(10):
        M, N = int(rng.integers(1, 20)), int(rng.integers(1, 20))
        C_app = rng.uniform(0, 2, (M, N)).astype(np.float32)
        bp = synth.random_boxes(rng, M, 720, 1280)
        bc = synth.random_boxes(rng, N, 720, 1280)
        cp, cc = rng.uniform(0.05, 1, M), rng.uniform(0.05, 1, N)
        C = synth.lsap_matrix(rng, M, N, float(rng.choice([0.0, 0.8])))
        yield dict(C_app=C_app, boxes_prev=bp, boxes_cur=bc, conf_prev=cp, conf_cur=cc), C


def _assignment(out, p, m, ut, ud):
    out[p + "matches"] = np.array(m, dtype=np.int64).reshape(-1, 2)
    out[p + "ut"], out[p + "ud"] = np.array(ut, dtype=np.int64), np.array(ud, dtype=np.int64)


def record_tracker_fuzz(seed, make_tracker, state):
    """Runs tracker case `seed` through make_tracker(overrides) and returns what every update returned (the three
    lists of all frames concatenated, their lengths per frame in "counts") and, under "st_", the final state of every
    track in ascending id; state(track) returns (x, P, ema, history length, miss_count, age).  "inputs" sums the case's
    inputs, so that a change of the generators shows."""
    over, frames = tracker_fuzz_case(seed)
    trk = make_tracker(over)
    out = {"over": np.array([over[k] for k in LIVE_TUNABLES], dtype=np.float64),
           "inputs": np.array([sum(float(np.sum(np.asarray(o[k], np.float64))) for o in frames)
                               for k in ("bboxes", "confs", "embs")])}
    res = [trk.update(obj) for obj in frames]
    out["counts"] = np.array([[len(m), len(ut), len(ud)] for m, ut, ud in res], dtype=np.int64)
    _assignment(out, "", [p for m, _, _ in res for p in m], [t for _, ut, _ in res for t in ut],
                [d for _, _, ud in res for d in ud])
    ids = sorted(trk.tracks)
    st = [state(trk.tracks[i]) for i in ids]
    out["st_ids"], out["st_next_id"] = np.array(ids, dtype=np.int64), np.int64(trk.next_id)
    out["st_x"] = np.array([np.asarray(s[0], np.float64).reshape(-1) for s in st]).reshape(-1, 8)
    out["st_P"] = np.array([np.asarray(s[1], np.float64) for s in st]).reshape(-1, 8, 8)
    out["st_ema"] = np.array([np.asarray(s[2], np.float32) for s in st]).reshape(-1, 128)
    out["st_hist_miss_age"] = np.array([s[3:] for s in st], dtype=np.int64).reshape(-1, 3)
    return out


def record_cost_fuzz(cal_cost, hungarian_assign):
    """cost_fuzz_cases through cal_cost(**inputs) -> dict of [M, N] float32 terms and hungarian_assign(C, cost_max=50),
    under "k<case>_"."""
    out = {}
    for idx, (kw, C) in enumerate(cost_fuzz_cases()):
        p = "k%d_" % idx
        terms = cal_cost(**kw)
        for k in ("C_total", "C_bbox", "C_center", "C_scale", "C_conf"):
            out[p + k] = np.asarray(terms[k], np.float32)
        _assignment(out, p, *hungarian_assign(C, cost_max=50.0))
        out[p + "inputs"] = np.array([float(np.sum(np.asarray(v, np.float64))) for v in kw.values()] + [float(C.sum())])
    return out


def reference_tracker(over):
    trk = reference_loader.new_tracking()
    for k, v in over.items():
        assert hasattr(trk, k), k
        setattr(trk, k, v)
    return trk


def reference_state(tr):
    return tr.kf.x, tr.kf.P, tr.memory.encoder_feat, len(tr.memory.feat_historical), tr.miss_count, tr.age


def reference_cal_cost(**kw):
    import torch
    ref = reference_loader.load()
    r = ref.costCard.cal_cost(C_app=torch.from_numpy(kw["C_app"]), boxes_prev=kw["boxes_prev"].tolist(),
                              boxes_cur=kw["boxes_cur"].tolist(), input_hw=(720, 1280),
                              conf_prev=kw["conf_prev"].tolist(), conf_cur=kw["conf_cur"].tolist())
    return {k: v.cpu().numpy() for k, v in r.items() if k.startswith("C_")}


def run_live_fuzz_cases():
    """The randomised tracker, cost and assignment cases of tests/test_oracle_live_reference.py, as the reference
    returns them.  The live_fuzz.npz in the tree was recorded by these same record_* functions with the oracle in the
    reference's place (tests/test_oracle_live_reference.py::_oracle_*): tracker_ref, cost_ref, lsap_ref, kalman_ref,
    the filterpy shim and the generators in synth.py are unchanged since that test first compared them with the
    reference on these cases.  Running this function where the reference is mounted records them from the reference."""
    out = {}
    for seed in range(6):
        out.update({"t%d_%s" % (seed, k): v for k, v in record_tracker_fuzz(seed, reference_tracker, reference_state).items()})
    out.update({"cost_" + k: v for k, v in record_cost_fuzz(reference_cal_cost, reference_loader.load().hung.hungarian_assign).items()})
    np.savez_compressed(os.path.join(OUT, "live_fuzz.npz"), **out)
    print("live_fuzz: ok")


if __name__ == "__main__":
    assert reference_loader.available(), "mount the reference at /root/reference"
    if len(sys.argv) > 1:                      # regenerate only the named fixtures, e.g. `make_golden.py roi_wrappers`
        for name in sys.argv[1:]:
            globals()["run_%s_cases" % name]()
        sys.exit(0)
    run_roi_wrapper_cases()
    run_live_fuzz_cases()
    run_roi_cases()
    run_lsap_cases()
    run_kalman_cases()
    run_cost_cases()
    # c1-shaped steady tracking (tracking.py shapes): 8 identities, no drops.
    run_tracker_case("c1_steady", seed=0, n=8, H=640, W=640, frames=40, overrides={}, scene_kw={})
    # births / misses / re-activation / long-lost ReID stage / purge, with short horizons.
    run_tracker_case("churn", seed=1, n=10, H=640, W=640, frames=60,
                     overrides={"lost_reid_after": 3, "max_age": 9, "hist_max": 6},
                     scene_kw={"drop": 0.25, "churn": 0.2, "churn_every": 7}, empty_frames=(17, 18, 41))
