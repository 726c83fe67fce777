"""CPU: the oracle restatements against fixtures produced by the live reference
(tests/golden/make_golden.py) and against the installed third-party ops."""
import numpy as np
import pytest

from conftest import assert_close, load_golden, load_roi_wrappers_golden
from oracle import cost_ref, kalman_ref, lsap_ref, native, roi_wrappers_ref, tracker_ref


def test_roi_oracle_vs_golden():
    g = load_golden("roi")
    for tag in "abcd":
        ph, pw, sr, al = (int(v) for v in g["arg_" + tag])
        got = native.roi_align(g["feat"], g["rois"], (ph, pw), 20 / 640.0, sr, bool(al))
        assert_close(got, g["out_" + tag], what="roi " + tag)


def test_roi_wrapper_oracle_vs_golden():
    """tracking.py:193-221 and trainingCard.py:24-79 restated, against fixtures recorded from the reference's own
    methods (make_golden.py::run_roi_wrapper_cases)."""
    g = load_roi_wrappers_golden()
    for tag in ("sq", "wide"):
        feat, boxes, hw = g[tag + "_feat"], g[tag + "_boxes"], tuple(int(v) for v in g[tag + "_hw"])
        for ps in (7, 10):
            got = roi_wrappers_ref.roi_align_from_input_boxes(feat, boxes.tolist(), hw, out_size=(ps, ps))
            assert_close(got, g["%s_r1_%d" % (tag, ps)], what="%s r1 %d" % (tag, ps))
        assert_close(roi_wrappers_ref.preprocess_roi(feat, boxes, hw), g[tag + "_r2_10"], what=tag + " r2")
        assert_close(roi_wrappers_ref.preprocess_roi(feat, boxes, hw, output_size=(7, 7), enforce_min_size=0.0),
                     g[tag + "_r2_7_nomin"], what=tag + " r2 nomin")


def test_roi_oracle_vs_installed_torchvision():
    torch = pytest.importorskip("torch")
    tv = pytest.importorskip("torchvision")
    rng = np.random.default_rng(7)
    feat = rng.standard_normal((3, 8, 17, 23), dtype=np.float32)
    boxes = rng.uniform(-60, 800, (40, 4))
    rois = np.concatenate([rng.integers(0, 3, (40, 1)).astype(np.float64), boxes], 1).astype(np.float32)
    for ps, sr, al, sc in [((10, 10), 2, True, 17 / 544.0), ((7, 7), 0, False, 1 / 32.0), ((2, 9), 1, True, 0.05)]:
        want = tv.ops.roi_align(torch.from_numpy(feat), torch.from_numpy(rois), ps, sc, sr, al).numpy()
        assert_close(native.roi_align(feat, rois, ps, sc, sr, al), want, what="roi tv")


def test_lsap_oracle_vs_golden():
    g = load_golden("lsap")
    idx = 0
    while "m%d_C" % idx in g:
        p = "m%d_" % idx
        m, ut, ud = lsap_ref.hungarian_assign(g[p + "C"], cost_max=50.0)
        assert np.array_equal(np.array(m, dtype=np.int64).reshape(-1, 2), g[p + "matches"])
        assert ut == g[p + "ut"].tolist() and ud == g[p + "ud"].tolist()
        idx += 1
    assert idx == 8
    idx = 0
    while "tie%d_C" % idx in g:
        r, c = lsap_ref.linear_sum_assignment(g["tie%d_C" % idx])
        assert np.array_equal(r, g["tie%d_rows" % idx]) and np.array_equal(c, g["tie%d_cols" % idx])
        idx += 1
    assert idx == 4


def test_lsap_oracle_bit_exact_vs_installed_scipy():
    opt = pytest.importorskip("scipy.optimize")
    rng = np.random.default_rng(0)
    for trial in range(60):
        m, n = rng.integers(1, 40, 2)
        kind = trial % 4
        if kind == 0:
            C = rng.uniform(0, 2, (m, n)).astype(np.float32)
        elif kind == 1:
            C = rng.integers(0, 3, (m, n)).astype(np.float64)
        elif kind == 2:
            C = rng.uniform(0, 2, (m, n)).astype(np.float32)
            C[rng.uniform(size=(m, n)) < 0.8] = 1e9
        else:
            C = rng.normal(0, 100, (m, n))
        r, c = opt.linear_sum_assignment(C)
        r2, c2 = lsap_ref.linear_sum_assignment(C)
        assert np.array_equal(r, r2) and np.array_equal(c, c2), (trial, m, n)


def test_lsap_oracle_errors():
    with pytest.raises(ValueError):
        lsap_ref.linear_sum_assignment(np.array([[1.0, np.nan]]))
    with pytest.raises(ValueError):
        lsap_ref.linear_sum_assignment(np.array([[np.inf, np.inf], [1.0, 2.0]]))
    assert lsap_ref.hungarian_assign(np.zeros((0, 3))) == ([], [], [0, 1, 2])
    assert lsap_ref.hungarian_assign(np.zeros((2, 0))) == ([], [0, 1], [])
    assert lsap_ref.hungarian_assign(np.zeros((0, 0))) == ([], [], [])


def test_cost_oracle_vs_golden():
    g = load_golden("cost")
    for idx in range(4):
        p = "k%d_" % idx
        M = len(g[p + "cp"])
        N = len(g[p + "cq"])
        out = cost_ref.cal_cost(C_app=g[p + "Capp"], boxes_prev=g[p + "bp"].tolist(), boxes_cur=g[p + "bc"].tolist(),
                                input_hw=(640, 640), conf_prev=g[p + "cp"].tolist(), conf_cur=g[p + "cq"].tolist(),
                                assign=[(i % N) if i % 3 else -1 for i in range(M)])
        for key in ("C_total", "C_bbox", "C_center", "C_scale", "C_conf"):
            assert_close(out[key], g[p + key], what=key)
        assert abs(out["total_cost"] - float(g[p + "total_cost"])) <= 1e-5 * abs(float(g[p + "total_cost"]))


def test_kalman_oracle_vs_golden():
    g = load_golden("kalman")
    for idx in range(4):
        p = "t%d_" % idx
        kf = kalman_ref.init_kf_from_bbox(g[p + "box0"].tolist())
        for s in range(12):
            kf.predict()
            box = g[p + "boxes"][s].tolist()
            d_pre = kalman_ref.gating_distance_maha(kf, box)
            if g[p + "upd"][s]:
                kf.update(kalman_ref.bbox_xyxy_to_z(box))
            d_post = kalman_ref.gating_distance_maha(kf, box)
            assert_close(kf.x.reshape(-1), g[p + "x"][s], rtol=1e-12, atol=0, what="x")
            assert_close(kf.P, g[p + "P"][s], rtol=1e-12, atol=0, what="P")
            assert_close(d_pre, g[p + "d2pre"][s], rtol=1e-12, atol=0)
            assert_close(d_post, g[p + "d2post"][s], rtol=1e-12, atol=0)
        assert_close(kalman_ref.x_to_bbox_xyxy(kf.x.reshape(-1)), g[p + "pred_bbox"], rtol=1e-12, atol=0)
        # dtype migration of SURVEY.md section 8 row K
        assert kf.x.dtype == np.float64 and kf.P.dtype == np.float64


def test_kalman_shim_algebra():
    """The Joseph-form update must agree with the information-form posterior."""
    kf = kalman_ref.init_kf_from_bbox([10, 20, 50, 90])
    kf.predict()
    P, x = kf.P.astype(np.float64), kf.x.astype(np.float64)
    H, R = kf.H.astype(np.float64), kf.R.astype(np.float64)
    z = kalman_ref.bbox_xyxy_to_z([12, 21, 53, 95]).reshape(4, 1).astype(np.float64)
    P_info = np.linalg.inv(np.linalg.inv(P) + H.T @ np.linalg.inv(R) @ H)
    x_info = P_info @ (np.linalg.inv(P) @ x + H.T @ np.linalg.inv(R) @ z)
    kf.update(z.astype(np.float32))
    assert_close(kf.P, P_info, rtol=2e-3, atol=1e-3)
    assert_close(kf.x, x_info, rtol=1e-4, atol=1e-3)


def replay_tracker(name, make_tracker, compare_frame):
    g = load_golden("tracker_" + name)
    cfg = {k[4:]: float(g[k]) for k in g.files if k.startswith("cfg_")}
    for k in ("lost_reid_after", "max_age", "hist_max"):
        if k in cfg:
            cfg[k] = int(cfg[k])
    trk = make_tracker(cfg)
    n_stage2 = 0
    for f in range(int(g["n_frames"])):
        p = "f%03d_" % f
        obj = {"embs": [e for e in g[p + "embs"]], "bboxes": g[p + "boxes"].tolist(),
               "confs": g[p + "confs"].tolist(), "input_hw": (int(g["H"]), int(g["W"])), "frame_id": f}
        n_stage2 += compare_frame(trk, obj, g, p)
    return n_stage2


def _check_oracle_frame(trk, obj, g, p):
    trace = {}
    m, ut, ud = trk.update(obj, trace=trace)
    assert np.array_equal(np.array(m, dtype=np.int64).reshape(-1, 2), g[p + "matches"]), p
    assert list(ut) == g[p + "unmatched_tracks"].tolist(), p
    assert list(ud) == g[p + "unmatched_dets"].tolist(), p
    mats = [trace[k] for k in ("C_gated", "C_reid") if k in trace]
    for s, C in enumerate(mats):
        assert_close(C, g[p + "C%d" % s], what=p + "C%d" % s)
    assert (p + "C%d" % len(mats)) not in g
    if p + "st_ids" in g:
        ids = sorted(trk.tracks)
        assert ids == g[p + "st_ids"].tolist() and trk.next_id == int(g[p + "st_next_id"])
        assert_close([trk.tracks[i].kf.x.reshape(-1) for i in ids], g[p + "st_x"], rtol=1e-9, atol=1e-12)
        assert_close([trk.tracks[i].kf.P for i in ids], g[p + "st_P"], rtol=1e-9, atol=1e-12)
        assert_close([trk.tracks[i].ema for i in ids], g[p + "st_ema"], what="ema")
        assert [len(trk.tracks[i].bank) for i in ids] == g[p + "st_bank_len"].tolist()
        assert [trk.tracks[i].miss_count for i in ids] == g[p + "st_miss"].tolist()
        assert [trk.tracks[i].age for i in ids] == g[p + "st_age"].tolist()
        assert_close([trk.tracks[i].last_bbox for i in ids], g[p + "st_last_bbox"], rtol=1e-12, atol=0)
        for r, i in enumerate(ids):
            n = len(trk.tracks[i].bank)
            if n:
                assert_close(np.stack(trk.tracks[i].bank), g[p + "st_bank"][r, :n], what="bank")
    return int("C_reid" in trace)


@pytest.mark.parametrize("name,min_stage2", [("c1_steady", 0), ("churn", 3)])
def test_tracker_oracle_vs_golden(name, min_stage2):
    n2 = replay_tracker(name, lambda cfg: tracker_ref.TrackerRef(cfg), _check_oracle_frame)
    assert n2 >= min_stage2, "fixture no longer exercises the long-lost ReID stage"
