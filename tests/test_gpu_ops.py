"""GPU parity of the operator-level C ABI (cost, Kalman, assignment) against the oracle and the
golden fixtures produced by the live reference."""
import numpy as np
import pytest
import torch

from conftest import assert_close, load_golden
from oracle import cost_ref, kalman_ref, lsap_ref, native

pytestmark = pytest.mark.gpu

import alufe_b200  # noqa: E402,F401
from alufe_b200 import cost, hung, kalman, synth  # noqa: E402


# ---------------------------------------------------------------- assignment (bit-exact) ------
def _check_lsap(C, cost_max=50.0):
    want = lsap_ref.hungarian_assign(C, cost_max=cost_max)
    got = hung.hungarian_assign(C, cost_max=cost_max)
    assert got == want


def test_lsap_vs_golden():
    g = load_golden("lsap")
    for idx in range(8):
        p = "m%d_" % idx
        m, ut, ud = hung.hungarian_assign(g[p + "C"], cost_max=50.0)
        assert np.array_equal(np.array(m, dtype=np.int64).reshape(-1, 2), g[p + "matches"])
        assert ut == g[p + "ut"].tolist() and ud == g[p + "ud"].tolist()
    for idx in range(4):                     # scipy's tie-breaking, raw col_ind
        C = g["tie%d_C" % idx]
        col, _, st = hung.lsap_batched(torch.from_numpy(C).cuda()[None], 1e9)
        col = col[0].cpu().numpy()
        rows = np.nonzero(col >= 0)[0]
        assert int(st[0]) == 0
        assert np.array_equal(rows, g["tie%d_rows" % idx]) and np.array_equal(col[rows], g["tie%d_cols" % idx])


@pytest.mark.parametrize("m,n,gated", [(1, 1, 0), (8, 8, 0), (64, 64, 0), (64, 64, 0.9), (64, 64, 0.98), (100, 64, 0.9),
                                       (64, 100, 0.9), (128, 128, 0.5), (130, 257, 0.7), (300, 200, 0.9),
                                       (512, 512, 0.0), (512, 512, 0.9), (600, 700, 0.95)])
def test_lsap_vs_oracle_sizes(m, n, gated):
    rng = np.random.default_rng(m * 1000 + n)
    _check_lsap(synth.lsap_matrix(rng, m, n, gated))


def test_lsap_ties_and_degenerate_exact_vs_oracle():
    rng = np.random.default_rng(2)
    mats = [np.zeros((9, 9), np.float32), np.ones((5, 12), np.float32), np.full((40, 40), 1e9, np.float32)]
    mats += [rng.integers(0, 3, (m, n)).astype(np.float32) for m, n in [(17, 17), (33, 20), (20, 33), (70, 140)]]
    # 257..512 columns: the 16-columns-per-lane warp solver (ties, a NaN-free but -0.0 / inf-sprinkled matrix)
    mats += [rng.integers(0, 4, (m, n)).astype(np.float32) for m, n in [(260, 260), (300, 512), (400, 290), (512, 511)]]
    wide = rng.integers(0, 50, (384, 448)).astype(np.float32)
    wide[rng.random(wide.shape) < 0.3] = np.inf
    wide[np.arange(384), rng.permutation(448)[:384]] = -0.0
    mats.append(wide)
    for C in mats:
        c4r, _ = native.lsap(C)
        col, _, st = hung.lsap_batched(torch.from_numpy(C).cuda()[None], 1e9)
        assert int(st[0]) == 0 and np.array_equal(col[0].cpu().numpy().astype(np.int64), c4r)


@pytest.mark.parametrize("n", [8, 64, 100, 128, 200, 300, 512])
def test_lsap_known_first_step_shortcut_is_exact(n):
    """Tracker-like matrices: most rows have one clearly best column (the solvers skip their search), some
    rows compete for the same column (full search, duals move, later shortcuts must notice), some rows tie,
    some minima are -0.0 / +0.0 pairs.  Column-for-column equality with the scipy restatement."""
    rng = np.random.default_rng(n)
    mats = []
    for conflict, density in [(0.0, 0.02), (0.3, 0.05), (0.6, 0.3), (0.1, 1.0)]:
        m = n - n // 7
        C = np.full((m, n), 1e9, np.float32)
        mask = rng.random((m, n)) < density
        C[mask] = rng.uniform(0.5, 2.0, int(mask.sum())).astype(np.float32)
        perm = rng.permutation(n)[:m]
        clash = rng.random(m) < conflict
        perm[clash] = rng.choice(perm, int(clash.sum()))           # several rows want the same column
        C[np.arange(m), perm] = rng.uniform(0.05, 0.3, m).astype(np.float32)
        mats += [C, np.ascontiguousarray(C.T)]
    T = rng.integers(0, 5, (n, n)).astype(np.float32) + 1.0        # ties everywhere, unique minima in some rows
    rows = rng.choice(n, n // 2, replace=False)
    T[rows, rng.integers(0, n, n // 2)] = 0.5
    Z = rng.uniform(1, 2, (n, n)).astype(np.float32)               # -0.0 next to +0.0 must count as a tie
    Z[:, 0] = -0.0
    Z[:, n - 1] = 0.0
    mats += [T, Z]
    for C in mats:
        want, _ = native.lsap(C)
        col, _, st = hung.lsap_batched(torch.from_numpy(C).cuda()[None], 1e9)
        assert int(st[0]) == 0 and np.array_equal(col[0].cpu().numpy().astype(np.int64), want), C.shape


def test_lsap_batched_and_errors():
    rng = np.random.default_rng(4)
    C = np.stack([synth.lsap_matrix(rng, 40, 48, 0.6) for _ in range(9)])
    C[3, 2, 5] = np.nan
    C[5, 7, :] = np.inf                      # a row with no finite entry: infeasible (wide matrix)
    col, ok, st = hung.lsap_batched(torch.from_numpy(C).cuda(), 50.0)
    st = st.cpu().numpy()
    assert st[3] == -4 and st[5] == -5 and (np.delete(st, [3, 5]) == 0).all()
    for b in (0, 1, 2, 4, 6, 7, 8):
        want, _ = native.lsap(C[b])
        assert np.array_equal(col[b].cpu().numpy().astype(np.int64), want)
        m = [(i, int(want[i])) for i in range(40) if want[i] >= 0 and C[b, i, want[i]] <= 50.0]
        assert [i for i in range(40) if ok[b, i]] == [i for i, _ in m]
    with pytest.raises(ValueError):
        hung.hungarian_assign(np.array([[1.0, np.nan]], dtype=np.float32))
    with pytest.raises(ValueError):
        hung.hungarian_assign(np.array([[np.inf, np.inf], [1.0, 2.0]], dtype=np.float32))
    assert hung.hungarian_assign(np.zeros((0, 3))) == ([], [], [0, 1, 2])
    assert hung.hungarian_assign(np.zeros((2, 0))) == ([], [0, 1], [])
    assert hung.hungarian_assign(np.zeros((0, 0))) == ([], [], [])
    # cost_max is compared in float64 against the float32 entry (hung.py:36-37)
    C = np.array([[np.float32(0.4)]], dtype=np.float32)
    assert hung.hungarian_assign(C, cost_max=0.4) == lsap_ref.hungarian_assign(C, cost_max=0.4) == ([], [0], [0])


# ---------------------------------------------------------------- cost operators ---------------
def test_cost_ops_vs_golden():
    g = load_golden("cost")
    for idx in range(4):
        p = "k%d_" % idx
        M, N = len(g[p + "cp"]), len(g[p + "cq"])
        assign = [(i % N) if i % 3 else -1 for i in range(M)]
        out = cost.cal_cost(C_app=torch.from_numpy(g[p + "Capp"]).cuda(), boxes_prev=g[p + "bp"].tolist(),
                            boxes_cur=g[p + "bc"].tolist(), input_hw=(640, 640), conf_prev=g[p + "cp"].tolist(),
                            conf_cur=g[p + "cq"].tolist(), assign=assign)
        for key in ("C_total", "C_bbox", "C_center", "C_scale", "C_conf"):
            assert out[key].is_cuda
            assert_close(out[key].cpu().numpy(), g[p + key], what=key)
        assert abs(out["total_cost"] - float(g[p + "total_cost"])) <= 1e-5 * abs(float(g[p + "total_cost"]))
        bb = cost.bbox_cost(g[p + "bp"].tolist(), g[p + "bc"].tolist(), (640, 640), alpha=1.0, beta=0.5)
        assert_close(bb["C_bbox"].cpu().numpy(), g[p + "C_bbox"])
        assert_close(cost.conf_cost(g[p + "cp"].tolist(), g[p + "cq"].tolist()).cpu().numpy(), g[p + "C_conf"])
    z = cost.bbox_cost([], [[0, 0, 1, 1]], (1, 1))
    assert z["C_bbox"].shape == (0, 1)
    assert cost.conf_cost([0.5], []).shape == (1, 0)


@pytest.mark.parametrize("M,N,T", [(1, 1, 1), (8, 8, 30), (64, 64, 30), (13, 70, 6), (5, 129, 64), (40, 40, 33),
                                   # large enough for the tensor-core kernel (T <= 32, M * N >= 4096): ragged tiles in both
                                   # directions, full 32-row banks, short banks
                                   (100, 130, 30), (70, 64, 32), (200, 65, 7), (33, 257, 1), (512, 512, 30)])
def test_app_cost_vs_oracle(M, N, T):
    rng = np.random.default_rng(M + 7 * N + T)
    lens = rng.integers(0, T + 1, M)
    lens[0] = T
    if M > 2:
        lens[1], lens[2] = 0, 1
    bank = rng.standard_normal((M, T, 128)).astype(np.float32)
    bank /= np.linalg.norm(bank, axis=2, keepdims=True)
    ema = rng.standard_normal((M, 128)).astype(np.float32)
    det = rng.standard_normal((N, 128)).astype(np.float32) * 3.0      # not unit: re-normalised inside
    banks = [[bank[i, t] for t in range(lens[i])] for i in range(M)]
    for topk, mean, fb in [(5, True, True), (5, True, False), (3, False, True), (50, True, True)]:
        want = cost_ref.app_cost_topk(banks, list(det), topk=topk, use_topk_mean=mean,
                                      fallback_embs=list(ema) if fb else None)
        got = cost.app_cost_topk(torch.from_numpy(bank).cuda(), torch.from_numpy(lens.astype(np.int32)).cuda(),
                                 torch.from_numpy(det).cuda(), topk=topk, use_topk_mean=mean,
                                 fallback=torch.from_numpy(ema).cuda() if fb else None)
        assert_close(got.cpu().numpy(), want, rtol=1e-5, atol=2e-6, what="C_app")


# nseg = the number of segments each bank tile's walk is split into on 148 SMs: clamp(148 // m_tiles, 1, n_tiles) with
# m_tiles = ceil(M / 4) bank tiles and n_tiles = ceil(N / 64) detection tiles.  Every shape has M * N >= 64 * 64.
@pytest.mark.parametrize("M,N,T", [(260, 130, 30),     # nseg 2: segments of 2 and 1 steps (ragged last segment)
                                   (300, 64, 9),       # nseg 1: 75 bank tiles, one step
                                   (512, 512, 30),     # nseg 1: BASELINE config 4, 8 steps
                                   (70, 64, 32),       # nseg 1: 18 bank tiles but a single detection tile
                                   (257, 1000, 32),    # nseg 2: 8 steps each
                                   (392, 512, 30),     # nseg 1: 98 bank tiles, 8 steps
                                   (16, 260, 30),      # nseg 5 = n_tiles < 148 // 4: segments of exactly one step
                                   (100, 900, 30),     # nseg 5: segments of exactly three steps
                                   (40, 2000, 32),     # nseg 14: segments of 3 and 2 steps, ragged last tile
                                   (64, 4096, 30)])    # nseg 9 < n_tiles = 64: segments of 8 and 7 steps
def test_app_cost_tensor_core_kernels_vs_oracle(M, N, T):
    """The tcgen05 dense appearance cost (a CTA per bank tile and segment keeps its bank image resident and walks the
    segment's detection tiles: two TMEM accumulators, the tensor core one tile ahead of the epilogue) on every case of
    its launch: one segment, several, ragged, of one step and of enough steps that both buffers and both accumulators
    are reused.  Ragged tiles in both directions, empty / short / full banks, the EMA fallback, top-k beyond five and
    the max-similarity variant.  Each call is the two tensor-core launches (prep + walk), not the float32 kernel."""
    rng = np.random.default_rng(3 * M + 11 * N + T)
    lens = rng.integers(0, T + 1, M)
    lens[0], lens[1], lens[2], lens[M - 1] = T, 0, 1, T
    bank = rng.standard_normal((M, T, 128)).astype(np.float32)
    ema = rng.standard_normal((M, 128)).astype(np.float32)
    det = rng.standard_normal((N, 128)).astype(np.float32) * 0.3
    banks = [[bank[i, t] for t in range(lens[i])] for i in range(M)]
    lib = alufe_b200._lib.lib()
    for topk, mean, fb in [(5, True, True), (5, True, False), (1, False, True), (9, True, True)]:
        want = cost_ref.app_cost_topk(banks, list(det), topk=topk, use_topk_mean=mean,
                                      fallback_embs=list(ema) if fb else None)
        launches = lib.b200_launch_count()
        got = cost.app_cost_topk(torch.from_numpy(bank).cuda(), torch.from_numpy(lens.astype(np.int32)).cuda(),
                                 torch.from_numpy(det).cuda(), topk=topk, use_topk_mean=mean,
                                 fallback=torch.from_numpy(ema).cuda() if fb else None)
        assert lib.b200_launch_count() - launches == 2
        assert_close(got.cpu().numpy(), want, rtol=1e-5, atol=2e-6, what="C_app topk %d" % topk)


def test_app_cost_c4_size_properties():
    """512 x 512 x 30 banks (BASELINE config 4): a track whose bank holds a detection's own
    embedding k times scores exactly that detection with cost ~0; costs lie in [0, 2]."""
    rng = np.random.default_rng(0)
    M = N = 512
    det = rng.standard_normal((N, 128)).astype(np.float32)
    det /= np.linalg.norm(det, axis=1, keepdims=True)
    bank = rng.standard_normal((M, 30, 128)).astype(np.float32)
    bank /= np.linalg.norm(bank, axis=2, keepdims=True)
    bank[:, :5] = det[:, None, :]
    lens = torch.full((M,), 30, dtype=torch.int32).cuda()
    C = cost.app_cost_topk(torch.from_numpy(bank).cuda(), lens, torch.from_numpy(det).cuda()).cpu().numpy()
    assert np.abs(np.diag(C)).max() < 1e-5 and C.min() > -1e-5 and C.max() < 2.0 + 1e-5
    assert (np.argmin(C, axis=1) == np.arange(M)).all()
    want = cost_ref.app_cost_topk([list(bank[i]) for i in range(M)], list(det))
    assert_close(C, want, rtol=1e-5, atol=2e-6)


# ---------------------------------------------------------------- Kalman -------------------------
def test_kalman_vs_golden_stepwise():
    g = load_golden("kalman")
    for idx in range(4):
        p = "t%d_" % idx
        kf = kalman.init_kf_from_bbox(g[p + "box0"].tolist())
        for s in range(12):
            kf.predict()
            box = g[p + "boxes"][s].tolist()
            d_pre = kalman.gating_distance_maha(kf, box)
            if g[p + "upd"][s]:
                kf.update(kalman.bbox_xyxy_to_z(box))
            d_post = kalman.gating_distance_maha(kf, box)
            assert_close(kf.x_host.reshape(-1), g[p + "x"][s], rtol=1e-5, atol=1e-7, what="x step %d" % s)
            assert_close(kf.P_host, g[p + "P"][s], rtol=1e-5, atol=1e-6, what="P step %d" % s)
            assert_close(d_pre, g[p + "d2pre"][s], rtol=1e-5, atol=1e-9)
            assert_close(d_post, g[p + "d2post"][s], rtol=1e-5, atol=1e-9)
        assert kf.x_host.dtype == np.float64 and kf.P_host.dtype == np.float64
        assert_close(kalman.x_to_bbox_xyxy(kf.x_host.reshape(-1)), g[p + "pred_bbox"], rtol=1e-5, atol=1e-6)


def test_kalman_batched_vs_oracle_from_identical_state():
    """Per-step parity from identical inputs (what BASELINE.json north_star asks): many tracks,
    mixed update masks, so all three dtype stages are live in one launch."""
    rng = np.random.default_rng(1)
    M = 300
    boxes = synth.random_boxes(rng, M, 1280, 1280)
    ref = [kalman_ref.init_kf_from_bbox(b.tolist()) for b in boxes]
    bk = kalman.BatchedKalman(boxes)
    for step in range(6):
        pb = bk.predict(want_boxes=True).cpu().numpy()
        for i, kf in enumerate(ref):
            kf.predict()
        want_pb = np.array([kalman_ref.x_to_bbox_xyxy(kf.x.reshape(-1)) for kf in ref])
        assert_close(pb, want_pb, rtol=1e-5, atol=1e-5, what="pred boxes")
        boxes = boxes + rng.normal(0, 2.0, boxes.shape)
        sel = rng.uniform(size=M) < 0.6
        det_of = np.where(sel, rng.permutation(M), -1).astype(np.int32)
        d2 = bk.maha(boxes).cpu().numpy()
        pick = rng.choice(M, 12, replace=False)
        for i in pick:
            for j in pick:
                assert_close(d2[i, j], kalman_ref.gating_distance_maha(ref[i], boxes[j].tolist()), rtol=1e-5, atol=1e-9)
        bk.update(det_of, boxes)
        for i, kf in enumerate(ref):
            if det_of[i] >= 0:
                kf.update(kalman_ref.bbox_xyxy_to_z(boxes[det_of[i]].tolist()))
        x = bk.x.cpu().numpy()
        P = bk.P.cpu().numpy()
        assert_close(x, np.array([kf.x.reshape(-1) for kf in ref]), rtol=1e-5, atol=1e-6, what="x")
        assert_close(P, np.array([kf.P for kf in ref]), rtol=1e-5, atol=1e-5, what="P")
        # carry the oracle's state over so that every step starts from identical inputs
        bk.x.copy_(torch.from_numpy(np.array([kf.x.reshape(-1).astype(np.float64) for kf in ref])))
        bk.P.copy_(torch.from_numpy(np.array([kf.P.astype(np.float64) for kf in ref])))
        stage = bk.stage.cpu().numpy()
        assert [int(s) for s in stage] == [int(kf.x.dtype == np.float64) + int(kf.P.dtype == np.float64) for kf in ref]


def test_maha_gate_in_place():
    rng = np.random.default_rng(3)
    boxes = synth.random_boxes(rng, 20, 640, 640)
    bk = kalman.BatchedKalman(boxes)
    bk.predict()
    dets = boxes + rng.normal(0, 30.0, boxes.shape)
    C = torch.rand((20, 20), device="cuda")
    C0 = C.clone()
    d2 = bk.maha(dets, C=C, maha_thr=9.49, INF=1e9)
    far = d2 > 9.49
    assert torch.equal(C[far], torch.full_like(C[far], 1e9)) and torch.equal(C[~far], C0[~far])
    assert far.any() and (~far).any()
