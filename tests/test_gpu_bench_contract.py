"""bench.py on a GPU: one JSON line with the keys the driver reads (a short run on a small stream group)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_bench_line_has_the_contract_keys():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "4", "--warmup", "3", "--streams", "8",
                        "--no-extra", "--no-cpu-baseline"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, r.stdout[-2000:]
    d = json.loads(lines[0])
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
              "vs_baseline", "dtype", "data", "config", "clocks", "e2e", "gpu_launches", "roofline", "cpu_baseline"):
        assert k in d, k
    assert d["n_gpus"] == 1 and d["steps"] == 4 and d["value"] > 0 and d["higher_is_better"] is True
    assert d["gpu_launches"] > 0 and "workload" in d["config"]
    for k in ("value", "unit", "h2d_bytes_per_step", "d2h_bytes_per_step"):
        assert k in d["e2e"], k
    assert d["e2e"]["h2d_bytes_per_step"] > 0 and d["e2e"]["d2h_bytes_per_step"] > 0
    for k in ("bound", "achieved", "peak", "unit", "frac", "traffic"):
        assert k in d["roofline"], k
    assert d["roofline"]["bound"] == "hbm" and 0.0 < d["roofline"]["frac"] < 1.2


def test_bench_dump_outputs_is_repeatable(tmp_path):
    """--dump-outputs: float32 / float64 arrays of the last of exactly --steps timed steps, at most 64 MB, the same
    in two runs with the same arguments; the tracker results are the oracle's for that frame of the seeded scenes."""
    import bench
    from alufe_b200.tracking import R_HDR, R_NMATCH, R_NUD, R_NUT, R_STATUS
    from oracle import tracker_ref
    dumps = []
    for run in ("a", "b"):
        out = tmp_path / run
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "5", "--warmup", "3", "--streams",
                            "8", "--no-extra", "--no-cpu-baseline", "--dump-outputs", str(out)],
                           capture_output=True, text=True, timeout=600, cwd=ROOT)
        assert r.returncode == 0, r.stderr[-2000:]
        d = json.loads(r.stdout)
        assert d["steps"] == 5 and d["step_ms"]["n"] == 5
        dumps.append({f.name: np.load(f) for f in sorted(out.iterdir())})
    a, b = dumps
    assert sorted(a) == ["roi_align_patches.npy", "roi_align_rows.npy", "tracker_results.npy"]
    assert sum(v.nbytes for v in a.values()) <= 64 << 20
    for name, v in a.items():
        assert v.dtype in (np.float32, np.float64), name
        assert np.array_equal(v, b[name]), name
    assert a["roi_align_patches.npy"].shape == (128, 512, 10, 10) and np.abs(a["roi_align_patches.npy"]).max() > 0
    res = a["tracker_results.npy"].astype(np.int64)
    assert res.shape[0] == 8 and (res[:, R_STATUS] == 0).all() and (res[:, R_NMATCH] > 0).all()
    # stream s of the group is seeded s (rank 0); the last timed step is frame setup + warm-up + steps - 1
    sh = bench.WORKLOADS["c2"]
    last = d["setup_steps"] + d["warmup"] + d["steps"] - 1
    MD = sh.NBOX
    MT = res.shape[1] - R_HDR - 3 * MD
    for s in (0, 7):
        ref = tracker_ref.TrackerRef(tracker_ref.SHIPPED_CONF)
        for obj in bench.make_frames(sh, s, last + 1)[0]:
            want = ref.update(obj)
        row = res[s]
        nm, nut, nud = row[R_NMATCH], row[R_NUT], row[R_NUD]
        got = ([tuple(m) for m in row[R_HDR:R_HDR + 2 * nm].reshape(-1, 2).tolist()],
               row[R_HDR + 2 * MD:R_HDR + 2 * MD + nut].tolist(), row[R_HDR + 2 * MD + MT:R_HDR + 2 * MD + MT + nud].tolist())
        assert got == tuple(list(w) for w in want), "stream %d, frame %d" % (s, last)
