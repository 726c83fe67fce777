"""The oracle restatements against the original project on randomised hyper-parameters, scenes and matrices, beyond the
cases of test_oracle_golden.py: against the recorded outputs of these cases (tests/golden/live_fuzz.npz; where they
come from: make_golden.py::run_live_fuzz_cases) and, where the original's tree is mounted, against the original
itself.  This is
what pins oracle/tracker_ref.py, cost_ref.py and lsap_ref.py away from the shipped hyper-parameters; nothing on the
GPU / smoke / bench paths imports the original."""
import numpy as np
import pytest

from conftest import assert_close, load_golden
from golden import make_golden
from oracle import cost_ref, lsap_ref, reference_loader, tracker_ref


def _oracle_tracker(over):
    return tracker_ref.TrackerRef(dict(tracker_ref.SHIPPED_CONF, **over))


def _oracle_state(tr):
    return tr.kf.x, tr.kf.P, tr.ema, len(tr.bank), tr.miss_count, tr.age


def _oracle_cal_cost(**kw):
    return cost_ref.cal_cost(input_hw=(720, 1280), **kw)


def _recorded(prefix):
    g = load_golden("live_fuzz")
    return {k[len(prefix):]: g[k] for k in g.files if k.startswith(prefix)}


def _check_same(got, want, what):
    """Assignments, ids, counters and inputs exactly; Kalman states and embeddings within the parity bar."""
    assert sorted(got) == sorted(want), what
    for k in sorted(want):
        if "C_" in k or k.endswith(("_x", "_ema")):
            assert_close(got[k], want[k], what="%s %s" % (what, k))
        elif k.endswith("_P"):
            assert_close(got[k], want[k], rtol=1e-5, atol=1e-5, what="%s %s" % (what, k))
        elif k.endswith("inputs"):
            assert_close(got[k], want[k], rtol=1e-12, atol=0, what="%s %s: the seeded inputs changed" % (what, k))
        else:
            assert np.array_equal(got[k], want[k]), "%s %s" % (what, k)


@pytest.mark.parametrize("seed", range(6))
def test_tracker_oracle_vs_live_reference_fuzz(seed):
    """Random hyper-parameters and scene dynamics (misses, births, empty frames, the ReID-only stage): the oracle
    returns exactly what the reference's Tracking.update returns, frame by frame, and ends in the same state."""
    got = make_golden.record_tracker_fuzz(seed, _oracle_tracker, _oracle_state)
    _check_same(got, _recorded("t%d_" % seed), "seed %d vs recorded" % seed)
    if reference_loader.available():
        live = make_golden.record_tracker_fuzz(seed, make_golden.reference_tracker, make_golden.reference_state)
        _check_same(got, live, "seed %d vs live" % seed)


def test_cost_and_assignment_oracles_vs_live_reference_random():
    got = make_golden.record_cost_fuzz(_oracle_cal_cost, lsap_ref.hungarian_assign)
    _check_same(got, _recorded("cost_"), "cost vs recorded")
    if reference_loader.available():
        live = make_golden.record_cost_fuzz(make_golden.reference_cal_cost, reference_loader.load().hung.hungarian_assign)
        _check_same(got, live, "cost vs live")
