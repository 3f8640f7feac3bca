"""The rare branches of one iteration against the oracle, on problems where the oracle is seen to take them
(oracle_event_counts): the ACM-remark backtrack of subsm (src/lbfgsb.f90:2830-2879) -- which on the fused path
follows a speculative step and needs the direction pass of k_subsm_lsinit --, the 'ascent direction in
projection' restart of lnsrlb (:2247-2253, :734-769) -- which withdraws that speculative step --, skipped
updates and an abnormal termination of the line search."""
import numpy as np
import pytest

import harness as H
from oracle import oracle_py as O
from test_gpu_drivers import DISCRETE, RTOL_EARLY, RTOL_LATE

pytestmark = pytest.mark.gpu


def _run_pair(n, m, l_odd, x0, dtype, budget, tie_mode=0, tie_limit=None):
    import lbfgsb_b200
    import os

    def recorder(log):
        inner = H.iteration_budget_stop(budget)

        def stop(isave, dsave, f):
            log.append(O.event_counts(reset=False))
            return inner(isave, dsave, f)
        return stop
    O.set_sum_mode(1)
    O.set_tie_mode(tie_mode)
    try:
        O.event_counts()
        ev = []
        x, l, u, nbd = H.rosenbrock_problem(n, dtype=dtype, l_odd=l_odd, x0=x0)
        ref = H.run_driver(O.OracleSetulb(dtype), O.rosenbrock_fg, n, m, x, l, u, nbd, 0.0, 0.0, stop=recorder(ev))
        total = O.event_counts()
    finally:
        O.set_sum_mode(0)
        O.set_tie_mode(0)
    x, l, u, nbd = H.rosenbrock_problem(n, dtype=dtype, l_odd=l_odd, x0=x0)
    old = os.environ.get("LBFGSB_B200_TIE_LIMIT")
    if tie_limit is not None:
        os.environ["LBFGSB_B200_TIE_LIMIT"] = str(tie_limit)   # read when the workspace is created (host twin: at START)
    try:
        gpu = H.run_driver(lbfgsb_b200.HostSetulb(dtype), O.rosenbrock_fg, n, m, x, l, u, nbd, 0.0, 0.0,
                           stop=H.iteration_budget_stop(budget))
    finally:
        if tie_limit is not None:
            if old is None:
                del os.environ["LBFGSB_B200_TIE_LIMIT"]
            else:
                os.environ["LBFGSB_B200_TIE_LIMIT"] = old
    return gpu, ref, ev, total


def _first_event(ev, kind):
    """1-based iterate whose computation contained the first event of this kind."""
    prev = 0
    for k, c in enumerate(ev):
        if c[kind] > prev:
            return k + 1
        prev = c[kind]
    return None


def _compare(gpu, ref, upto, early=10):
    assert len(gpu[0]) >= upto and len(ref[0]) >= upto, (len(gpu[0]), len(ref[0]), gpu[1], ref[1])
    for a, b in list(zip(gpu[0], ref[0]))[:upto]:
        for kk in DISCRETE:
            assert a[kk] == b[kk], (kk, a, b)
        tol = RTOL_EARLY if b["iter"] <= early else RTOL_LATE
        assert abs(a["f"] - b["f"]) <= tol * abs(b["f"]) + 1e-300, (a, b)


CASES = [(1000, 5, 2.0, 3.0), (3001, 3, 2.5, 5.0), (50001, 3, 1.3, 5.0), (200000, 10, 1.3, 5.0), (200000, 5, 2.5, 5.0)]


@pytest.mark.parametrize("n,m,l_odd,x0", CASES)
def test_exit_inside_tied_breakpoints_follows_the_heap_and_backtrack_follows(n, m, l_odd, x0):
    """On these problems the Cauchy search of iteration 2 ends inside a group of equal breakpoints: the members of
    the group that get fixed are the first ones in hpsolb's pop order (heap replay on the device).  The partly
    fixed group then makes subsm's projected step an ascent direction and the ACM-remark backtrack runs -- on the
    fused path after a speculative step, with the direction pass of k_subsm_lsinit."""
    gpu, ref, ev, total = _run_pair(n, m, l_odd, x0, np.float64, 40)
    assert total[0] >= 1, "the oracle did not backtrack on this problem: the case no longer covers the branch"
    it = _first_event(ev, 0)
    assert it is not None and it > 1      # iter > 0: the fused subspace pass had stepped speculatively
    _compare(gpu, ref, min(len(ref[0]), it + 4))


def test_tie_exit_among_millions_of_breakpoints_is_replayed_on_the_host():
    """The same exit inside a group of equal breakpoints at n = 4e6 (2e6 breakpoints in the call, far beyond what one
    device thread can replay): the heap is popped on the engine's host thread from a copy of the breakpoint list, and the
    active set (hash) of every iterate equals the oracle's."""
    n, m, l_odd, x0 = 4_000_001, 3, 2.5, 5.0
    gpu, ref, ev, total = _run_pair(n, m, l_odd, x0, np.float64, 6)
    _compare(gpu, ref, min(len(ref[0]), 6))
    # the search of iteration 2 ends inside the tied group (nseg < breakpoints) and the tie order decides the active
    # set there: the oracle run with ties in variable order gives another set (otherwise the case proves nothing)
    assert 1 < ref[0][1]["nseg"] < n // 2
    O.set_sum_mode(1); O.set_tie_mode(1)
    try:
        x, l, u, nbd = H.rosenbrock_problem(n, l_odd=l_odd, x0=x0)
        other = H.run_driver(O.OracleSetulb(), O.rosenbrock_fg, n, m, x, l, u, nbd, 0.0, 0.0, stop=H.iteration_budget_stop(2))
    finally:
        O.set_sum_mode(0); O.set_tie_mode(0)
    assert other[0][1]["hash"] != ref[0][1]["hash"] and gpu[0][1]["hash"] == ref[0][1]["hash"]


@pytest.mark.parametrize("n,m,l_odd,x0", CASES[:3])
def test_without_heap_replay_ties_are_taken_in_variable_order(n, m, l_odd, x0):
    """Replay switched off (what happens beyond the replay limit and on sharded workspaces): the engine equals the
    oracle run with equal breakpoints taken in variable order -- the tie order is the only difference."""
    gpu, ref, ev, total = _run_pair(n, m, l_odd, x0, np.float64, 40, tie_mode=1, tie_limit=0)
    it = _first_event(ev, 0) or 2
    _compare(gpu, ref, min(len(ref[0]), it + 4))
    # and the two tie orders do differ on this problem (otherwise the case proves nothing)
    O.set_sum_mode(1)
    try:
        x, l, u, nbd = H.rosenbrock_problem(n, l_odd=l_odd, x0=x0)
        heap = H.run_driver(O.OracleSetulb(), O.rosenbrock_fg, n, m, x, l, u, nbd, 0.0, 0.0, stop=H.iteration_budget_stop(3))
    finally:
        O.set_sum_mode(0)
    assert heap[0][1]["hash"] != ref[0][1]["hash"]


def test_abnormal_termination_in_lnsrch_matches():
    gpu, ref, ev, total = _run_pair(1000, 10, 2.5, 3.0, np.float64, 40)
    assert ref[1].startswith("ABNORMAL_TERMINATION_IN_LNSRCH")
    it = _first_event(ev, 0) or 1
    _compare(gpu, ref, min(len(ref[0]), it + 4))
    assert gpu[1] == ref[1] or len(gpu[0]) >= it + 4


# (cases found with the oracle in REAL32 device-order mode, shape VEC = 2 / UNROLL = 8 of lbfgsb_b200_shape.h)
F32_ASCENT_CASES = [(1500, 5, 1.0, 3.0), (10000, 10, 1.0, 3.0), (3001, 20, 1.0, 5.0), (25000, 20, 1.0, 3.0), (1500, 20, 1.0, 3.0),
                    (1000, 3, 1.0, 3.0), (1000, 20, 1.0, 2.0), (4000, 20, 1.0, 2.0)]


def test_ascent_direction_restart_withdraws_speculative_step_f32():
    """REAL32 near convergence: lnsrlb meets gd >= 0 at its first entry, the memory is reset and the iteration
    restarts from the unchanged iterate.  Every run must stay a descent sequence from feasible points and end like
    the oracle's.  The oracle meets the event on every one of these problems; rounding decides whether the GPU run
    meets it on the same problem (the two sides differ in the order in which formk's entering/leaving rows are
    added), so the GPU is required to take the branch -- a restart shows as col dropping back -- on at least one."""
    gpu_restarts = 0
    for n, m, l_odd, x0 in F32_ASCENT_CASES:
        gpu, ref, ev, total = _run_pair(n, m, l_odd, x0, np.float32, 120)
        assert total[1] >= 1, ("the oracle met no ascent direction on this problem: the case no longer covers the branch", n, m, x0)
        assert total[2] >= 1, ("the oracle did not reset its memory on this problem", n, m, x0, total)
        fs = [r["f"] for r in gpu[0]]
        assert all(b <= a for a, b in zip(fs, fs[1:])), (n, m, x0, fs)
        assert gpu[1].split(":")[0] == ref[1].split(":")[0], (n, m, x0, gpu[1], ref[1])
        assert abs(gpu[3] - ref[3]) <= 1e-3 * max(abs(ref[3]), 1e-6), (n, m, x0, gpu[3], ref[3])
        cols = [r["col"] for r in gpu[0]]
        gpu_restarts += any(b < a for a, b in zip(cols, cols[1:]))
    assert gpu_restarts >= 1, "no GPU run restarted from an ascent direction: the branch is no longer covered on the device"


def test_fast_and_general_pipelines_agree_through_ascent_restarts():
    """The fast NEW_X pipeline (merged scalar kernels, one read-back) against the general one (LBFGSB_B200_NO_FAST=1) on
    the REAL32 problems above, whose runs restart from an ascent direction after a speculative step (x = t must be put
    back before the iteration restarts): every iterate bit for bit, and the final x."""
    import os
    import lbfgsb_b200
    restarts = 0
    for n, m, l_odd, x0 in F32_ASCENT_CASES + [(3001, 20, 1.0, 5.0), (50001, 10, 1.0, 5.0), (4000, 20, 1.0, 5.0)]:
        runs = []
        for no_fast in ("0", "1"):
            old = os.environ.get("LBFGSB_B200_NO_FAST")
            os.environ["LBFGSB_B200_NO_FAST"] = no_fast
            try:
                x, l, u, nbd = H.rosenbrock_problem(n, dtype=np.float32, l_odd=l_odd, x0=x0)
                runs.append(H.run_driver(lbfgsb_b200.HostSetulb(np.float32), O.rosenbrock_fg, n, m, x, l, u, nbd, 0.0, 0.0,
                                         stop=H.iteration_budget_stop(120)))
            finally:
                if old is None:
                    del os.environ["LBFGSB_B200_NO_FAST"]
                else:
                    os.environ["LBFGSB_B200_NO_FAST"] = old
        a, b = runs
        assert a[1] == b[1] and len(a[0]) == len(b[0]), (n, m, x0, a[1], b[1], len(a[0]), len(b[0]))
        for ra, rb in zip(a[0], b[0]):
            for k in H.TRACE_FIELDS:
                assert ra[k] == rb[k], (n, m, x0, k, ra, rb)
        assert np.array_equal(a[2], b[2])
        cols = [r["col"] for r in a[0]]
        restarts += any(q < p for p, q in zip(cols, cols[1:]))
    assert restarts >= 1, "no run restarted: the branch is not covered"
