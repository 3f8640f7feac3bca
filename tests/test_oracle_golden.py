"""Pins the CPU oracle against the reference's own golden outputs
(test/OUTPUTS/output_90_{1,2,3}, iterate.dat -> tests/golden/reference_outputs.json).

Discrete quantities (iteration count, nfg per iterate, nseg, nact, sub, itls, Tnint, Skip,
termination message) must match exactly.  Printed reals must match digit-for-digit while the
reference's own two builds (output_77_* vs output_90_*) still agree with each other, and
within the drift those two builds show afterwards (SURVEY.md section 4: summation/contraction
order alone moves the late iterates).
"""
import numpy as np
import pytest

import harness as H
from oracle import oracle_py as O


def _run(n, m, factr, pgtol, stop=None, l_odd=1.0):
    x, l, u, nbd = H.rosenbrock_problem(n, l_odd=l_odd)
    s = O.OracleSetulb()
    return H.run_driver(s, O.rosenbrock_fg, n, m, x, l, u, nbd, factr, pgtol, stop=stop)


def _d2f(s):
    return float(s.replace("D", "E"))


def test_driver1_matches_output_90_1_and_iterate_dat(golden):
    tr, task, x, f, isave, dsave = _run(25, 5, 1.0e7, 1.0e-5)
    g = golden["driver1_90"]
    assert task == g["task"]
    assert len(tr) == g["summary"]["tit"] == 23
    assert tr[-1]["nfgv"] == g["summary"]["tnf"] == 28
    assert int(isave[21]) == g["summary"]["tnint"] == 47      # isave(22) = nintol
    assert int(isave[25]) == g["summary"]["skip"] == 0        # isave(26) = nskip
    assert tr[-1]["nact"] == g["summary"]["nact"] == 0
    # every printed iterate, digit for digit (1p,d12.5)
    for row, ref in zip(tr, g["iterates"][1:]):
        assert row["iter"] == ref["iter"]
        assert H.fortran_d(row["f"], 12, 5).strip() == ref["f_str"], row
        assert H.fortran_d(row["sbgnrm"], 12, 5).strip() == ref["pg_str"], row
    # F to >= 10 significant digits (the reference's F77 and F90 builds differ at 5e-11)
    assert abs(f - g["final_f"]) / g["final_f"] < 1e-10
    assert abs(golden["driver1_77"]["final_f"] - g["final_f"]) / g["final_f"] > 1e-11
    # iterate.dat: it nf nseg nact sub itls stepl tstep projg f
    word = {0: "con", 1: "bnd", 5: "TNT"}
    for row, ref in zip(tr, golden["iterate_dat"][1:]):
        assert row["iter"] == ref["it"] and row["nfgv"] == ref["nf"]
        assert str(row["nseg"]) == ref["nseg"] and str(row["nact"]) == ref["nact"]
        assert word.get(row["iword"], "---") == ref["sub"]
        assert str(row["iback"]) == ref["itls"]
        assert H.fortran_d(row["stp"], 7, 1).strip() == ref["stepl"]
        assert H.fortran_d(row["xstep"], 7, 1).strip() == ref["tstep"]
        assert H.fortran_d(row["sbgnrm"], 10, 3).strip() == ref["projg"]
        assert H.fortran_d(row["f"], 10, 3).strip() == ref["f"]


def _check_driver23(tr, task, x, g90, g77, exact_upto):
    assert task == g90["task"]
    assert len(tr) == len(g90["iterates"])
    for row, r90, r77 in zip(tr, g90["iterates"], g77["iterates"]):
        assert row["iter"] == r90["iter"] and row["nfgv"] == r90["nfg"]
        f90, p90, f77, p77 = _d2f(r90["f_str"]), _d2f(r90["pg_str"]), _d2f(r77["f_str"]), _d2f(r77["pg_str"])
        if row["iter"] <= exact_upto:
            assert H.fortran_d(row["f"], 12, 5).strip() == r90["f_str"], row
            assert H.fortran_d(row["sbgnrm"], 12, 5).strip() == r90["pg_str"], row
        else:
            # late iterates: within a small multiple of the drift between the reference's own builds
            assert abs(row["f"] - f90) <= 4 * abs(f90 - f77) + 2e-3 * abs(f90), row
            assert abs(row["sbgnrm"] - p90) <= 4 * abs(p90 - p77) + 2e-2 * abs(p90), row
    xr = np.array([_d2f(s) for s in g90["final_x_str"]])
    assert xr.shape == x.shape
    assert np.max(np.abs(x - xr)) <= 5.1e-5 * max(1.0, np.max(np.abs(xr)))   # printed to 5 digits


def test_driver2_matches_output_90_2(golden):
    tr, task, x, f, isave, dsave = _run(25, 5, 0.0, 0.0, stop=H.driver2_stop(99))
    assert len(tr) == 46 and tr[-1]["nfgv"] == 53
    _check_driver23(tr, task, x, golden["driver2_90"], golden["driver2_77"], exact_upto=34)


def test_driver3_matches_output_90_3(golden):
    tr, task, x, f, isave, dsave = _run(1000, 10, 0.0, 0.0, stop=H.driver2_stop(900))
    assert len(tr) == 49 and tr[-1]["nfgv"] == 58
    _check_driver23(tr, task, x, golden["driver3_90"], golden["driver3_77"], exact_upto=30)


def test_float32_build_runs_driver1():
    """-DREAL32 analogue (lbfgsb_kinds_module.F90:29-37): epsmch = epsilon(1.0_real32)."""
    x, l, u, nbd = H.rosenbrock_problem(25, dtype=np.float32)
    s = O.OracleSetulb(np.float32)
    tr, task, x, f, isave, dsave = H.run_driver(s, O.rosenbrock_fg, 25, 5, x, l, u, nbd, 10.0, 1.0e-3)
    assert task.startswith("CONVERGENCE") or task.startswith("ABNORMAL")
    assert abs(float(dsave[4]) - 1.1920929e-07) < 1e-12
    assert f < 1.0e-3


def test_device_order_sum_mode_same_discrete_trace():
    """Summation order alone must not move the discrete trace on the sample problem."""
    ref = _run(1000, 10, 0.0, 0.0, stop=H.driver2_stop(900))[0]
    O.set_sum_mode(1)
    try:
        dev = _run(1000, 10, 0.0, 0.0, stop=H.driver2_stop(900))[0]
    finally:
        O.set_sum_mode(0)
    n = min(len(ref), len(dev), 30)
    for a, b in zip(ref[:n], dev[:n]):
        for k in ("iter", "nfgv", "nseg", "nact", "nfree", "iword", "iback", "hash"):
            assert a[k] == b[k], (k, a, b)
        assert abs(a["f"] - b["f"]) <= 1e-6 * abs(a["f"]) + 1e-18


@pytest.mark.parametrize("n,m,l_odd,factr,pgtol", [(1_000_000, 5, 1.0, 1.0e7, 1.0e-5), (400_000, 10, 1.1, 0.0, 0.0)])
def test_device_order_vs_reference_order_at_config_sizes(n, m, l_odd, factr, pgtol):
    """Leg (ii) of the parity chain at the size of BASELINE.json configs[1] (n = 1e6, m = 5, the reference's stopping
    test) and on the configs[2] problem (odd lower bound 1.1, m = 10, fixed budget): the oracle in the reference's
    summation order and in the device's order (the mode the GPU is gated against) take the same number of iterations
    and the same discrete decisions at every iterate (nseg, free/active counts, entering/leaving counts, line-search
    trials, active-set identity); the drift of f, which summation order alone causes, is bounded and printed."""
    stop = None if factr > 0 else H.iteration_budget_stop(25)

    def run():
        x, l, u, nbd = H.rosenbrock_problem(n, l_odd=l_odd)
        return H.run_driver(O.OracleSetulb(), O.rosenbrock_fg, n, m, x, l, u, nbd, factr, pgtol, stop=stop)
    ref = run()
    O.set_sum_mode(1)
    try:
        dev = run()
    finally:
        O.set_sum_mode(0)
    assert ref[1] == dev[1], (ref[1], dev[1])
    assert len(ref[0]) == len(dev[0]), (len(ref[0]), len(dev[0]))
    worst = 0.0
    for a, b in zip(ref[0], dev[0]):
        for k in ("iter", "nfgv", "nseg", "nact", "nfree", "nenter", "nleave", "iword", "iback", "col", "nskip", "hash", "hcount"):
            assert a[k] == b[k], (k, a, b)
        rel = abs(a["f"] - b["f"]) / max(abs(a["f"]), 1e-300)
        worst = max(worst, rel)
        assert rel <= (1e-10 if a["iter"] <= 5 else 1e-5), (a["iter"], rel)
    print("n=%d m=%d: %d iterates, identical discrete trace; worst relative drift of f from summation order alone: %.2e" % (
        n, m, len(ref[0]), worst))


@pytest.mark.parametrize("bad", ["nbd", "lu", "factr", "m"])
def test_errclb_messages(bad):
    """errclb :1601-1643 -- later errors overwrite earlier ones; k = last offending index."""
    n, m = 10, 3
    x, l, u, nbd = H.rosenbrock_problem(n)
    factr = 1e7
    if bad == "nbd":
        nbd[3] = 7
        nbd[6] = -1
        want, k = "ERROR: INVALID NBD", 7
    elif bad == "lu":
        nbd[2] = 5
        l[8] = 200.0
        want, k = "ERROR: NO FEASIBLE SOLUTION", 9
    elif bad == "factr":
        factr = -1.0
        want, k = "ERROR: FACTR < 0", 0
    else:
        m = 0
        want, k = "ERROR: M <= 0", 0
    s = O.OracleSetulb()
    mm = max(m, 1)
    wa, iwa = s.workspace(n, mm)
    task = H.make_task("START")
    csave = H.make_task("")
    lsave = np.zeros(4, np.int32)
    isave = np.zeros(44, np.int32)
    dsave = np.zeros(29)
    f = np.zeros(1)
    g = np.zeros(n)
    s(n, m, x, l, u, nbd, f, g, factr, 1e-5, wa, iwa, task, -1, csave, lsave, isave, dsave)
    assert H.task_str(task) == want
    assert int(isave[41]) == k


def test_event_counters_memory_reset_and_skipped_update():
    """oracle_event_counts slots 2 (mainlb's "refresh the lbfgs memory" restarts) and 3 (skipped updates, :826-834)
    fire on problems known to take those branches, and stay at zero on one that takes neither."""
    from test_gpu_edge import _nonconvex
    O.set_sum_mode(1)
    try:
        # REAL32 sample problem near convergence: lnsrlb meets an ascent direction with pairs in the memory
        O.event_counts()
        n, m = 1500, 5
        x, l, u, nbd = H.rosenbrock_problem(n, dtype=np.float32)
        H.run_driver(O.OracleSetulb(np.float32), O.rosenbrock_fg, n, m, x, l, u, nbd, 0.0, 0.0,
                     stop=H.iteration_budget_stop(120), want_hash=False)
        ev = O.event_counts()
        assert ev[1] >= 1 and ev[2] >= ev[1], ev
        # a concave share: s'y <= 0 along the step, the update is skipped
        n, m = 400, 5
        fg, mk = _nonconvex(n, 0, 0.5, 0.3)
        x, l, u, nbd = mk()
        tr = H.run_driver(O.OracleSetulb(), fg, n, m, x, l, u, nbd, 0.0, 0.0, stop=H.iteration_budget_stop(30),
                          want_hash=False)
        ev = O.event_counts()
        assert ev[3] >= 1 and ev[3] == tr[0][-1]["nskip"], (ev, tr[0][-1])
        # driver1: neither
        x, l, u, nbd = H.rosenbrock_problem(25)
        H.run_driver(O.OracleSetulb(), O.rosenbrock_fg, 25, 5, x, l, u, nbd, 1.0e7, 1.0e-5, want_hash=False)
        assert O.event_counts()[2:4] == [0, 0]
    finally:
        O.set_sum_mode(0)
