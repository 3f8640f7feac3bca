"""The task loop of a batch on the device (lbfgsb_batch_minimize_graph_*, BatchProblem.solve_graph) against the same loop
run call by call on the host (BatchProblem.solve, or for max_fg the small host loop `host_solve` below that applies
limit_stop's rule), with the same objective -- the batched sample objective, masked by the batch's fg_mask -- on fresh
copies of the same inputs.  Every comparison is bit for bit: x, g and f; task, csave, lsave, isave, dsave and iwhere;
and the number of calls."""
import numpy as np
import pytest

import harness as H
from test_gpu_lockstep import _bits, far_box, unbounded

F64, F32 = np.float64, np.float32
STOP_ITER = "STOP: TOTAL NO. of ITERATIONS REACHED LIMIT"
STOP_FG = "STOP: TOTAL NO. of f AND g EVALUATIONS EXCEEDS LIMIT"
CALL_CAP = 128      # calls per graph launch (BatchEngine::kLoopCallCap)


# ---------------------------------------------------------------------------------------------------------------------
# problems: the families of test_gpu_batch_lockstep.py whose objective is the sample objective, and two that fail errclb


def _walk(n, dtype, seed):
    rng = np.random.default_rng(seed)
    x, l, u, nbd = H.rosenbrock_problem(n, dtype=dtype, l_odd=(1.1, 1.5)[seed % 2])
    return (x + 0.25 * rng.uniform(-1.0, 1.0, n)).astype(dtype), l, u, nbd


def _ties(n, dtype, seed):
    l_odd, x0 = ((2.0, 3.0), (2.5, 5.0))[seed % 2]
    return H.rosenbrock_problem(n, dtype=dtype, l_odd=l_odd, x0=x0)


def _err_infeasible(n, dtype, seed):
    x, l, u, nbd = far_box(n, dtype)
    l[n // 2] = u[n // 2] + 1.0         # l > u with nbd = 2: 'ERROR: NO FEASIBLE SOLUTION'
    return x, l, u, nbd


def _err_nbd(n, dtype, seed):
    x, l, u, nbd = far_box(n, dtype)
    nbd[n - 1] = 5                      # 'ERROR: INVALID NBD'
    return x, l, u, nbd


FAM = {"far": lambda n, dt, s: far_box(n, dt), "nbd0": lambda n, dt, s: unbounded(n, dt), "walk": _walk, "ties": _ties,
       "err_lu": _err_infeasible, "err_nbd": _err_nbd}
MIX = [("far", 0), ("walk", 0), ("walk", 1), ("ties", 0), ("ties", 1), ("nbd0", 0), ("err_lu", 0), ("err_nbd", 0)]


def make_batch(n, dtype, spec):
    cols = [FAM[f](n, np.dtype(dtype), s) for f, s in spec]
    return tuple(np.ascontiguousarray(np.stack([c[k] for c in cols])) for k in range(4))


def _tensors(X, L, U, N):
    import torch
    tdt = torch.float64 if X.dtype == F64 else torch.float32
    P, n = X.shape
    xd, ld, ud, nd = (torch.from_numpy(np.ascontiguousarray(a)).cuda() for a in (X, L, U, N))
    return xd, ld, ud, nd, torch.zeros(P, dtype=tdt, device="cuda"), torch.zeros((P, n), dtype=tdt, device="cuda")


def state_of(b, xd, fd, gd):
    """Everything the comparison looks at, as bit patterns and bytes."""
    return {"x": _bits(xd.cpu().numpy()), "g": _bits(gd.cpu().numpy()), "f": _bits(fd.cpu().numpy()),
            "task": b.task.copy(), "csave": b.csave.copy(), "lsave": b.lsave.copy(), "isave": b.isave.copy(),
            "dsave": _bits(b.dsave), "iwhere": b.iwhere()}


def assert_same(got, want, what=""):
    for k in want:
        a, w = got[k], want[k]
        if not np.array_equal(a, w):
            bad = np.argwhere(a != w)[0]
            raise AssertionError("%s%s differs first at %s: %r vs %r" % (what, k, tuple(bad), a[tuple(bad)], w[tuple(bad)]))


def host_solve(b, xd, ld, ud, nd, fd, gd, factr, pgtol, max_iter=0, max_fg=0):
    """solve's loop with limit_stop's rule (engine.cu) at NEW_X: max_iter before max_fg."""
    calls = 0
    while True:
        b.setulb_dev(xd, ld, ud, nd, fd, gd, factr, pgtol)
        calls += 1
        nfg, nnew, _ = b.counts()
        if nfg == 0 and nnew == 0:
            return calls
        if nfg:
            b.rosenbrock_fg(xd, gd, fd)
        for p in np.nonzero(b.task[:, 0] == ord("N"))[0]:
            text = None
            if max_fg > 0 and b.isave[p, 33] >= max_fg:
                text = STOP_FG
            if max_iter > 0 and b.isave[p, 29] >= max_iter:
                text = STOP_ITER
            if text:
                b.set_task(int(p), text)


def run_solve(m, X, L, U, N, factr, pgtol, max_iter=0, max_fg=0, cols=None):
    """Reference: solve (or host_solve when max_fg is set) on a fresh batch; cols collects isave col at every NEW_X."""
    import lbfgsb_b200
    P, n = X.shape
    xd, ld, ud, nd, fd, gd = _tensors(X, L, U, N)
    b = lbfgsb_b200.BatchProblem(P, n, m, X.dtype)
    try:
        if max_fg:
            calls = host_solve(b, xd, ld, ud, nd, fd, gd, factr, pgtol, max_iter, max_fg)
        else:
            def on_newx(bp):
                if cols is not None:
                    for p in np.nonzero(bp.task[:, 0] == ord("N"))[0]:
                        cols[p].append(int(bp.isave[p, 27]))
            calls = b.solve(xd, ld, ud, nd, fd, gd, factr, pgtol, max_iter=max_iter, on_newx=on_newx)
        return state_of(b, xd, fd, gd), calls
    finally:
        b.close()


def run_graph(m, X, L, U, N, factr, pgtol, max_iter=0, max_fg=0):
    import lbfgsb_b200
    P, n = X.shape
    xd, ld, ud, nd, fd, gd = _tensors(X, L, U, N)
    b = lbfgsb_b200.BatchProblem(P, n, m, X.dtype)
    try:
        calls = b.solve_graph(xd, ld, ud, nd, fd, gd, factr, pgtol, max_iter=max_iter, max_fg=max_fg)
        assert b.counts() == (0, 0, P)
        return state_of(b, xd, fd, gd), calls, b.graph_stats()
    finally:
        b.close()


def _kinds(state):
    return {bytes(t).decode().split(":")[0].split(" ")[0] for t in state["task"]}


# ---------------------------------------------------------------------------------------------------------------------
# cover: sizes, both real kinds, all three pass instances (m 1-5, 6-10, 11-20), problems that end at different calls

# (n, m, real kind, factr, pgtol, max_iter).  REAL32 takes factr = 10: with driver1's 1e7 the stopping tolerance
# factr * epsmch is about 1.2 in single precision and every problem converges after one iteration.  max_iter lies between
# the iterations at which the problems of the mix end on their own, so that in every batch some converge and some stop at
# the limit (test_cover_cases_converge_and_stop checks this with the oracle).
COVER = [
    (25, 5, F64, 1.0e7, 1.0e-5, 40),
    (25, 20, F32, 10.0, 1.0e-5, 40),
    (2049, 1, F32, 10.0, 1.0e-5, 30),
    (2049, 10, F64, 1.0e7, 1.0e-5, 30),
    (4097, 17, F32, 10.0, 1.0e-5, 25),
    (4097, 20, F64, 1.0e7, 1.0e-5, 35),
    (65536, 17, F64, 1.0e7, 1.0e-5, 20),
    (131072, 10, F32, 10.0, 1.0e-5, 12),
]


@pytest.mark.gpu
@pytest.mark.parametrize("case", COVER, ids=lambda c: "n%d-m%d-%s" % (c[0], c[1], "f64" if c[2] == F64 else "f32"))
def test_solve_graph_matches_solve(case):
    n, m, dtype, factr, pgtol, max_iter = case
    X, L, U, N = make_batch(n, dtype, MIX)
    want, want_calls = run_solve(m, X, L, U, N, factr, pgtol, max_iter=max_iter)
    got, calls, stats = run_graph(m, X, L, U, N, factr, pgtol, max_iter=max_iter)
    assert_same(got, want)
    assert calls == want_calls and stats[0] == 1 and stats[2] == calls
    kinds = _kinds(want)
    assert {"CONVERGENCE", "STOP", "ERROR"} <= kinds, kinds      # the problems of the batch end at different calls


@pytest.mark.gpu
@pytest.mark.parametrize("n,m,l_odd,x0,dtype,max_iter", [
    (2049, 5, 1.0, 3.0, F32, 45),       # gd >= 0 at lnsrlb's first entry: restart inside the iteration
    (1500, 10, 2.5, 3.0, F64, 45),      # line search fails with col > 0: memory reset, restart at FG_LNSRCH
], ids=["f32-ascent", "f64-lnsrch-failure"])
def test_solve_graph_matches_solve_through_restarts(n, m, l_odd, x0, dtype, max_iter):
    """The two restart branches of test_restart_in_every_cta_of_a_launch, 8 identical copies and 2 perturbed ones, with
    the batched device objective.  The shapes there were chosen with the oracle's objective and do not restart with this
    one (test_restart_shapes_reset_with_the_batched_objective finds these with the oracle): solve's col history shows the
    memory reset, and solve_graph matches it."""
    X = []
    for k in range(10):
        x, l, u, nbd = H.rosenbrock_problem(n, dtype=dtype, l_odd=l_odd, x0=x0)
        if k >= 8:
            x = (x + 0.05 * (k - 7) * np.random.default_rng(k).uniform(-1.0, 1.0, n)).astype(dtype)
        X.append(x)
    X = np.stack(X)
    L, U, N = np.tile(l, (10, 1)), np.tile(u, (10, 1)), np.tile(nbd, (10, 1))
    cols = [[] for _ in range(10)]
    want, want_calls = run_solve(m, X, L, U, N, 0.0, 0.0, max_iter=max_iter, cols=cols)
    assert any(b < a and a > 0 for a, b in zip(cols[0], cols[0][1:])), ("no memory reset", cols[0])
    got, calls, _ = run_graph(m, X, L, U, N, 0.0, 0.0, max_iter=max_iter)
    assert_same(got, want)
    assert calls == want_calls


# ---------------------------------------------------------------------------------------------------------------------
# limits


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [F64, F32], ids=["f64", "f32"])
@pytest.mark.parametrize("max_iter,max_fg", [(7, 0), (0, 9), (6, 9), (9, 6)], ids=["iter", "fg", "both-iter-first", "both-fg-first"])
def test_limits(dtype, max_iter, max_fg):
    """max_iter alone against solve(max_iter=...); max_fg and both limits against host_solve (the iteration text wins
    when both are reached at the same NEW_X)."""
    X, L, U, N = make_batch(2049, dtype, MIX)
    want, want_calls = run_solve(5, X, L, U, N, 0.0, 0.0, max_iter=max_iter, max_fg=max_fg)
    got, calls, _ = run_graph(5, X, L, U, N, 0.0, 0.0, max_iter=max_iter, max_fg=max_fg)
    assert_same(got, want)
    assert calls == want_calls
    texts = {bytes(t).decode().rstrip() for t in want["task"]}
    assert STOP_ITER in texts or STOP_FG in texts, texts
    if max_fg and not max_iter:
        assert STOP_FG in texts and STOP_ITER not in texts, texts
    if max_iter and not max_fg:
        assert STOP_ITER in texts and STOP_FG not in texts, texts


# ---------------------------------------------------------------------------------------------------------------------
# launch cap, graph cache


@pytest.mark.gpu
def test_a_long_solve_takes_several_launches():
    X, L, U, N = make_batch(2049, F64, [("far", 0), ("walk", 0), ("ties", 1)])
    want, want_calls = run_solve(5, X, L, U, N, 0.0, 0.0, max_iter=200)
    got, calls, (builds, launches, total) = run_graph(5, X, L, U, N, 0.0, 0.0, max_iter=200)
    assert calls > CALL_CAP + 1, calls
    assert builds == 1 and launches >= 2 and launches == -(-(calls - 1) // CALL_CAP), (builds, launches, calls)
    assert_same(got, want)
    assert calls == want_calls


@pytest.mark.gpu
def test_graph_is_kept_until_an_argument_changes():
    import torch
    import lbfgsb_b200
    X, L, U, N = make_batch(2049, F64, MIX)
    P, n = X.shape
    xd, ld, ud, nd, fd, gd = _tensors(X, L, U, N)
    x0 = torch.from_numpy(X).cuda()
    b = lbfgsb_b200.BatchProblem(P, n, 10, F64)
    try:
        c1 = b.solve_graph(xd, ld, ud, nd, fd, gd, 1.0e7, 1.0e-5, max_iter=20)
        first = state_of(b, xd, fd, gd)
        assert b.graph_stats()[0] == 1
        xd.copy_(x0)
        c2 = b.solve_graph(xd, ld, ud, nd, fd, gd, 1.0e7, 1.0e-5, max_iter=20)
        assert b.graph_stats()[0] == 1 and c2 == c1
        assert_same(state_of(b, xd, fd, gd), first, "second solve: ")
        f2 = torch.zeros_like(fd)
        xd.copy_(x0)
        b.solve_graph(xd, ld, ud, nd, f2, gd, 1.0e7, 1.0e-5, max_iter=20)
        assert b.graph_stats()[0] == 2
        assert_same(state_of(b, xd, f2, gd), first, "new f buffer: ")
        xd.copy_(x0)
        b.solve_graph(xd, ld, ud, nd, f2, gd, 1.0e7, 1.0e-5, max_iter=21)
        assert b.graph_stats()[0] == 3
        xd.copy_(x0)
        b.solve_graph(xd, ld, ud, nd, f2, gd, 1.0e7, 1.0e-5, max_iter=21)
        assert b.graph_stats()[0] == 3
    finally:
        b.close()


# ---------------------------------------------------------------------------------------------------------------------
# stream order, caller views, failures, the handle afterwards


@pytest.mark.gpu
def test_solve_graph_waits_for_torchs_current_stream():
    """x0 is written on torch's current stream behind a ~50 ms sleep kernel: the result is bitwise that of a run whose
    inputs were synchronised first."""
    import torch
    import lbfgsb_b200
    X, L, U, N = make_batch(4097, F64, [("walk", 0), ("walk", 1), ("ties", 0), ("far", 0)])
    P, n = X.shape

    def run(sleep):
        xd, ld, ud, nd, fd, gd = _tensors(np.zeros_like(X), L, U, N)
        xs = torch.from_numpy(X).cuda()
        b = lbfgsb_b200.BatchProblem(P, n, 5, F64)
        torch.cuda.synchronize()
        try:
            if sleep:
                torch.cuda._sleep(100_000_000)     # ~50 ms at the B200's clock
            xd.copy_(xs)
            if not sleep:
                torch.cuda.synchronize()
            calls = b.solve_graph(xd, ld, ud, nd, fd, gd, 0.0, 0.0, max_iter=10)
            return state_of(b, xd, fd, gd), calls
        finally:
            b.close()
    want, wc = run(False)
    got, gc = run(True)
    assert_same(got, want)
    assert gc == wc


PAD = 4096     # bytes of poison in front of and behind every caller buffer


@pytest.mark.gpu
@pytest.mark.parametrize("n,dtype", [(2049, F64), (4097, F32)], ids=["f64", "f32"])
def test_solve_graph_reads_and_writes_nothing_outside_its_rows(n, dtype):
    import torch
    import lbfgsb_b200
    X, L, U, N = make_batch(n, dtype, MIX[:6])
    P = X.shape[0]
    want, want_calls = run_solve(6, X, L, U, N, 0.0, 0.0, max_iter=10)
    tdt = torch.float64 if dtype == F64 else torch.float32
    bufs, views = [], []
    for a in (X, L, U, N, np.zeros(P, dtype), np.zeros((P, n), dtype)):
        es = a.dtype.itemsize
        k0 = PAD // es
        buf = torch.full((2 * k0 + a.size,), 7 if a.dtype == np.int32 else float("nan"),
                         dtype=torch.int32 if a.dtype == np.int32 else tdt, device="cuda")
        v = buf[k0:k0 + a.size].view(a.shape)
        v.copy_(torch.from_numpy(a))
        bufs.append((buf, k0, a.size, buf.view(torch.int64 if es == 8 else torch.int32).clone()))
        views.append(v)
    assert views[0][1].data_ptr() % 16 != 0
    xd, ld, ud, nd, fd, gd = views
    b = lbfgsb_b200.BatchProblem(P, n, 6, dtype)
    try:
        calls = b.solve_graph(xd, ld, ud, nd, fd, gd, 0.0, 0.0, max_iter=10)
        got = state_of(b, xd, fd, gd)
    finally:
        b.close()
    assert_same(got, want)
    assert calls == want_calls
    for name, (buf, k0, size, before) in zip(("x", "l", "u", "nbd", "f", "g"), bufs):
        after = buf.view(before.dtype)
        for lo, hi, side in ((0, k0, "in front of"), (k0 + size, buf.numel(), "behind")):
            bad = torch.nonzero(after[lo:hi] != before[lo:hi])
            assert bad.numel() == 0, "%s: %d poisoned elements %s the rows were written" % (name, bad.numel(), side)


@pytest.mark.gpu
def test_a_failing_objective_stops_the_unfinished_problems_and_leaves_the_handle_usable():
    import lbfgsb_b200
    X, L, U, N = make_batch(65, F64, [("far", 0), ("walk", 0), ("err_lu", 0)])
    P, n = X.shape
    xd, ld, ud, nd, fd, gd = _tensors(X, L, U, N)
    b = lbfgsb_b200.BatchProblem(P, n, 5, F64)

    def bad(xp, gp, fp, mp, stream):
        raise RuntimeError("objective refuses")
    try:
        with pytest.raises(lbfgsb_b200.LbfgsbB200Error, match="returned 2.*callback"):
            b.solve_graph(xd, ld, ud, nd, fd, gd, 0.0, 0.0, fg_enqueue=bad, max_iter=10)
        assert b.task_str(0) == b.task_str(1) == "STOP: THE OBJECTIVE CALLBACK FAILED"
        assert b.task_str(2).startswith("ERROR: NO FEASIBLE SOLUTION"), b.task_str(2)
        assert b.counts() == (0, 0, P)
        assert b.graph_stats()[0] == 0
        # the handle still works: a solve from START equals one on a fresh batch
        for p in range(P):
            b.set_task(p, "START")
        xd, ld, ud, nd, fd, gd = _tensors(X, L, U, N)
        calls = b.solve(xd, ld, ud, nd, fd, gd, 0.0, 0.0, max_iter=10)
        got = state_of(b, xd, fd, gd)
    finally:
        b.close()
    want, want_calls = run_solve(5, X, L, U, N, 0.0, 0.0, max_iter=10)
    assert_same(got, want)
    assert calls == want_calls


@pytest.mark.gpu
def test_setulb_after_solve_graph_advances_no_problem():
    """Afterwards the handle is as solve leaves it: a further call finds no problem at FG or NEW_X (the limit-stopped
    ones count as ended by the caller's STOP), and changes no task."""
    import lbfgsb_b200
    X, L, U, N = make_batch(25, F64, MIX)
    P, n = X.shape
    for graph in (False, True):
        xd, ld, ud, nd, fd, gd = _tensors(X, L, U, N)
        b = lbfgsb_b200.BatchProblem(P, n, 5, F64)
        try:
            if graph:
                b.solve_graph(xd, ld, ud, nd, fd, gd, 1.0e7, 1.0e-5, max_iter=8)
            else:
                b.solve(xd, ld, ud, nd, fd, gd, 1.0e7, 1.0e-5, max_iter=8)
            before = b.task.copy()
            assert any(b.task_str(p) == STOP_ITER for p in range(P))
            b.setulb_dev(xd, ld, ud, nd, fd, gd, 1.0e7, 1.0e-5)
            assert b.counts() == (0, 0, P)
            assert np.array_equal(b.task, before)
        finally:
            b.close()


@pytest.mark.parametrize("n,m,l_odd,x0,dtype,max_iter", [(2049, 5, 1.0, 3.0, F32, 45), (1500, 10, 2.5, 3.0, F64, 45)],
                         ids=["f32-ascent", "f64-lnsrch-failure"])
def test_restart_shapes_reset_with_the_batched_objective(n, m, l_odd, x0, dtype, max_iter):
    """CPU, oracle alone in device-order mode, with the batched sample objective's own arithmetic (rosenbrock_terms and
    the fixed-shape sum of test_gpu_batch_lockstep): the restart shapes of the GPU test take their branch -- an ascent
    direction (REAL32) or a failed line search (REAL64) -- and reset their memory with col > 0."""
    from oracle import oracle_py as O
    from test_gpu_batch_lockstep import device_order_dot, rosenbrock_terms

    def fg(x, g):
        gr, terms = rosenbrock_terms(x)
        g[:] = gr
        return x.dtype.type(4) * device_order_dot(terms, np.ones(x.shape[0], x.dtype))
    x, l, u, nbd = H.rosenbrock_problem(n, dtype=dtype, l_odd=l_odd, x0=x0)
    O.set_sum_mode(1)
    O.set_tie_mode(0)
    try:
        O.event_counts()
        tr = H.run_driver(O.OracleSetulb(dtype), fg, n, m, x.copy(), l, u, nbd, 0.0, 0.0,
                          stop=H.iteration_budget_stop(max_iter))
        ev = O.event_counts()
    finally:
        O.set_sum_mode(0)
    cols = [r["col"] for r in tr[0]]
    assert ev[2] >= 1 and any(b < a for a, b in zip(cols, cols[1:])), (ev, cols)
    if dtype == F32:
        assert ev[1] >= 1, ev
    else:
        assert ev[1] == 0 and tr[1].startswith("ABNORMAL_TERMINATION_IN_LNSRCH"), (ev, tr[1])


@pytest.mark.parametrize("case", COVER, ids=lambda c: "n%d-m%d-%s" % (c[0], c[1], "f64" if c[2] == F64 else "f32"))
def test_cover_cases_converge_and_stop(case):
    """CPU, oracle alone in device-order mode with the batched objective's arithmetic (the batch computes the same bits):
    in every cover batch at least one problem of the mix converges before max_iter and at least one reaches it."""
    from oracle import oracle_py as O
    from test_gpu_batch_lockstep import device_order_dot, rosenbrock_terms

    def fg(x, g):
        gr, terms = rosenbrock_terms(x)
        g[:] = gr
        return x.dtype.type(4) * device_order_dot(terms, np.ones(x.shape[0], x.dtype))
    n, m, dtype, factr, pgtol, max_iter = case
    ends = []
    O.set_sum_mode(1)
    O.set_tie_mode(0)
    try:
        for fam, seed in MIX[:6]:
            x, l, u, nbd = FAM[fam](n, np.dtype(dtype), seed)
            tr = H.run_driver(O.OracleSetulb(dtype), fg, n, m, x.copy(), l, u, nbd, factr, pgtol,
                              stop=H.iteration_budget_stop(max_iter), want_hash=False)
            ends.append(tr[1].split(":")[0])
    finally:
        O.set_sum_mode(0)
    assert "CONVERGENCE" in ends and "STOP" in ends, ends


def test_cover_has_every_kind_and_pass_instance():
    mt = {(np.dtype(c[2]).name, 5 if c[1] <= 5 else (10 if c[1] <= 10 else 20)) for c in COVER}
    assert mt == {(k, t) for k in ("float64", "float32") for t in (5, 10, 20)}
    assert {1, 5, 10, 17, 20} <= {c[1] for c in COVER}
    assert {(c[0], np.dtype(c[2]).name) for c in COVER} >= {(65536, "float64"), (131072, "float32"), (25, "float64"),
                                                            (2049, "float64"), (4097, "float32")}
