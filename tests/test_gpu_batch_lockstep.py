"""Lock-step, bit-for-bit parity of the batched engine (batch.cuh, include/lbfgsb_b200.h section 6) with the oracle in
device-order mode, call by call, one oracle per problem.

One `lbfgsb_batch_setulb_dev_*` call advances every problem of the batch; then every problem whose task asked for work
(START, FG_*, NEW_X) gets exactly one `OracleSetulb` call on its own arrays, with `oracle_set_sum_mode(1)` and equal
breakpoints in hpsolb's heap order (tie mode 0).  f and g are evaluated on the host for both sides with the same routine
per problem and copied into the batch's [nprob, n] tensors.  After every call, for every problem that was advanced, task,
csave, lsave, the exported isave/dsave slots (not the clock slots dsave[5:10]), f and x must have identical bits; at
every NEW_X also iwhere, the S/Y ring columns in ring order from head, t, the previous gradient (the oracle's r) and d,
and the float64 checks of test_gpu_lockstep.LockStep.independent run on the batch's own vectors
(lbfgsb_batch_vector_copy).  A failure names the problem, its family, the call, the iteration, the task and the field,
and for a vector the first differing index and its tile (2048 REAL64, 4096 REAL32 variables).

The batched engine forms every O(n) sum in the engine's fixed shape with one tile per grid block, forms formk's
entering/leaving sums as masked full-range sums and pops the Cauchy breakpoints from hpsolb's heap (DESIGN.md section
15): so walking, tie, mixed-bound, skipping and restarting problems are all expected to match in every bit here.

Problems stop at their own iteration budget ('STOP: ITERATION BUDGET' on both sides), so one launch mixes idle, FG and
NEW_X problems, and different families in one batch take different paths in the same launch.  The CPU tests at the end
check with the oracle alone that every case still takes the branches it is listed for."""
import ctypes as C

import numpy as np
import pytest

import harness as H
from oracle import oracle_py as O
from test_gpu_lockstep import LockStep, Mismatch, _bits, _Side, far_box, pinned, pinned_fg, unbounded
from test_gpu_edge import _nonconvex, sweep_problem

F64, F32 = np.float64, np.float32
TILE = {np.dtype(F64): 2048, np.dtype(F32): 4096}
N_MAX = {np.dtype(F64): 65536, np.dtype(F32): 131072}      # one CTA per problem: 32 tiles


def mt_of(m):
    return 5 if m <= 5 else (10 if m <= 10 else 20)


# ---------------------------------------------------------------------------------------------------------------------
# families: (n, dtype, seed) -> Problem.  make_fg() gives a fresh objective (the wrong-gradient family counts its
# evaluations), so each side of the lock step gets its own.


class Problem:
    def __init__(self, family, x, l, u, nbd, make_fg, dtype):
        self.family = family
        self.x, self.l, self.u = (np.ascontiguousarray(a, dtype=dtype) for a in (x, l, u))
        self.nbd = np.ascontiguousarray(nbd, dtype=np.int32)
        self.make_fg = make_fg


def _rosen(n, dtype):
    return lambda: O.rosenbrock_fg


def fam_far(n, dtype, seed):
    """far box: the sample objective, a box that is never reached (ring wraps, no walk)"""
    x, l, u, nbd = far_box(n, dtype)
    return Problem("far", x, l, u, nbd, _rosen(n, dtype), dtype)


def fam_pinned(n, dtype, seed):
    """40 % of the variables pinned on a bound for good (constant active set), coupled quartic"""
    x, l, u, nbd = pinned(n, dtype)
    return Problem("pinned", x, l, u, nbd, lambda: pinned_fg(n, dtype), dtype)


def fam_nbd0(n, dtype, seed):
    """nbd = 0 everywhere: the cauchy_mode = 1 branch once the history holds a pair"""
    x, l, u, nbd = unbounded(n, dtype)
    return Problem("nbd0", x, l, u, nbd, _rosen(n, dtype), dtype)


def fam_walk(n, dtype, seed):
    """bound-heavy Rosenbrock (l_odd 1.1 or 1.5), perturbed start: breakpoint walks, entering/leaving variables"""
    rng = np.random.default_rng(seed)
    x, l, u, nbd = H.rosenbrock_problem(n, dtype=dtype, l_odd=(1.1, 1.5)[seed % 2])
    x = (x + 0.25 * rng.uniform(-1.0, 1.0, n)).astype(dtype)
    return Problem("walk", x, l, u, nbd, _rosen(n, dtype), dtype)


def fam_ties(n, dtype, seed):
    """equal breakpoints (l_odd 2.0 / 2.5 with x0 3 / 5): the Cauchy search ends inside a tied group, then subsm's
    backtrack"""
    l_odd, x0 = ((2.0, 3.0), (2.5, 5.0))[seed % 2]
    x, l, u, nbd = H.rosenbrock_problem(n, dtype=dtype, l_odd=l_odd, x0=x0)
    return Problem("ties", x, l, u, nbd, _rosen(n, dtype), dtype)


def fam_mixed(n, dtype, seed):
    """nbd 0-3, 3 % fixed variables (l = u, iwhere 3), a coupled quartic (test_gpu_edge.sweep_problem)"""
    _, _, fg, mk = sweep_problem(seed, n=n)
    x, l, u, nbd = mk()
    return Problem("mixed", x, l, u, nbd, lambda: fg, dtype)


def fam_nonconvex(n, dtype, seed):
    """a concave share (test_gpu_edge._nonconvex): skipped updates with col > 0, line-search backtracks"""
    share, a_c = ((0.5, 0.3), (0.3, 1.0), (0.1, 2.0))[seed % 3]
    fg, mk = _nonconvex(n, seed, share, a_c)
    x, l, u, nbd = mk()
    return Problem("nonconvex", x, l, u, nbd, lambda: fg, dtype)


def fam_badgrad(n, dtype, seed):
    """driver1's Rosenbrock whose gradient is negated after the seed-th evaluation: the line search fails with col > 0,
    the memory is reset and the iteration restarts at FG_LNSRCH (REAL64: the second failure, at col = 0, ends the run
    with ABNORMAL_TERMINATION_IN_LNSRCH)"""
    x, l, u, nbd = H.rosenbrock_problem(n, dtype=dtype)

    def make():
        count = [0]

        def fg(x, g):
            f = O.rosenbrock_fg(x, g)
            count[0] += 1
            if count[0] > seed:
                np.negative(g, out=g)
            return f
        return fg
    return Problem("badgrad", x, l, u, nbd, make, dtype)


FAMILIES = {"far": fam_far, "pinned": fam_pinned, "nbd0": fam_nbd0, "walk": fam_walk, "ties": fam_ties,
            "mixed": fam_mixed, "nonconvex": fam_nonconvex, "badgrad": fam_badgrad}
# what each family is in the table for (checked with the oracle by the CPU tests below)
ROLE = {"far": "ring", "pinned": "ring", "nbd0": "ring", "walk": "walk", "ties": "tie", "mixed": "walk",
        "nonconvex": "skip", "badgrad": "restart"}

# (n, m, real kind, [(family, seed, iteration budget), ...]).  One batch per row; every row mixes families.
# Ring budgets are at least m + 3 (the S/Y ring wraps); the wrong-gradient seed is the evaluation after which g is
# negated, chosen (with the oracle) so that the line search fails with col > 0 at that shape.
BATCHES = [
    (65, 5, F64, [("far", 0, 8), ("walk", 1, 12), ("mixed", 21, 10), ("nonconvex", 1, 14), ("badgrad", 15, 40)]),
    (2047, 11, F64, [("far", 0, 14), ("walk", 0, 12), ("ties", 0, 10), ("mixed", 22, 10), ("badgrad", 15, 40)]),
    (2048, 10, F64, [("pinned", 0, 13), ("walk", 1, 12), ("ties", 1, 10), ("nonconvex", 1, 14), ("badgrad", 10, 40)]),
    (2049, 10, F64, [("nbd0", 0, 13), ("walk", 0, 12), ("mixed", 23, 10), ("badgrad", 15, 40), ("badgrad", 5, 40)]),
    (4097, 6, F64, [("far", 0, 9), ("walk", 1, 12), ("ties", 0, 10), ("nonconvex", 2, 14), ("badgrad", 15, 40)]),
    (65535, 1, F64, [("pinned", 0, 5), ("walk", 0, 10), ("mixed", 24, 8), ("badgrad", 15, 40)]),
    (65536, 17, F64, [("far", 0, 20), ("walk", 1, 10), ("ties", 1, 8), ("badgrad", 15, 40)]),
    (65, 20, F32, [("far", 0, 23), ("walk", 0, 12), ("mixed", 25, 10), ("nonconvex", 1, 14)]),
    (4095, 5, F32, [("pinned", 0, 8), ("walk", 1, 12), ("ties", 0, 10), ("nonconvex", 0, 14), ("badgrad", 15, 40)]),
    (4096, 6, F32, [("far", 0, 9), ("walk", 0, 12), ("mixed", 26, 10), ("badgrad", 7, 40)]),
    (4097, 17, F32, [("nbd0", 0, 20), ("walk", 1, 12), ("ties", 1, 10), ("nonconvex", 1, 14), ("badgrad", 15, 40)]),
    (131071, 10, F32, [("far", 0, 13), ("walk", 0, 10), ("mixed", 27, 8), ("badgrad", 10, 40)]),
    (131072, 1, F32, [("pinned", 0, 5), ("walk", 1, 10), ("ties", 0, 8), ("badgrad", 12, 40)]),
]


def _batch_id(b):
    return "n%d-m%d-%s" % (b[0], b[1], "f64" if b[2] == F64 else "f32")


# ---------------------------------------------------------------------------------------------------------------------
# the lock-step harness


class _BatchSide:
    """One problem of the batch, seen through the attributes LockStep.scalars / independent read."""

    def __init__(self, b, p, x, g, f):
        self.task, self.csave, self.lsave, self.isave, self.dsave = b.task[p], b.csave[p], b.lsave[p], b.isave[p], b.dsave[p]
        self.x, self.g, self.f = x, g, f


class BatchLockStep(LockStep):
    """LockStep's per-call and float64 checks for one problem of a batch (exact class: every bit)."""

    def __init__(self, n, m, dtype, prob, index):
        super().__init__(n, m, dtype, prob.l, prob.u, prob.nbd, True, "problem %d (%s)" % (index, prob.family))

    def vec(self, ctx, field, a, b, tol=None):
        bad = np.nonzero(_bits(a) != _bits(b))[0]
        if bad.size:
            i = int(bad[0])
            self.fail(ctx, field, "%d of %d elements differ; first at index %d (tile %d): batch %r, oracle %r" % (
                bad.size, a.size, i, i // TILE[self.dtype], a[i], b[i]))

    def at_newx(self, ctx, b, p, iw, e, o):
        n, m = self.n, self.m
        self.vec(ctx, "iwhere", iw, o.iwa[n:2 * n])
        d = b.vector(p, 2).cpu().numpy()
        gold = b.vector(p, 8).cpu().numpy()
        col, head, itail = int(e.isave[27]), int(e.isave[26]), int(e.isave[28])
        ws = wy = None
        if col > 0:
            ws = b.vector(p, 5, m * self.ldw).cpu().numpy()
            wy = b.vector(p, 6, m * self.ldw).cpu().numpy()
        mn = m * n
        for k in range(col):
            j = (head - 1 + k) % m
            self.vec(ctx, "ws column %d (ring position %d of %d)" % (j, k, col), ws[j * self.ldw:j * self.ldw + n],
                     o.wa[j * n:(j + 1) * n])
            self.vec(ctx, "wy column %d (ring position %d of %d)" % (j, k, col), wy[j * self.ldw:j * self.ldw + n],
                     o.wa[mn + j * n:mn + (j + 1) * n])
        z0 = 2 * mn + 11 * m * m            # oracle wa: ws, wy, sy, ss, wt, wn, snd, then z, r, d, t, xp
        self.vec(ctx, "t (previous x)", b.vector(p, 3).cpu().numpy(), o.wa[z0 + 3 * n:z0 + 4 * n])
        self.vec(ctx, "previous gradient (oracle r)", gold, o.wa[z0 + n:z0 + 2 * n])
        self.vec(ctx, "d (lnsrlb direction)", d, o.wa[z0 + 2 * n:z0 + 3 * n])
        self.independent(ctx, e, d, gold, ws, wy, col, itail)
        self.prev = (e.g.copy(), gold, d, e.dsave[13], int(e.isave[30]))


class BatchRun:
    """Result of batch_lockstep: per problem the NEW_X rows (iter, col, nseg, nenter, nleave, iback, nskip), the final
    task, the oracle's event counts (O.event_counts order) and the harnesses."""

    def __init__(self, probs):
        self.rows = [[] for _ in probs]
        self.cols = [[] for _ in probs]      # (call, iteration, col) after every call that advanced the problem
        self.tasks = [None] * len(probs)
        self.events = [[0] * 8 for _ in probs]
        self.checks = []
        self.calls = 0


def batch_lockstep(n, m, dtype, probs, budgets, factr=0.0, pgtol=0.0):
    import torch
    import lbfgsb_b200
    dtype = np.dtype(dtype)
    P = len(probs)
    tdt = torch.float64 if dtype == F64 else torch.float32
    xd, ld, ud = (torch.from_numpy(np.stack([getattr(p, k) for p in probs])).cuda() for k in ("x", "l", "u"))
    nd = torch.from_numpy(np.stack([p.nbd for p in probs])).cuda()
    gd = torch.zeros((P, n), dtype=tdt, device="cuda")
    fd = torch.zeros(P, dtype=tdt, device="cuda")
    b = lbfgsb_b200.BatchProblem(P, n, m, dtype)
    sides = [_Side(O.OracleSetulb(dtype), n, m, p.x.copy(), dtype) for p in probs]
    efg = [p.make_fg() for p in probs]
    ofg = [p.make_fg() for p in probs]
    run = BatchRun(probs)
    run.checks = [BatchLockStep(n, m, dtype, p, k) for k, p in enumerate(probs)]
    O.set_sum_mode(1)
    O.set_tie_mode(0)
    try:
        for call in range(1, 20 * max(budgets) + 100):
            pre = [b.task_str(p) for p in range(P)]
            active = [t == "START" or t[:2] == "FG" or t[:5] == "NEW_X" for t in pre]
            if not any(active):
                break
            b.setulb_dev(xd, ld, ud, nd, fd, gd, factr, pgtol)
            run.calls = call
            xh, gh, fh = xd.cpu().numpy(), gd.cpu().numpy(), fd.cpu().numpy()
            iw = b.iwhere() if (b.task[:, 0] == ord("N")).any() else None
            for p in np.nonzero(active)[0]:
                o, ls = sides[p], run.checks[p]
                before = O.event_counts(reset=False)
                o.call(n, m, probs[p].l, probs[p].u, probs[p].nbd, factr, pgtol)
                run.events[p] = [a + (c - q) for a, c, q in zip(run.events[p], O.event_counts(reset=False), before)]
                e = _BatchSide(b, p, xh[p], gh[p], fh[p:p + 1])
                ctx = "call %d (iteration %d, task %r)" % (call, int(o.isave[29]), H.task_str(o.task))
                try:
                    ls.scalars(ctx, e, o)
                except Mismatch:
                    raise Mismatch(_report(run))
                run.cols[p].append((call, int(b.isave[p, 29]), int(b.isave[p, 27])))
                t = b.task_str(p)
                if t[:2] == "FG":
                    fh[p] = efg[p](xh[p], gh[p])
                    o.f[0] = ofg[p](o.x, o.g)
                elif t[:5] == "NEW_X":
                    ls.at_newx(ctx, b, p, iw[p], e, o)
                    i = b.isave[p]
                    run.rows[p].append((int(i[29]), int(i[27]), int(i[32]), int(i[40]), n + 1 - int(i[39]), int(i[24]), int(i[25])))
                    if i[29] >= budgets[p]:
                        b.set_task(int(p), "STOP: ITERATION BUDGET")
                        o.task[:] = H.make_task("STOP: ITERATION BUDGET")
                else:
                    run.tasks[p] = t
            gd.copy_(torch.from_numpy(gh))
            fd.copy_(torch.from_numpy(fh))
    finally:
        O.set_sum_mode(0)
        b.close()
    for p in range(P):
        run.tasks[p] = run.tasks[p] or b.task_str(p)
    if any(ls.errors for ls in run.checks):
        raise Mismatch(_report(run))
    return run


def _report(run):
    bad = [ls for ls in run.checks if ls.errors]
    return "%d problem(s) differ:\n" % len(bad) + "\n".join(
        "%s: %s" % (ls.label, "\n    ".join(e[1] for e in ls.errors[:6])) for ls in bad)


def _build(n, dtype, spec):
    return [FAMILIES[f](n, dtype, s) for f, s, _ in spec], [bud for _, _, bud in spec]


def _col_drop(cols):
    """(call, iteration) of the first return at which col fell back (the memory was reset), or None"""
    return next(((b[0], b[1]) for a, b in zip(cols, cols[1:]) if b[2] < a[2]), None)


@pytest.mark.gpu
@pytest.mark.parametrize("batch", BATCHES, ids=_batch_id)
def test_batch_lockstep_bit_exact(batch):
    n, m, dtype, spec = batch
    probs, budgets = _build(n, dtype, spec)
    run = batch_lockstep(n, m, dtype, probs, budgets)
    for p, (fam, _, bud) in enumerate(spec):
        rows, ev = run.rows[p], run.events[p]
        where = "problem %d (%s): %s" % (p, fam, run.tasks[p])
        if ROLE[fam] == "ring":
            assert len(rows) == bud and rows[-1][1] == min(m, bud), where
        elif ROLE[fam] == "walk" or ROLE[fam] == "tie":
            assert any(r[2] > 1 or r[3] or r[4] for r in rows), where
        elif fam == "nonconvex":
            assert ev[3] >= 1 and any(r[5] > 0 for r in rows), (where, ev)
        elif fam == "badgrad":
            assert ev[2] >= 1 and _col_drop(run.cols[p]) is not None, (where, ev)
            if dtype == F64:
                assert run.tasks[p].startswith("ABNORMAL_TERMINATION_IN_LNSRCH"), where


# ---------------------------------------------------------------------------------------------------------------------
# restart stress: every CTA of the launch restarts in the same call


@pytest.mark.gpu
@pytest.mark.parametrize("n,m,l_odd,x0,dtype,budget,event", [
    (1500, 5, 1.0, 3.0, F32, 45, 1),      # gd >= 0 at lnsrlb's first entry (iteration 34): restart inside body()
    (1000, 10, 2.5, 3.0, F64, 45, 2),     # line search fails with col > 0: reset and restart at FG_LNSRCH
], ids=["f32-ascent", "f64-lnsrch-failure"])
def test_restart_in_every_cta_of_a_launch(n, m, l_odd, x0, dtype, budget, event):
    copies, perturbed = 128, 4
    probs = []
    for k in range(copies + perturbed):
        x, l, u, nbd = H.rosenbrock_problem(n, dtype=dtype, l_odd=l_odd, x0=x0)
        if k >= copies:
            x = (x + 0.05 * (k - copies + 1) * np.random.default_rng(k).uniform(-1.0, 1.0, n)).astype(dtype)
        probs.append(Problem("stress", x, l, u, nbd, _rosen(n, dtype), dtype))
    run = batch_lockstep(n, m, dtype, probs, [budget] * len(probs))
    # every copy took the branch: the oracle of each reset its memory, and col fell back at the same call and
    # iteration on both sides (the per-call isave comparison of the lock step holds col equal)
    assert run.events[0][2] >= 1 and run.events[0][event] >= 1, run.events[0]
    drop = _col_drop(run.cols[0])
    assert drop is not None
    for p in range(copies):
        assert run.events[p] == run.events[0] and _col_drop(run.cols[p]) == drop and run.tasks[p] == run.tasks[0], p


# ---------------------------------------------------------------------------------------------------------------------
# the batched sample objective against its formula


def rosenbrock_terms(x):
    """g of k_rosenbrock_batch (engine.cu) in the real kind of x, operation by operation, and the summands of f/4."""
    dt = x.dtype.type
    n = x.shape[0]
    xp = np.concatenate([np.zeros(1, x.dtype), x[:-1]])
    xn = np.concatenate([x[1:], np.zeros(1, x.dtype)])
    t2 = x - xp * xp
    t1 = xn - x * x
    g = dt(8) * t2 - dt(16) * x * t1
    if n > 1:
        g[n - 1] = dt(8) * t2[n - 1]
    g[0] = dt(2) * (x[0] - dt(1)) - dt(16) * x[0] * t1[0]
    terms = t2 * t2
    terms[0] = dt(0.25) * (x[0] - dt(1)) * (x[0] - dt(1))
    return g, terms


def device_order_dot(a, b):
    if a.dtype == F64:
        fn = O.lib().oracle_device_order_dot_f64
        fn.restype = C.c_double
    else:
        fn = O.lib().oracle_device_order_dot_f32
        fn.restype = C.c_float
    return a.dtype.type(fn(C.c_int64(a.shape[0]), a.ctypes.data_as(C.c_void_p), b.ctypes.data_as(C.c_void_p)))


@pytest.mark.gpu
@pytest.mark.parametrize("n,dtype", [(1, F64), (2, F64), (65, F64), (2049, F64), (65536, F64), (4097, F32), (131072, F32)])
def test_batched_rosenbrock_objective_matches_its_formula(n, dtype):
    import torch
    import lbfgsb_b200
    P = 5
    rng = np.random.default_rng(n)
    x = rng.uniform(-2.0, 2.0, (P, n)).astype(dtype)
    mask = np.array([1, 0, 1, 0, 1], np.int32)
    tdt = torch.float64 if dtype == F64 else torch.float32
    xd = torch.from_numpy(x).cuda()
    gd = torch.full((P, n), float("nan"), dtype=tdt, device="cuda")
    fd = torch.full((P,), float("nan"), dtype=tdt, device="cuda")
    gd[1].fill_(-7.5)
    fd[3] = 1.25
    g_before, f_before = gd.clone(), fd.clone()
    md = torch.from_numpy(mask).cuda()
    fn = getattr(lbfgsb_b200.lib(), "lbfgsb_problem_rosenbrock_batch_" + ("f64" if dtype == F64 else "f32"))
    torch.cuda.synchronize()
    assert fn(P, C.c_int64(n), C.c_void_p(xd.data_ptr()), C.c_void_p(gd.data_ptr()), C.c_void_p(fd.data_ptr()),
              C.c_void_p(md.data_ptr()), None) == 0
    torch.cuda.synchronize()
    g, f = gd.cpu().numpy(), fd.cpu().numpy()
    assert torch.equal(xd.cpu(), torch.from_numpy(x))
    for p in range(P):
        if not mask[p]:
            assert np.array_equal(_bits(g[p]), _bits(g_before[p].cpu().numpy())), p
            assert _bits(f[p:p + 1])[0] == _bits(f_before[p:p + 1].cpu().numpy())[0], p
            continue
        gr, terms = rosenbrock_terms(x[p])
        bad = np.nonzero(_bits(g[p]) != _bits(gr))[0]
        assert bad.size == 0, (p, int(bad[0]), g[p][bad[0]], gr[bad[0]])
        fr = x.dtype.type(4) * device_order_dot(terms, np.ones(n, dtype))
        assert _bits(f[p:p + 1])[0] == _bits(np.array([fr], dtype))[0], (p, f[p], fr)


# ---------------------------------------------------------------------------------------------------------------------
# small invariants of the batch


def _trace(nprob, n, m, dtype, x0, l, u, nbd, budget, views=None):
    """Per problem and NEW_X: isave (not the handle slots 16-19), dsave bits (not the clock slots 5-9), f bits; and the
    final x.  The batch's own objective; views = (x, l, u, nbd, f, g) caller tensors, else exact-size ones."""
    import torch
    import lbfgsb_b200
    tdt = torch.float64 if np.dtype(dtype) == F64 else torch.float32
    if views is None:
        xd, ld, ud, nd = (torch.from_numpy(np.ascontiguousarray(a)).cuda() for a in (x0, l, u, nbd))
        fd, gd = torch.zeros(nprob, dtype=tdt, device="cuda"), torch.zeros((nprob, n), dtype=tdt, device="cuda")
    else:
        xd, ld, ud, nd, fd, gd = views
    b = lbfgsb_b200.BatchProblem(nprob, n, m, dtype)
    rows = [[] for _ in range(nprob)]

    def on_newx(bp):
        fh = fd.cpu().numpy()
        for p in np.nonzero(bp.task[:, 0] == ord("N"))[0]:
            isv = np.concatenate([bp.isave[p, :16], bp.isave[p, 20:]])
            dsv = np.concatenate([bp.dsave[p, :5], bp.dsave[p, 10:]])
            rows[p].append((isv.copy(), _bits(dsv).copy(), _bits(fh[p:p + 1]).copy()))
    try:
        b.solve(xd, ld, ud, nd, fd, gd, 0.0, 0.0, max_iter=budget, on_newx=on_newx)
        tasks = [b.task_str(p) for p in range(nprob)]
    finally:
        b.close()
    return rows, tasks, xd.cpu().numpy()


def _same(a, b):
    return len(a) == len(b) and all(np.array_equal(p[0], q[0]) and np.array_equal(p[1], q[1]) and np.array_equal(p[2], q[2])
                                    for p, q in zip(a, b))


def _bound_heavy_batch(nprob, n, dtype, seed):
    rng = np.random.default_rng(seed)
    x, l, u, nbd = H.rosenbrock_problem(n, dtype=dtype, l_odd=1.1)
    X = (x + 0.25 * rng.uniform(-1.0, 1.0, (nprob, n))).astype(dtype)
    return X, np.tile(l, (nprob, 1)), np.tile(u, (nprob, 1)), np.tile(nbd, (nprob, 1))


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [F64, F32], ids=["f64", "f32"])
def test_problem_trace_does_not_depend_on_its_batch(dtype):
    """A problem alone gives the same bits as at index 0 and at the last index of a 64-problem batch; reversing the
    order of the problems changes no problem's trace."""
    P, n, m, budget = 64, 2049, 10, 12
    X, L, U, N = _bound_heavy_batch(P, n, dtype, 5)
    many, tasks, xm = _trace(P, n, m, dtype, X, L, U, N, budget)
    rev, tasks_r, xr = _trace(P, n, m, dtype, X[::-1], L[::-1], U[::-1], N[::-1], budget)
    assert all(len(r) == budget for r in many)
    for p in range(P):
        assert _same(many[p], rev[P - 1 - p]) and tasks[p] == tasks_r[P - 1 - p], p
        assert np.array_equal(_bits(xm[p]), _bits(xr[P - 1 - p])), p
    for p in (0, P - 1):
        one, t1, x1 = _trace(1, n, m, dtype, X[p:p + 1], L[p:p + 1], U[p:p + 1], N[p:p + 1], budget)
        assert _same(one[0], many[p]) and t1[0] == tasks[p] and np.array_equal(_bits(x1[0]), _bits(xm[p])), p


PAD = 4096     # bytes of poison in front of and behind every caller buffer


@pytest.mark.gpu
@pytest.mark.parametrize("n,dtype", [(2049, F64), (4097, F32)], ids=["f64", "f32"])
def test_batch_reads_and_writes_nothing_outside_its_rows(n, dtype):
    """[nprob, n] caller tensors as views of larger buffers with 4 KB of poison on each side (NaN for the reals, 7 for
    nbd), odd n so that rows are not 16-byte aligned: the trace is bit for bit that of a run on exact-size tensors and
    the poison is byte for byte unchanged."""
    import torch
    P, m, budget = 5, 6, 10
    X, L, U, N = _bound_heavy_batch(P, n, dtype, 9)
    want, want_t, want_x = _trace(P, n, m, dtype, X, L, U, N, budget)
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
    got, got_t, got_x = _trace(P, n, m, dtype, X, L, U, N, budget, views=views)
    assert got_t == want_t
    for p in range(P):
        assert _same(got[p], want[p]), p
    assert np.array_equal(_bits(got_x), _bits(want_x))
    for name, (buf, k0, size, before) in zip(("x", "l", "u", "nbd", "f", "g"), bufs):
        after = buf.view(before.dtype)
        for lo, hi, side in ((0, k0, "in front of"), (k0 + size, buf.numel(), "behind")):
            bad = torch.nonzero(after[lo:hi] != before[lo:hi])
            assert bad.numel() == 0, "%s: %d poisoned elements %s the rows were written" % (name, bad.numel(), side)


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [F64, F32], ids=["f64", "f32"])
def test_batch_vector_copy_refuses_out_of_range_requests(dtype):
    import torch
    import lbfgsb_b200
    P, n, m = 3, 1000, 5
    ldw, es = 1024, np.dtype(dtype).itemsize
    b = lbfgsb_b200.BatchProblem(P, n, m, dtype)
    dst = torch.zeros(m * ldw * es + 256, dtype=torch.uint8, device="cuda")
    copy = lbfgsb_b200.lib().lbfgsb_batch_vector_copy
    try:
        for which, cap in ((2, ldw * es), (3, ldw * es), (5, m * ldw * es), (6, m * ldw * es), (7, ldw * 4), (8, ldw * es)):
            for p in (0, P - 1):
                assert copy(C.c_void_p(b.h), p, which, C.c_void_p(dst.data_ptr()), C.c_int64(cap)) == 0, (which, p)
                assert copy(C.c_void_p(b.h), p, which, C.c_void_p(dst.data_ptr()), C.c_int64(cap + 1)) == 1, (which, p)
            for p in (-1, P):
                assert copy(C.c_void_p(b.h), p, which, C.c_void_p(dst.data_ptr()), C.c_int64(es)) == 1, (which, p)
        with pytest.raises(lbfgsb_b200.LbfgsbB200Error, match="out of range"):
            b.vector(P, 2)
        assert b.vector(P - 1, 5, count=m * ldw).numel() == m * ldw
    finally:
        b.close()


@pytest.mark.gpu
def test_batch_waits_for_an_objective_on_torchs_current_stream():
    """A torch objective on torch's current stream, held back ~50 ms by a sleep kernel before it writes f and g: the
    batch's trace is bitwise that of the same objective followed by a host synchronisation."""
    import torch
    P, n, m, budget = 4, 4097, 5, 8
    X, L, U, N = _bound_heavy_batch(P, n, F64, 13)

    def run(sleep):
        xd, ld, ud, nd = (torch.from_numpy(np.ascontiguousarray(a)).cuda() for a in (X, L, U, N))
        gd = torch.zeros((P, n), dtype=torch.float64, device="cuda")
        fd = torch.zeros(P, dtype=torch.float64, device="cuda")
        import lbfgsb_b200
        b = lbfgsb_b200.BatchProblem(P, n, m, F64)
        rows = []

        def fg(x, g, f):
            if sleep:
                torch.cuda._sleep(100_000_000)     # ~50 ms at the B200's clock
            t2 = x[:, 1:] - x[:, :-1] * x[:, :-1]
            g.copy_(torch.cat([2.0 * (x[:, :1] - 1.0), torch.zeros_like(x[:, 1:])], 1))
            g[:, 1:] += 8.0 * t2
            g[:, :-1] -= 16.0 * x[:, :-1] * t2
            f.copy_(4.0 * (0.25 * (x[:, 0] - 1.0) ** 2 + (t2 * t2).sum(1)))
            if not sleep:
                torch.cuda.synchronize()

        def on_newx(bp):
            rows.append((bp.isave.copy(), _bits(bp.dsave[:, 10:]).copy(), _bits(fd.cpu().numpy()).copy()))
        try:
            b.solve(xd, ld, ud, nd, fd, gd, 0.0, 0.0, fg=fg, max_iter=budget, on_newx=on_newx)
        finally:
            b.close()
        return rows, xd.cpu().numpy()
    want, want_x = run(False)
    got, got_x = run(True)
    assert len(want) == budget
    assert len(got) == len(want) and all(
        np.array_equal(a[0][:, 20:], b[0][:, 20:]) and np.array_equal(a[1], b[1]) and np.array_equal(a[2], b[2])
        for a, b in zip(got, want)), "the batch read f and g before the objective on torch's stream wrote them"
    assert np.array_equal(_bits(got_x), _bits(want_x))


# ---------------------------------------------------------------------------------------------------------------------
# CPU: creation limits, and the case table still covers what it claims (oracle only)


@pytest.mark.parametrize("nprob,n,m,kind,msg", [
    (4, 65537, 5, 8, "exceeds the one-CTA-per-problem limit of 65536"),
    (4, 131073, 5, 4, "exceeds the one-CTA-per-problem limit of 131072"),
    (4, 1000, 0, 8, "0 < m <= 20"),
    (4, 1000, 21, 8, "0 < m <= 20"),
    (0, 1000, 5, 8, "nprob > 0"),
])
def test_batch_create_refuses_what_it_cannot_hold(nprob, n, m, kind, msg):
    import lbfgsb_b200
    h = lbfgsb_b200.lib().lbfgsb_batch_create(nprob, n, m, kind, None)
    assert not h
    assert msg in lbfgsb_b200.last_error(), lbfgsb_b200.last_error()


def test_every_kind_and_instance_has_a_walking_and_a_restarting_problem():
    have = {(np.dtype(b[2]).name, mt_of(b[1]), ROLE[f]) for b in BATCHES for f, _, _ in b[3]}
    for d in (F64, F32):
        for t in (5, 10, 20):
            for role in ("walk", "restart"):
                assert (np.dtype(d).name, t, role) in have, (np.dtype(d).name, t, role)
    shapes = {(np.dtype(b[2]).name, b[0]) for b in BATCHES}
    for n in (65, 2047, 2048, 2049, 4097, 65535, 65536):
        assert ("float64", n) in shapes, n
    for n in (65, 4095, 4096, 4097, 131071, 131072):
        assert ("float32", n) in shapes, n
    assert {1, 5, 6, 10, 11, 17, 20} <= {b[1] for b in BATCHES}
    assert all(b[0] >= 65 and b[0] <= N_MAX[np.dtype(b[2])] for b in BATCHES)


def _oracle_alone(n, m, dtype, fam, seed, budget, tie_mode=0):
    prob = FAMILIES[fam](n, dtype, seed)
    O.set_sum_mode(1)
    O.set_tie_mode(tie_mode)
    try:
        O.event_counts()
        tr = H.run_driver(O.OracleSetulb(dtype), prob.make_fg(), n, m, prob.x.copy(), prob.l, prob.u, prob.nbd, 0.0, 0.0,
                          stop=H.iteration_budget_stop(budget), want_hash=(ROLE[fam] == "tie"))
        return tr, O.event_counts()
    finally:
        O.set_sum_mode(0)
        O.set_tie_mode(0)


CASES = [(b[0], b[1], b[2], f, s, bud) for b in BATCHES for f, s, bud in b[3]]
CASES = sorted(set(CASES), key=CASES.index)


def _case_id(c):
    return "%s-n%d-m%d-%s-s%d" % (c[3], c[0], c[1], "f64" if c[2] == F64 else "f32", c[4])


@pytest.mark.parametrize("case", CASES, ids=_case_id)
def test_case_takes_its_branch(case):
    n, m, dtype, fam, seed, budget = case
    tr, ev = _oracle_alone(n, m, dtype, fam, seed, budget)
    rows, task = tr[0], tr[1]
    role = ROLE[fam]
    if role == "ring":
        assert budget >= m + 3 and len(rows) == budget and rows[-1]["col"] == min(m, budget - 1), (len(rows), task)
        assert all(r["nenter"] == 0 and r["nleave"] == 0 for r in rows)
    elif role in ("walk", "tie"):
        assert any(r["nseg"] > 1 or r["nenter"] or r["nleave"] for r in rows), "no iterate walked or changed the free set"
        if fam == "mixed":
            prob = FAMILIES[fam](n, dtype, seed)
            assert (prob.nbd == 0).any() and (prob.nbd == 1).any() and (prob.nbd == 3).any() and (prob.l == prob.u).any()
    if role == "tie":
        other, _ = _oracle_alone(n, m, dtype, fam, seed, budget, tie_mode=1)
        assert any(a["hash"] != b["hash"] for a, b in zip(rows, other[0])), "the tie order makes no difference here"
    if fam == "nonconvex":
        assert ev[3] >= 1 and any(r["iback"] > 0 for r in rows), ev
        assert any(b["nskip"] > a["nskip"] and a["col"] > 0 for a, b in zip(rows, rows[1:])), "no skip with col > 0"
    if role == "restart":
        assert ev[2] >= 1, ("no memory reset", ev)
        if dtype == F64:
            assert task.startswith("ABNORMAL_TERMINATION_IN_LNSRCH"), task
