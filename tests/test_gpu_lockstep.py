"""Lock-step parity of the CUDA engine with the oracle in device-order mode, call by call.

The host twin (`lbfgsb_b200.HostSetulb`) and the oracle (`OracleSetulb`, `oracle_set_sum_mode(1)`) are driven in one
loop.  Each side evaluates f and g at its own x with the same host routine.  After every return (FG_START, every
FG_LNSRCH trial point, NEW_X, the final task) the task and csave strings, lsave, the isave/dsave slots the engine
exports (`export_state_of` in engine.cu; not the handle slots isave[16:19] and not the clock slots dsave[5:10]) and x
are compared; at every NEW_X also iwhere (by code), the ring columns of S and Y in ring order from head, t (the
previous iterate), the previous gradient (the oracle keeps it in r) and lnsrlb's direction d.  z, xp and subsm's
direction are left out: the fused pipeline keeps them lazy (DESIGN.md section 6, "Lazy vectors").

Bit-exact class: problems that by construction never pass a breakpoint in the Cauchy search (nseg <= 1) and never
have a variable enter or leave the free set.  There the two sides differ in nothing (DESIGN.md section 3) and every
field must have identical bits, REAL64 and REAL32 alike.  The CPU tests at the end of the file check with the oracle
alone that each case still has that property and still runs past m + 2 iterations (the ring of S/Y columns wraps).

Walk class: the bound-heavy problems of the other parity tests, where the breakpoint walk and formk's
entering/leaving corrections add in another order.  There the discrete state must be equal after every call, iwhere
element for element at every NEW_X, and x at every call within the tolerances the scalar traces use.

Independent float64 checks at every NEW_X, from the engine's own vectors: ||proj g|| (dsave[12]) is the max of the
projected gradient exactly; the newest S/Y column is stp * d and g - gold of the previous NEW_X exactly; theta,
dtd and dnorm lie within the rounding bound gamma_n * sum|terms| of sums recomputed with math.fsum.

A difference is reported with the call number, iteration, task and field, and for a vector with the first
differing index and where it lies in the fixed reduction shape (include/lbfgsb_b200_shape.h): tile, TMA stage
(512 elements, 256 for the half sub-tiles of REAL64 with m > 10), wave of 592 tiles, and whether the stage is the
ragged one that the consumer warps fill themselves (tma_pipe.cuh)."""
import ctypes as C
import math

import numpy as np
import pytest

import harness as H
from oracle import oracle_py as O
from test_gpu_drivers import RTOL_EARLY, RTOL_LATE

GRID = 592
ISAVE_SLOTS = {21: "nintol", 24: "iback", 25: "nskip", 26: "head", 27: "col", 28: "itail", 29: "iter", 30: "iupdat",
               32: "nseg", 33: "nfgv", 34: "info", 35: "ifun", 36: "iword", 37: "nfree", 38: "nact", 39: "ileave",
               40: "nenter", 42: "brackt", 43: "stage"}
DSAVE_SLOTS = dict([(0, "theta"), (1, "fold"), (2, "tol"), (3, "dnorm"), (4, "epsmch"), (10, "gd"), (11, "stpmx"),
                    (12, "sbgnrm"), (13, "stp"), (14, "gdold"), (15, "dtd")] +
                   [(16 + q, "dcsrch[%d]" % q) for q in range(13)])
PIPES = {"fast": {}, "nofast": {"LBFGSB_B200_NO_FAST": "1"}, "nofusion": {"LBFGSB_B200_NO_FUSION": "1"}}


# ---------------------------------------------------------------------------------------------------------------------
# problems


def far_box(n, dtype):
    """The sample objective with a box so far away that no variable ever reaches it (no breakpoint is passed)."""
    x = np.full(n, 3.0, dtype=dtype)
    return x, np.full(n, -1.0e3, dtype=dtype), np.full(n, 1.0e3, dtype=dtype), np.full(n, 2, np.int32)


def _pinned_data(n):
    rng = np.random.default_rng(n)
    pin = np.zeros(n, bool)
    pin[0::5] = True
    pin[2::5] = True
    a = rng.uniform(0.5, 2.0, n)
    c = np.where(pin, -1.0, rng.uniform(-1.0, 1.0, n))
    return pin, a, c


def pinned(n, dtype):
    """40 % of the variables start on their lower bound 0 with their target -1 below it and stay there: a constant
    active set; the others move freely inside [-1e3, 1e3]."""
    pin, _, _ = _pinned_data(n)
    x = np.where(pin, 0.0, 1.0).astype(dtype)
    l = np.where(pin, 0.0, -1.0e3).astype(dtype)
    return x, l, np.full(n, 1.0e3, dtype=dtype), np.where(pin, 1, 2).astype(np.int32)


def pinned_fg(n, dtype):
    """f = sum a (x - c)^2 + 1/4 (x - c)^4 + kappa/2 sum (x[i+1] - x[i])^2, evaluated in the real kind of x."""
    _, a, c = _pinned_data(n)
    a, c, kappa = a.astype(dtype), c.astype(dtype), dtype(0.05)

    def fg(x, g):
        r = x - c
        t = x[1:] - x[:-1]
        g[:] = dtype(2) * a * r + r * r * r
        g[1:] += kappa * t
        g[:-1] -= kappa * t
        return (a * r * r).sum() + dtype(0.25) * (r * r * r * r).sum() + dtype(0.5) * kappa * (t * t).sum()
    return fg


def unbounded(n, dtype):
    """nbd = 0 everywhere: no Cauchy point once the history holds a pair (the :607-611 branch)."""
    return np.full(n, 1.5, dtype=dtype), np.zeros(n, dtype), np.zeros(n, dtype), np.zeros(n, np.int32)


FAMILIES = {"far": (far_box, lambda n, dt: O.rosenbrock_fg),
            "pinned": (pinned, pinned_fg),
            "nbd0": (unbounded, lambda n, dt: O.rosenbrock_fg)}

F64, F32 = np.float64, np.float32
N_WAVE64 = GRID * 2048 + 1       # one tile into the second wave, REAL64 (2048-variable tiles)
N_WAVE32 = GRID * 4096 + 1       # the same for REAL32 (4096-variable tiles)

# (family, n, m, dtype, pipeline, iteration budget).  Every combination of the real kind, the instance of the streaming
# passes (MT = 5, 10, 20: m <= 5, m <= 10, m <= 20) and the pipeline runs at least once (test_bit_exact_cases_cover_
# every_kind_instance_and_pipeline), among them REAL64 m = 10 on the default pipeline (bench.py's headline shape); the
# n of the list and the m of each instance are spread over those combinations (not every n with every pipeline).
# Every far-box budget is at least m + 3 so that the ring of S/Y columns wraps; the pinned family (which converges in
# 7-20 iterations) carries the small m.
EXACT_CASES = [
    ("far", 65, 5, F64, "fast", 9),
    ("far", 511, 10, F32, "nofast", 14),
    ("far", 513, 11, F64, "nofusion", 15),
    ("far", 2047, 17, F64, "fast", 21),
    ("far", 2049, 20, F32, "fast", 24),
    ("far", 4095, 6, F64, "nofast", 10),
    ("far", 4097, 10, F64, "fast", 14),
    ("nbd0", 2049, 10, F64, "fast", 13),
    ("pinned", 2047, 8, F64, "nofusion", 11),
    ("far", 4097, 10, F32, "nofusion", 14),
    ("far", 6143, 20, F64, "nofast", 24),
    ("far", 100003, 11, F32, "fast", 15),
    ("far", 6143, 17, F32, "nofast", 20),
    ("far", 513, 20, F32, "nofusion", 23),
    ("far", 100003, 17, F64, "nofusion", 21),
    ("far", N_WAVE64, 11, F64, "fast", 15),
    ("far", N_WAVE32, 3, F32, "fast", 6),
    ("pinned", 65, 1, F32, "fast", 5),
    ("pinned", 511, 1, F64, "nofast", 5),
    ("pinned", 513, 6, F32, "fast", 9),
    ("pinned", 2049, 2, F64, "nofusion", 6),
    ("pinned", 4097, 3, F32, "nofast", 7),
    ("pinned", 6143, 3, F64, "fast", 7),
    ("pinned", 100003, 2, F32, "nofusion", 6),
    ("nbd0", 65, 10, F64, "nofast", 14),
    ("nbd0", 2047, 5, F64, "fast", 9),
    ("nbd0", 4095, 3, F32, "nofusion", 7),
    ("nbd0", 100003, 6, F32, "fast", 10),
]


def _case_id(c):
    return "%s-n%d-m%d-%s-%s" % (c[0], c[1], c[2], "f64" if c[3] == F64 else "f32", c[4])


# ---------------------------------------------------------------------------------------------------------------------
# the lock-step harness


def _where(i, n, m, dtype):
    """Where variable i lies in the fixed reduction shape and the TMA ring of the streaming passes."""
    tile = 2048 if dtype == F64 else 4096
    stage = 256 if (dtype == F64 and m > 10) else 512
    t, s = i // tile, (i % tile) // stage
    base = t * tile + s * stage
    return "index %d (tile %d, stage %d of %d elements [%d, %d), wave %d, %s stage)" % (
        i, t, s, stage, base, base + stage, t // GRID, "ragged" if base + stage > n else "full")


def _bits(a):
    a = np.ascontiguousarray(a)
    return a.view({8: np.uint64, 4: np.uint32}[a.dtype.itemsize])


class Mismatch(AssertionError):
    pass


class _Side:
    def __init__(self, setulb, n, m, x, dtype):
        self.setulb = setulb
        self.x = x
        self.g = np.zeros(n, dtype)
        self.f = np.zeros(1, dtype)
        self.wa, self.iwa = setulb.workspace(n, m)
        self.task, self.csave = H.make_task("START"), H.make_task("")
        self.lsave, self.isave, self.dsave = np.zeros(4, np.int32), np.zeros(44, np.int32), np.zeros(29, dtype)

    def call(self, n, m, l, u, nbd, factr, pgtol):
        self.setulb(n, m, self.x, l, u, nbd, self.f, self.g, factr, pgtol, self.wa, self.iwa, self.task, -1, self.csave,
                    self.lsave, self.isave, self.dsave)
        return H.task_str(self.task)


def engine_vector(eng, which, count, dtype):
    """Copy of an engine work vector (lbfgsb_dev_vector_copy) as a numpy array."""
    import torch
    import lbfgsb_b200
    tdt = torch.int32 if which == 7 else (torch.float64 if dtype == F64 else torch.float32)
    out = torch.empty(count, dtype=tdt, device="cuda")
    rc = lbfgsb_b200.lib().lbfgsb_dev_vector_copy(C.c_void_p(eng), which, C.c_void_p(out.data_ptr()),
                                                  C.c_int64(out.numel() * out.element_size()))
    assert rc == 0, "lbfgsb_dev_vector_copy(%d) failed" % which
    return out.cpu().numpy()


def projected_gradient_norm(x, g, l, u, nbd):
    """projgr (:2594-2622) in the real kind of x."""
    lo = (nbd != 0) & (nbd <= 2) & (g >= 0)
    hi = (nbd >= 2) & (g < 0)
    gi = np.where(hi, np.maximum(x - u, g), np.where(lo, np.minimum(x - l, g), g))
    return np.abs(gi).max()


def _gamma(n, dtype):
    u = float(np.finfo(dtype).eps) / 2
    return n * u / (1 - n * u)


class LockStep:
    def __init__(self, n, m, dtype, l, u, nbd, exact, label):
        self.n, self.m, self.dtype, self.l, self.u, self.nbd = n, m, np.dtype(dtype), l, u, nbd
        self.exact, self.label = exact, label
        self.ldw = (n + 31) // 32 * 32
        self.prev = None          # (g, gold, d, stp, iupdat) of the previous NEW_X, engine side
        self.checked = {"theta": 0, "sy": 0}
        self.errors = []          # the first difference of every field, in the order met

    def fail(self, ctx, field, msg):
        """Records the first difference of a field; the run goes on (each side iterates from its own x) so that one
        failure shows every field that differs, the earliest first."""
        if field not in [e[0] for e in self.errors]:
            self.errors.append((field, "%s, %s: %s" % (ctx, field, msg)))

    def report(self):
        if self.errors:
            raise Mismatch("%s: %d field(s) differ; first:\n  " % (self.label, len(self.errors)) +
                           "\n  ".join(e[1] for e in self.errors[:12]))

    def vec(self, ctx, field, a, b, tol=None):
        if tol is None:
            bad = np.nonzero(_bits(a) != _bits(b))[0]
        else:
            bad = np.nonzero(~(np.abs(a.astype(F64) - b.astype(F64)) <= tol))[0]
        if bad.size:
            i = int(bad[0])
            self.fail(ctx, field, "%d of %d elements differ%s; first at %s: engine %r, oracle %r" % (
                bad.size, a.size, "" if tol is None else " by more than %.3g" % tol, _where(i, self.n, self.m, self.dtype),
                a[i], b[i]))

    def scalars(self, ctx, e, o):
        for k in ("task", "csave"):
            te, to = H.task_str(getattr(e, k)), H.task_str(getattr(o, k))
            if te != to:
                self.fail(ctx, k, "engine %r, oracle %r" % (te, to))
                self.report()        # the two sides no longer take the same branch: stop here
        if not np.array_equal(e.lsave, o.lsave):
            self.fail(ctx, "lsave", "engine %s, oracle %s" % (list(e.lsave), list(o.lsave)))
        for k, nm in ISAVE_SLOTS.items():
            if k == 39 and H.task_str(o.task) == "FG_START":
                continue     # ileave: set by freev (n + 1 when nothing leaves); the reference leaves it undefined before
            if e.isave[k] != o.isave[k]:
                self.fail(ctx, "isave[%d] (%s)" % (k, nm), "engine %d, oracle %d" % (e.isave[k], o.isave[k]))
        if self.exact:
            for k, nm in DSAVE_SLOTS.items():
                if _bits(e.dsave[k:k + 1])[0] != _bits(o.dsave[k:k + 1])[0]:
                    self.fail(ctx, "dsave[%d] (%s)" % (k, nm), "engine %r, oracle %r" % (e.dsave[k], o.dsave[k]))
            if _bits(e.f)[0] != _bits(o.f)[0]:
                self.fail(ctx, "f", "engine %r, oracle %r" % (e.f[0], o.f[0]))
            self.vec(ctx, "x", e.x, o.x)
        else:
            tol = (RTOL_EARLY if o.isave[29] <= 10 else RTOL_LATE) * max(1.0, float(np.abs(o.x).max()))
            self.vec(ctx, "x", e.x, o.x, tol=tol)

    def at_newx(self, ctx, eng, e, o):
        n, m, dt = self.n, self.m, self.dtype
        iw = engine_vector(eng, 7, n, dt)
        self.vec(ctx, "iwhere", iw, o.iwa[n:2 * n])
        d = engine_vector(eng, 2, n, dt)
        gold = engine_vector(eng, 8, n, dt)
        col, head, itail = int(e.isave[27]), int(e.isave[26]), int(e.isave[28])
        ws = wy = None
        if col > 0:
            ws = engine_vector(eng, 5, m * self.ldw, dt)
            wy = engine_vector(eng, 6, m * self.ldw, dt)
        if self.exact:
            mn = m * n
            for k in range(col):
                j = (head - 1 + k) % m
                self.vec(ctx, "ws column %d (ring position %d of %d)" % (j, k, col), ws[j * self.ldw:j * self.ldw + n],
                         o.wa[j * n:(j + 1) * n])
                self.vec(ctx, "wy column %d (ring position %d of %d)" % (j, k, col), wy[j * self.ldw:j * self.ldw + n],
                         o.wa[mn + j * n:mn + (j + 1) * n])
            z0 = 2 * mn + 11 * m * m            # oracle wa: ws, wy, sy, ss, wt, wn, snd, then z, r, d, t, xp
            self.vec(ctx, "t (previous x)", engine_vector(eng, 3, n, dt), o.wa[z0 + 3 * n:z0 + 4 * n])
            self.vec(ctx, "previous gradient (oracle r)", gold, o.wa[z0 + n:z0 + 2 * n])
            self.vec(ctx, "d (lnsrlb direction)", d, o.wa[z0 + 2 * n:z0 + 3 * n])
        self.independent(ctx, e, d, gold, ws, wy, col, itail)
        self.prev = (e.g.copy(), gold, d, e.dsave[13], int(e.isave[30]))

    def independent(self, ctx, e, d, gold, ws, wy, col, itail):
        """Checks of the engine's own state against float64 recomputations (not against the oracle)."""
        dt, n = self.dtype, self.n
        u = float(np.finfo(dt).eps) / 2
        pg = projected_gradient_norm(e.x, e.g, self.l, self.u, self.nbd)
        if _bits(np.array([pg], dt))[0] != _bits(e.dsave[12:13])[0]:
            self.fail(ctx, "dsave[12] (sbgnrm) vs max |proj g| from x, g, l, u", "engine %r, numpy %r" % (e.dsave[12], pg))
        # dtd and dnorm of lnsrlb's first entry, from the stored direction
        dd = d.astype(F64)
        dtd = math.fsum(dd * dd)
        gam = _gamma(n, dt)
        if not abs(float(e.dsave[15]) - dtd) <= gam * dtd:
            self.fail(ctx, "dsave[15] (dtd) vs fsum(d*d)", "engine %r, fsum %r, bound %.3g" % (e.dsave[15], dtd, gam * dtd))
        if not abs(float(e.dsave[3]) - math.sqrt(dtd)) <= (gam / 2 + 2 * u) * math.sqrt(dtd):
            self.fail(ctx, "dsave[3] (dnorm) vs sqrt(fsum(d*d))", "engine %r, fsum %r" % (e.dsave[3], math.sqrt(dtd)))
        if self.prev is None or col == 0 or int(e.isave[30]) != self.prev[4] + 1:
            return
        # an S/Y pair was added since the previous NEW_X: the newest column is that iteration's step and gradient change
        gp, goldp, dp, stpp, _ = self.prev
        j = itail - 1
        s = ws[j * self.ldw:j * self.ldw + n]
        y = wy[j * self.ldw:j * self.ldw + n]
        s_ref = dp if stpp == 1 else (dt.type(stpp) * dp).astype(dt)
        self.vec(ctx, "newest ws column %d vs stp * d of the previous NEW_X" % j, s, s_ref)
        self.vec(ctx, "newest wy column %d vs g - gold of the previous NEW_X" % j, y, (gp - goldp).astype(dt))
        self.checked["sy"] += 1
        # theta = y'y / dr, dr = (g.d - gold.d) * stp (matupd :2338, mainlb :817-824)
        sf, yf = s.astype(F64), y.astype(F64)
        rr, sy = math.fsum(yf * yf), math.fsum(sf * yf)
        if sy <= 0:
            return
        dpf = dp.astype(F64)
        g2 = _gamma(n + 4, dt)
        e_dr = g2 * (float(stpp) * (math.fsum(np.abs(gp.astype(F64) * dpf)) + math.fsum(np.abs(goldp.astype(F64) * dpf)))
                     + math.fsum(np.abs(sf * yf)))
        rel = gam + e_dr / sy
        th = rr / sy
        if not abs(float(e.dsave[0]) - th) <= th * (rel + 2 * u) / (1 - rel):
            self.fail(ctx, "dsave[0] (theta) vs fsum(y*y)/fsum(s*y)", "engine %r, fsum %r, bound %.3g" % (
                e.dsave[0], th, th * (rel + 2 * u) / (1 - rel)))
        self.checked["theta"] += 1


def lockstep(fg, mk, n, m, dtype, factr, pgtol, budget, exact, label):
    """Drives the host twin and the oracle call by call; returns the engine side's trace of (iter, nseg, nenter,
    nleave) per NEW_X and the harness (for its counters)."""
    import lbfgsb_b200
    x, l, u, nbd = mk()
    ls = LockStep(n, m, dtype, l, u, nbd, exact, label)
    host = lbfgsb_b200.HostSetulb(dtype)
    e = _Side(host, n, m, x.copy(), dtype)
    o = _Side(O.OracleSetulb(dtype), n, m, x.copy(), dtype)
    rows = []
    calls = 0
    O.set_sum_mode(1)
    try:
        while True:
            ts = H.task_str(e.task)
            if not (ts[:2] == "FG" or ts[:5] == "NEW_X" or ts == "START" or ts.startswith("STOP")) or calls > 20 * budget + 50:
                break
            te = e.call(n, m, l, u, nbd, factr, pgtol)
            o.call(n, m, l, u, nbd, factr, pgtol)
            calls += 1
            ctx = "call %d (iteration %d, task %r)" % (calls, int(o.isave[29]), H.task_str(o.task))
            ls.scalars(ctx, e, o)
            if te[:2] == "FG":
                e.f[0] = fg(e.x, e.g)
                o.f[0] = fg(o.x, o.g)
            elif te[:5] == "NEW_X":
                ls.at_newx(ctx, host.engine(), e, o)
                rows.append((int(e.isave[29]), int(e.isave[32]), int(e.isave[40]), n + 1 - int(e.isave[39])))
                if e.isave[29] >= budget:
                    e.task[:] = H.make_task("STOP: ITERATION BUDGET")
                    o.task[:] = H.make_task("STOP: ITERATION BUDGET")
            else:
                break
    finally:
        O.set_sum_mode(0)
        host.release(e.isave)
    ls.report()
    return rows, ls


# ---------------------------------------------------------------------------------------------------------------------
# bit-exact class


@pytest.mark.gpu
@pytest.mark.parametrize("case", EXACT_CASES, ids=_case_id)
def test_lockstep_bit_exact(case, monkeypatch):
    fam, n, m, dtype, pipe, budget = case
    for k, v in PIPES[pipe].items():
        monkeypatch.setenv(k, v)     # read when the workspace is created (host twin: at START)
    mk, fgm = FAMILIES[fam]
    rows, ls = lockstep(fgm(n, dtype), lambda: mk(n, dtype), n, m, dtype, 0.0, 0.0, budget, True, _case_id(case))
    assert len(rows) == budget, (len(rows), budget)
    assert ls.checked["sy"] >= budget - 2 and ls.checked["theta"] >= budget - 2, ls.checked


# ---------------------------------------------------------------------------------------------------------------------
# walk class


def _bound_heavy(n, l_odd, x0=3.0):
    return lambda: H.rosenbrock_problem(n, l_odd=l_odd, x0=x0)


WALK_CASES = [
    # test_gpu_drivers.py::test_bound_heavy_rosenbrock
    ("bound-heavy-1000", 1000, 5, 1.0e7, 1.0e-5, 12, _bound_heavy(1000, 1.1), None),
    ("bound-heavy-4097", 4097, 10, 1.0e7, 1.0e-5, 12, _bound_heavy(4097, 1.1), None),
    ("bound-heavy-20000", 20000, 10, 1.0e7, 1.0e-5, 12, _bound_heavy(20000, 1.5), None),
    ("bound-heavy-100000", 100000, 5, 1.0e7, 1.0e-5, 12, _bound_heavy(100000, 1.0), None),
    # test_gpu_rare_paths.py: exits inside a group of tied breakpoints, then subsm's backtrack (its two n = 200 000
    # cases are left out to keep the file's wall time short: they take the same branches at a larger n)
    ("ties-1000", 1000, 5, 0.0, 0.0, 8, _bound_heavy(1000, 2.0, 3.0), None),
    ("ties-3001", 3001, 3, 0.0, 0.0, 8, _bound_heavy(3001, 2.5, 5.0), None),
    ("ties-50001", 50001, 3, 0.0, 0.0, 8, _bound_heavy(50001, 1.3, 5.0), None),
]


@pytest.mark.gpu
@pytest.mark.parametrize("case", WALK_CASES, ids=lambda c: c[0])
def test_lockstep_walk_class(case):
    label, n, m, factr, pgtol, budget, mk, _ = case
    rows, _ = lockstep(O.rosenbrock_fg, mk, n, m, F64, factr, pgtol, budget, False, label)
    assert len(rows) >= min(budget, 8)
    assert any(r[1] > 1 or r[2] or r[3] for r in rows), "no iterate walked or changed the free set: not a walk case"


@pytest.mark.gpu
@pytest.mark.parametrize("seed", [11, 12, 13, 14, 15, 16])
def test_lockstep_walk_class_mixed_bounds(seed):
    from test_gpu_edge import sweep_problem
    n, m, fg, mk = sweep_problem(seed)
    rows, _ = lockstep(fg, mk, n, m, F64, 1e3, 1e-8, 10, False, "sweep-%d" % seed)
    assert len(rows) >= 1
    assert any(r[1] > 1 or r[2] or r[3] for r in rows), "no iterate walked or changed the free set: not a walk case"


# ---------------------------------------------------------------------------------------------------------------------
# CPU: the bit-exact cases still cover what they claim


def test_bit_exact_cases_cover_every_kind_instance_and_pipeline():
    def mt(m):
        return 5 if m <= 5 else (10 if m <= 10 else 20)
    have = {(np.dtype(c[3]).name, mt(c[2]), c[4]) for c in EXACT_CASES}
    want = {(np.dtype(d).name, t, p) for d in (F64, F32) for t in (5, 10, 20) for p in PIPES}
    assert want <= have, sorted(want - have)
    assert ("far", N_WAVE64, 11, F64, "fast", 15) in EXACT_CASES and any(c[1] == N_WAVE32 and c[3] == F32 for c in EXACT_CASES)


@pytest.mark.parametrize("case", EXACT_CASES, ids=_case_id)
def test_bit_exact_case_never_walks_nor_changes_the_free_set(case):
    fam, n, m, dtype, pipe, budget = case
    mk, fgm = FAMILIES[fam]
    assert budget >= m + 3
    x, l, u, nbd = mk(n, dtype)
    O.set_sum_mode(1)
    try:
        tr = H.run_driver(O.OracleSetulb(dtype), fgm(n, dtype), n, m, x, l, u, nbd, 0.0, 0.0,
                          stop=H.iteration_budget_stop(budget), want_hash=False)
    finally:
        O.set_sum_mode(0)
    rows = tr[0]
    assert len(rows) == budget, (len(rows), tr[1])
    for r in rows:
        # nbd = 0: one segment at iteration 0 (col = 0), no Cauchy search after it
        assert r["nseg"] == (0 if fam == "nbd0" and r["iter"] > 1 else 1), r
        assert r["nenter"] == 0 and r["nleave"] == 0, r
        assert r["nskip"] == 0, r
    assert rows[-1]["col"] == min(m, budget - 1), rows[-1]


# ---------------------------------------------------------------------------------------------------------------------
# caller buffers of the device variant: nothing past n is read or written

PAD = 4096     # bytes of poison in front of and behind every caller buffer


def _device_trace(n, m, dtype, x, l, u, nbd, g, budget=10):
    import lbfgsb_b200
    prob = lbfgsb_b200.DeviceProblem(n, m, dtype)
    fg = lbfgsb_b200.RosenbrockDevice(dtype)
    rows = []
    try:
        for _ in range(50 * budget):
            prob.setulb_dev(x, l, u, nbd, g, 0.0, 0.0)
            t = prob.task_str()
            if t[:2] == "FG":
                prob.f[0] = fg(x, g)
            elif t[:5] == "NEW_X":
                isv = np.concatenate([prob.isave[:16], prob.isave[20:]])     # not the handle slots
                dsv = np.concatenate([prob.dsave[:5], prob.dsave[10:]])      # not the clock slots
                rows.append((t, isv.copy(), _bits(dsv).copy(), _bits(prob.f).copy()))
                if prob.isave[29] >= budget:
                    break
            else:
                break
    finally:
        prob.close()
    return rows, x.cpu().numpy()


@pytest.mark.gpu
@pytest.mark.parametrize("n", [4097, 100003])
@pytest.mark.parametrize("dtype", [F64, F32], ids=["f64", "f32"])
@pytest.mark.parametrize("shift", [0, 16], ids=["aligned512", "offset16"])
def test_device_variant_reads_and_writes_nothing_past_n(n, dtype, shift):
    """x, g, l, u, nbd passed as views into larger tensors whose 4 KB in front and behind are poisoned (NaN for the
    reals, 7 for nbd), the view starting on a 512-byte boundary or 16 bytes past one (the ABI's minimum alignment):
    the trace is bit for bit that of a run on exact-size tensors, and the poison is byte for byte unchanged."""
    import torch
    m = 5
    x0, l0, u0, nbd0 = H.rosenbrock_problem(n, dtype=dtype, l_odd=1.1)
    tdt = torch.float64 if dtype == F64 else torch.float32
    exact = [torch.from_numpy(a).cuda() for a in (x0, l0, u0, nbd0)] + [torch.zeros(n, dtype=tdt, device="cuda")]
    want, want_x = _device_trace(n, m, dtype, *exact)
    assert len(want) == 10

    bufs, views = [], []
    for a in (x0, l0, u0, nbd0, np.zeros(n, dtype)):
        es = a.dtype.itemsize
        buf = torch.full((2 * PAD // es + n + 16 // es,), 7 if a.dtype == np.int32 else float("nan"),
                         dtype=torch.int32 if a.dtype == np.int32 else tdt, device="cuda")
        assert buf.data_ptr() % 512 == 0
        k0 = (PAD + shift) // es
        v = buf[k0:k0 + n]
        v.copy_(torch.from_numpy(a))
        assert v.data_ptr() % 512 == shift
        bufs.append((buf, k0, buf.view(torch.int64 if es == 8 else torch.int32).clone()))
        views.append(v)
    got, got_x = _device_trace(n, m, dtype, *views)
    assert len(got) == len(want)
    for k, (a, b) in enumerate(zip(got, want)):
        assert a[0] == b[0] and np.array_equal(a[1], b[1]) and np.array_equal(a[2], b[2]) and np.array_equal(a[3], b[3]), (
            "NEW_X %d differs from the run on exact-size tensors" % (k + 1), a, b)
    assert np.array_equal(_bits(got_x), _bits(want_x))
    for name, (buf, k0, before) in zip(("x", "l", "u", "nbd", "g"), bufs):
        after = buf.view(before.dtype)
        for lo, hi, side in ((0, k0, "in front of"), (k0 + n, buf.numel(), "behind")):
            bad = torch.nonzero(after[lo:hi] != before[lo:hi])
            assert bad.numel() == 0, "%s: %d poisoned elements %s the view were written, first at offset %d" % (
                name, bad.numel(), side, int(bad[0, 0]) + lo - k0)


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [F64, F32], ids=["f64", "f32"])
def test_vector_copy_refuses_requests_beyond_the_allocation(dtype):
    import torch
    import lbfgsb_b200
    n, m = 1000, 5
    ldw, es = 1024, np.dtype(dtype).itemsize
    prob = lbfgsb_b200.DeviceProblem(n, m, dtype)
    dst = torch.zeros(m * ldw * es + 256, dtype=torch.uint8, device="cuda")
    try:
        for which, cap in ((0, ldw * es), (2, ldw * es), (3, ldw * es), (5, m * ldw * es), (6, m * ldw * es), (7, ldw * 4),
                           (8, ldw * es)):
            copy = lbfgsb_b200.lib().lbfgsb_dev_vector_copy
            assert copy(C.c_void_p(prob.h), which, C.c_void_p(dst.data_ptr()), C.c_int64(cap)) == 0, which
            assert copy(C.c_void_p(prob.h), which, C.c_void_p(dst.data_ptr()), C.c_int64(cap + 1)) == 1, which
        with pytest.raises(lbfgsb_b200.LbfgsbB200Error):
            prob.vector(5, count=m * ldw + 1)
        assert prob.vector(5, count=m * ldw).numel() == m * ldw
    finally:
        prob.close()
