"""Edge cases of the iteration path against the oracle (same f/g routine on both sides): tiny n, m = 1, m > n,
every variable fixed, start on the bounds, non-convex objectives that skip BFGS updates (:826-834) and backtrack in the line
search, and a seeded sweep over mixed bound kinds."""
import numpy as np
import pytest

import harness as H
from oracle import oracle_py as O
from test_gpu_drivers import DISCRETE, RTOL_EARLY, RTOL_LATE

pytestmark = pytest.mark.gpu


def _both(fg, mk, n, m, factr=1e7, pgtol=1e-5, budget=40, dtype=np.float64):
    import lbfgsb_b200
    stop = H.iteration_budget_stop(budget)
    x, l, u, nbd = mk()
    gpu = H.run_driver(lbfgsb_b200.HostSetulb(dtype), fg, n, m, x, l, u, nbd, factr, pgtol, stop=stop)
    x, l, u, nbd = mk()
    O.set_sum_mode(1)
    try:
        ref = H.run_driver(O.OracleSetulb(dtype), fg, n, m, x, l, u, nbd, factr, pgtol, stop=stop)
    finally:
        O.set_sum_mode(0)
    return gpu, ref


def _check(gpu, ref, upto=12, whole=False):
    k = min(len(ref[0]), upto)
    assert len(gpu[0]) >= k, (len(gpu[0]), len(ref[0]), gpu[1], ref[1])
    for a, b in list(zip(gpu[0], ref[0]))[:k]:
        for kk in DISCRETE:
            assert a[kk] == b[kk], (kk, a, b)
        tol = RTOL_EARLY if b["iter"] <= 10 else RTOL_LATE
        assert abs(a["f"] - b["f"]) <= tol * abs(b["f"]) + 1e-300, (a, b)
        assert abs(a["sbgnrm"] - b["sbgnrm"]) <= 10 * tol * abs(b["sbgnrm"]) + 1e-300, (a, b)
    if whole:
        assert gpu[1] == ref[1] and len(gpu[0]) == len(ref[0])


@pytest.mark.parametrize("n,m", [(1, 1), (1, 5), (2, 1), (2, 3), (3, 5), (5, 20), (7, 3), (33, 17)])
def test_tiny_problems(n, m):
    gpu, ref = _both(O.rosenbrock_fg, lambda: H.rosenbrock_problem(n), n, m)
    _check(gpu, ref, upto=15, whole=(n <= 3))


def test_all_variables_fixed_and_start_on_bounds():
    import lbfgsb_b200
    n, m = 1000, 5

    def fixed():
        x = np.full(n, 2.0)
        return x, np.full(n, 2.0), np.full(n, 2.0), np.full(n, 2, np.int32)
    gpu, ref = _both(O.rosenbrock_fg, fixed, n, m)
    assert gpu[1] == ref[1] and gpu[1].startswith("CONVERGENCE: NORM_OF_PROJECTED_GRADIENT") and len(gpu[0]) == len(ref[0]) == 0

    # x0 on the lower bounds with the gradient pointing out of the box: projected gradient zero at once
    def fq(x, g):
        g[:] = 1.0 + x
        return float((x + 0.5 * x * x).sum())

    def onb():
        return np.zeros(n), np.zeros(n), np.ones(n), np.full(n, 2, np.int32)
    gpu, ref = _both(fq, onb, n, m)
    assert gpu[1] == ref[1] and gpu[1].startswith("CONVERGENCE") and len(gpu[0]) == len(ref[0]) == 0
    # infeasible start: projected at START (active :983-1009), prjctd reported in lsave(1)
    def out():
        return np.full(n, -5.0), np.zeros(n), np.ones(n), np.full(n, 2, np.int32)
    gpu, ref = _both(fq, out, n, m)
    assert gpu[1] == ref[1] and np.array_equal(gpu[2], ref[2]) and np.all(gpu[2] == 0.0)
    del lbfgsb_b200


def _nonconvex(n, seed, share, a_c):
    """A box-constrained objective with a concave part: -a_c * a * x^2 on a share of the variables (the minimiser of
    those lies on a bound), a * (x - b)^2 on the others, coupled by 1/4 sum (x[i+1] - x[i])^2.  Along a step into
    the concave part s'y <= 0, and the update is skipped (:826-834)."""
    rng = np.random.default_rng(seed)
    conc = rng.random(n) < share
    a = rng.uniform(0.5, 2.0, n)
    b = rng.uniform(-1.0, 1.0, n)

    def fg(x, g):
        r = x - b
        t = x[1:] - x[:-1]
        g[:] = np.where(conc, -2.0 * a_c * a * x, 2.0 * a * r)
        g[1:] += 0.5 * t
        g[:-1] -= 0.5 * t
        return float(np.where(conc, -a_c * a * x * x, a * r * r).sum() + 0.25 * (t * t).sum())

    def mk():
        r2 = np.random.default_rng(seed + 100)
        return r2.uniform(-0.5, 0.5, n), np.full(n, -2.0), np.full(n, 2.0), np.full(n, 2, np.int32)
    return fg, mk


@pytest.mark.parametrize("n,m,seed,share,a_c", [(400, 5, 0, 0.5, 0.3), (3000, 10, 1, 0.3, 1.0), (20001, 7, 2, 0.1, 2.0)])
def test_nonconvex_objective_with_skips_and_line_search_backtracks(n, m, seed, share, a_c):
    fg, mk = _nonconvex(n, seed, share, a_c)
    O.event_counts()
    gpu, ref = _both(fg, mk, n, m, factr=0.0, pgtol=0.0, budget=30)
    ev = O.event_counts()
    _check(gpu, ref, upto=14)
    # the oracle skipped an update with pairs in the memory (col > 0) and backtracked in the line search
    assert ev[3] >= 1, ev
    assert any(b["nskip"] > a["nskip"] and a["col"] > 0 for a, b in zip(ref[0][:14], ref[0][1:14])), ref[0][:14]
    assert any(r["iback"] > 0 for r in ref[0][:14])


def sweep_problem(seed):
    """(n, m, fg, mk) of a seeded mixed-bound problem: nbd in {0, 1, 2, 3}, 3 % fixed variables, a coupled quartic."""
    rng = np.random.default_rng(seed)
    n = int(rng.integers(60, 6000))
    m = int(rng.integers(1, 13))
    a = rng.uniform(0.5, 3.0, n)
    b = rng.uniform(-2.0, 2.0, n)

    def fg(x, g):
        r = x - b
        t = x[1:] - x[:-1]
        f = float((a * r * r).sum() + 0.25 * float((r ** 4).sum()) + 0.5 * float((t * t).sum()))
        g[:] = 2 * a * r + r ** 3
        g[1:] += t
        g[:-1] -= t
        return f

    def mk():
        r2 = np.random.default_rng(seed + 1000)
        x = r2.uniform(-3, 3, n)
        l = r2.uniform(-2.5, 0.5, n)
        u = l + r2.uniform(0.0, 3.0, n)
        nbd = r2.integers(0, 4, n).astype(np.int32)
        fx = r2.random(n) < 0.03
        u[fx] = l[fx]
        nbd[fx] = 2
        return x, l, u, nbd
    return n, m, fg, mk


@pytest.mark.parametrize("seed", [11, 12, 13, 14, 15, 16])
def test_seeded_sweep_mixed_bounds(seed):
    n, m, fg, mk = sweep_problem(seed)
    gpu, ref = _both(fg, mk, n, m, factr=1e3, pgtol=1e-8, budget=25)
    _check(gpu, ref, upto=10)
