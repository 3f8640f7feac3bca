"""Development aid: the batch's task loop on the host (BatchProblem.solve) against the same loop on the device
(BatchProblem.solve_graph, include/lbfgsb_b200.h section 6) on the same seeded problems, alternating, three runs each, in
one process.  Problems of tools/batch_rate.py (driver1's box, perturbed start, factr 1e7, pgtol 1e-5), the batched sample
objective.  Prints one JSON line per shape and run with problems/s, calls, graph launches and us per call, checks that x of
both paths are bitwise equal, and names the card and its power limit.
    python tools/batch_graph_rate.py [--shapes 1000x25x5,10000x25x5,1000x2049x10] [--profile DIR]
--profile DIR: afterwards one solve and one solve_graph of the first shape under torch.profiler (CUDA activities), a
table of device time per kernel and the traces in DIR."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from batch_rate import problems  # noqa: E402


def card():
    import torch
    out = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        out["power_limit_and_max_sm_clock"] = q[0] if q else "unknown"
    except (OSError, subprocess.SubprocessError):
        out["power_limit_and_max_sm_clock"] = "unknown"
    return out


def one_run(b, path, x0, xd, ld, ud, nd, fd, gd, factr, pgtol):
    import torch
    xd.copy_(x0)
    gd.zero_()
    fd.zero_()
    torch.cuda.synchronize()
    builds0, launches0, _ = b.graph_stats()
    t0 = time.perf_counter()
    if path == "solve":
        for p in range(b.nprob):
            b.set_task(p, "START")
        calls = b.solve(xd, ld, ud, nd, fd, gd, factr, pgtol)
    else:
        calls = b.solve_graph(xd, ld, ud, nd, fd, gd, factr, pgtol)
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    builds, launches, _ = b.graph_stats()
    conv = int(sum(1 for p in range(b.nprob) if b.task[p, 0] == ord("C")))
    return {"path": path, "seconds": dt, "problems_per_s": b.nprob / dt, "calls": calls, "us_per_call": dt / calls * 1e6,
            "graph_launches": launches - launches0, "graph_builds": builds - builds0, "converged": conv,
            "iterations_total": int(b.isave[:, 29].sum())}, xd.cpu().numpy().copy()


def shape_runs(nprob, n, m, runs=3, factr=1.0e7, pgtol=1.0e-5):
    import torch
    import lbfgsb_b200
    X, L, U, N = problems(nprob, n)
    x0 = torch.from_numpy(X).cuda()
    ld, ud, nd = (torch.from_numpy(a).cuda() for a in (L, U, N))
    xd, gd = torch.empty_like(x0), torch.empty_like(x0)
    fd = torch.empty(nprob, dtype=torch.float64, device="cuda")
    b = lbfgsb_b200.BatchProblem(nprob, n, m, np.float64)
    out = []
    try:
        for r in range(runs):
            row = {"shape": "%d x (n %d, m %d)" % (nprob, n, m), "run": r}
            a, xa = one_run(b, "solve", x0, xd, ld, ud, nd, fd, gd, factr, pgtol)
            g, xg = one_run(b, "solve_graph", x0, xd, ld, ud, nd, fd, gd, factr, pgtol)
            row["solve"], row["solve_graph"] = a, g
            row["x_bitwise_equal"] = bool(np.array_equal(xa.view(np.uint64), xg.view(np.uint64)))
            row["speedup"] = a["seconds"] / g["seconds"]
            out.append(row)
            print(json.dumps(row), flush=True)
    finally:
        b.close()
    return out


def profile(nprob, n, m, outdir, factr=1.0e7, pgtol=1.0e-5):
    import torch
    import lbfgsb_b200
    from torch.profiler import ProfilerActivity, profile as tprof
    os.makedirs(outdir, exist_ok=True)
    X, L, U, N = problems(nprob, n)
    x0 = torch.from_numpy(X).cuda()
    ld, ud, nd = (torch.from_numpy(a).cuda() for a in (L, U, N))
    xd, gd = torch.empty_like(x0), torch.empty_like(x0)
    fd = torch.empty(nprob, dtype=torch.float64, device="cuda")
    b = lbfgsb_b200.BatchProblem(nprob, n, m, np.float64)
    try:
        for path in ("solve", "solve_graph"):
            one_run(b, path, x0, xd, ld, ud, nd, fd, gd, factr, pgtol)      # warm: modules, graph
            with tprof(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
                res, _ = one_run(b, path, x0, xd, ld, ud, nd, fd, gd, factr, pgtol)
            prof.export_chrome_trace(os.path.join(outdir, "batch_%s_trace.json" % path))
            dev = sum(e.self_device_time_total for e in prof.key_averages()) / 1e3
            print("== %s under the profiler: %.3f ms wall, %d calls, %.3f ms device time in kernels and copies" % (
                path, res["seconds"] * 1e3, res["calls"], dev))
            print(prof.key_averages().table(sort_by="self_device_time_total", row_limit=12))
    finally:
        b.close()


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--shapes", default="1000x25x5,10000x25x5,1000x2049x10")
    ap.add_argument("--runs", type=int, default=3)
    ap.add_argument("--profile", default=None)
    a = ap.parse_args()
    import torch
    assert torch.cuda.is_available(), "batch_graph_rate needs a GPU"
    print(json.dumps({"card": card()}), flush=True)
    shapes = [tuple(int(v) for v in s.split("x")) for s in a.shapes.split(",")]
    allrows = []
    for nprob, n, m in shapes:
        allrows += shape_runs(nprob, n, m, runs=a.runs)
    assert all(r["x_bitwise_equal"] for r in allrows), "solve and solve_graph gave different x"
    if a.profile:
        profile(*shapes[0], a.profile)
