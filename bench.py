"""bench.py -- L-BFGS-B iterations/s on B200 (BASELINE.json metric), one JSON line on stdout.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference]
                    [--workload rosenbrock|quadratic|driver3_f32] [--scaling auto|strong|weak] [--n N] [--m M]
                    [--dump-outputs DIR]

A "step" is one L-BFGS-B iteration: one pass of mainlb's main loop ending in 'NEW_X'
(src/lbfgsb.f90:599-872) plus the caller's f/g evaluations for it (a device kernel inside the timed region).

Headline workload (config.workload): BASELINE.json configs[2] -- bounded extended Rosenbrock of test/driver1.f90
with the odd-index lower bound raised to 1.1 (about half of the variables end at a bound), n = 1e8, m = 10,
real64, factr = pgtol = 0 and a fixed iteration budget.
  N = 1   n = 1e8 on one GPU.
  N > 1   the SAME n = 1e8 sharded over the N GPUs ("scaling": "strong" -- configs[2] as written: "n=1e8 ... at
          1/2/4/8 B200"; value grows with N).  The weak series (n = 1e8 per GPU, and configs[3]: the quadratic at
          1.25e8 per GPU, n = 1e9 on 8 GPUs) is measured in the same run and reported under `extra_configs`,
          each with an aggregate variable-iterations/s figure.  --scaling weak makes the weak series the headline.

  value         iterations/s with x, g, l, u, nbd resident in HBM (lbfgsb_setulb_dev_f64), all K timed steps
  steady/burst  the same K steps split into steady iterations and burst iterations (nseg > 1 or more than n/100
                variables entering/leaving the free set), CUDA events per iteration on the engine's stream
  e2e           the same iterations with HOST x, g: the per-call H2D copy of g and D2H copy of x are inside the
                timed region (N = 1: the C-ABI host twin lbfgsb_setulb_f64; N > 1: lbfgsb_b200.sharded.HostShard)
  roofline      the dominant kernel family: algorithmic bytes per launch / CUDA-event time on the engine's stream
  cpu_baseline  the CPU oracle (line-by-line port of the reference; the Fortran reference cannot be built in this
                image) on a bounded sample, 1 core
  extra_configs BASELINE.json configs[3] (quadratic), configs[4] (n = 4e8, m = 20, REAL32), configs[1]
                (n = 1e6, m = 5 solved to convergence), configs[0] x 1000 as one batch and the fixed cost per iteration
                at small n (caller loop vs the CUDA-graph loop) at N = 1; the weak series at N > 1
  parity        N > 1: a 2e5-variable problem solved sharded and on one GPU -- discrete trace and active-set hash equal

Warm-up: the driver's --warmup is raised to m + 4 iterations (history full, col = m) and extended (up to 10 more)
until fewer than n/100 variables enter or leave the free set; `warmup` echoes the flag, `warmup_effective` says
what ran.  The headline times exactly --steps iterations (default 20; 12 for the quadratic, which converges after
about 34 iterations); a solve that ends before them is an error.
--impl reference times the CPU port of the reference on the same workload (N = 1: the full n).

--dump-outputs DIR writes what the headline's last timed iteration left in the caller's hands: DIR/x.npy and DIR/g.npy
(the iterate and its gradient, in the workload's dtype, at the global indices of DIR/index.npy: every variable up to
2^20 of them, else one variable at a hashed position in each of 2^20 equal stretches, fixed by integer arithmetic
alone) and DIR/f.npy.  The inputs depend on the arguments only, so two builds run with the same arguments can be
compared file for file.
"""
import argparse
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)

L_ODD = 1.1
METRIC = "lbfgsb_iterations_per_s"
UNIT = "iterations/s"
QUAD_SEED = 0
QUAD_SCALE = 0.5
DUMP_SAMPLE = 1 << 20   # --dump-outputs: x, g and index at 8 bytes each come to 24 MiB
DUMP_SEED = 2024

# BASELINE.json configs: name -> (n per single-GPU problem, m, numpy dtype name, odd lower bound, default --steps)
WORKLOADS = {
    "rosenbrock": dict(n=100_000_000, m=10, dtype="float64", l_odd=L_ODD, config="configs[2]", steps=20),
    "quadratic": dict(n=125_000_000, m=10, dtype="float64", l_odd=None, config="configs[3]", steps=12),
    "driver3_f32": dict(n=400_000_000, m=20, dtype="float32", l_odd=1.0, config="configs[4]", steps=20),
}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None, help="timed iterations (default: the workload's, see the header)")
    ap.add_argument("--warmup", type=int, default=14, help="untimed iterations (raised to m + 4, see the header)")
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--workload", default="rosenbrock", choices=sorted(WORKLOADS))
    ap.add_argument("--scaling", default="auto", choices=["auto", "strong", "weak"],
                    help="N > 1: strong = the workload's n split over the GPUs (default), weak = n per GPU")
    ap.add_argument("--n", type=int, default=None, help="variables (per GPU under weak scaling)")
    ap.add_argument("--m", type=int, default=None)
    ap.add_argument("--cpu-n", type=int, default=10_000_000, help="sample size of the CPU baseline (about 30 s of one core)")
    ap.add_argument("--plain-fg", action="store_true", help="objective kernels without the line-search epilogue")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="headline only (no extra_configs, no parity solve)")
    ap.add_argument("--ref-budget-s", type=float, default=float(os.environ.get("LBFGSB_REF_BUDGET_S", "480")),
                    help="--impl reference: stop timing early when the run has taken this long")
    ap.add_argument("--profile-out", default=None, help="write the per-kernel-family table here (JSON)")
    ap.add_argument("--dump-outputs", default=None, metavar="DIR",
                    help="write x, g (sampled, see the header) and f of the last timed iteration as DIR/<name>.npy")
    a = ap.parse_args()
    wl = WORKLOADS[a.workload]
    if a.steps is None:
        a.steps = wl["steps"]
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the b200 arm")
    if a.n is None:
        a.n = wl["n"]
    if a.m is None:
        a.m = wl["m"]
    if a.scaling == "auto":
        a.scaling = "strong"
    return a


def workload_name(kind, n_global, n_local, m, world, dtype="float64", l_odd=L_ODD):
    real = "real64" if np.dtype(dtype) == np.float64 else "real32"
    tail = "n=%d%s, m=%d, %s" % (n_global, (" (%d per GPU)" % n_local) if world > 1 else "", m, real)
    if kind == "quadratic":
        return ("bound-constrained convex quadratic (A = tridiag(-1, 2+delta_i, -1), hashed delta and b, box [0, %.1f]), "
                % QUAD_SCALE) + tail
    return "bounded extended Rosenbrock (driver1 bounds, odd lower bound %.1f), " % l_odd + tail


def base_config(kind, n_global, n_local, m, world, scaling, dtype="float64", l_odd=L_ODD):
    """The part of `config` that names the workload: identical in the b200 arm and the reference arm."""
    w = np.dtype(dtype).itemsize
    return {"workload": workload_name(kind, n_global, n_local, m, world, dtype, l_odd), "baseline_config": WORKLOADS.get(
                kind, {}).get("config", "configs[2]"), "n": n_global, "n_per_gpu": n_local, "m": m, "scaling": scaling,
            "factr": 0.0, "pgtol": 0.0,
            "l2": ("working set (%.1f GB per GPU) is far larger than the 126 MB L2; no flush needed" if (2 * m + 9) * n_local * w > 1e9
                   else "working set (%.3f GB per GPU) fits the 126 MB L2: no flush, L2-resident by design at this n") % (
                (2 * m + 9) * n_local * w / 1e9)}


def host_problem(kind, n, l_odd=L_ODD):
    """(x, l, u, nbd, fg) on the host for the CPU arm."""
    import harness as H
    from oracle import oracle_py as O
    if kind == "quadratic":
        from lbfgsb_b200 import sharded
        x, l, u, nbd = sharded.quadratic_problem(n, np.float64, QUAD_SCALE)

        def fg(xx, gg):
            f, g2 = sharded.quadratic_shard_numpy(xx, 0, QUAD_SEED, 0.0, 0.0)
            gg[:] = g2
            return f
        return x, l, u, nbd, fg
    x, l, u, nbd = H.rosenbrock_problem(n, l_odd=l_odd)
    return x, l, u, nbd, O.rosenbrock_fg


def effective_warmup(W, m):
    return max(int(W), int(m) + 4)


def is_burst(nseg, nenter, nleave, n_global):
    return nseg > 1 or (nenter + nleave) > n_global // 100


def dump_index(n_global, size=None):
    """Global indices of the variables --dump-outputs writes (default size DUMP_SAMPLE): all of them up to `size`, else
    one in each of `size` equal stretches, at a position given by the splitmix64 hash of the stretch number and
    DUMP_SEED.  Sorted, and the same in every run, on every rank and with every numpy version (no random stream)."""
    size = DUMP_SAMPLE if size is None else int(size)
    if n_global <= size:
        return np.arange(n_global, dtype=np.int64)
    k = np.arange(size + 1, dtype=np.int64)
    edge = k * n_global // size
    z = (k[:-1] + DUMP_SEED + 1).astype(np.uint64) * np.uint64(0x9E3779B97F4A7C15)   # integer ops wrap mod 2^64
    z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
    z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
    z ^= z >> np.uint64(31)
    return edge[:-1] + (z % np.diff(edge).astype(np.uint64)).astype(np.int64)


def shard_positions(idx, lo, hi):
    """(positions in idx, local indices) of the global indices idx that lie in the shard [lo, hi)."""
    mine = (idx >= lo) & (idx < hi)
    return np.flatnonzero(mine), idx[mine] - lo


def write_outputs(path, outputs):
    """outputs: name -> float32 / float64 array, written as path/<name>.npy."""
    os.makedirs(path, exist_ok=True)
    for name, v in outputs.items():
        assert v.dtype in (np.float32, np.float64), (name, v.dtype)
        np.save(os.path.join(path, name + ".npy"), v)


# ---------------------------------------------------------------------------------------------
# CPU arm: the oracle port (test infrastructure used here only as the measured baseline)
# ---------------------------------------------------------------------------------------------
def cpu_run(n, m, warmup, steps, kind="rosenbrock", budget_s=None, l_odd=L_ODD):
    """Same warm-up rule as the GPU arm.  Returns dict(spi = seconds per iteration inside setulb over all timed
    iterations, k, warmup_effective, steady/burst split, wall)."""
    import harness as H
    from oracle import oracle_py as O
    t_start = time.perf_counter()
    x, l, u, nbd, fg = host_problem(kind, n, l_odd)
    s = O.OracleSetulb()
    g = np.zeros(n)
    f = np.zeros(1)
    wa, iwa = s.workspace(n, m)
    task = H.make_task("START")
    csave = H.make_task("")
    lsave = np.zeros(4, np.int32)
    isave = np.zeros(44, np.int32)
    dsave = np.zeros(29)
    W0 = effective_warmup(warmup, m)
    t_in = 0.0
    t_mark = None      # t_in at the end of the warm-up
    t_last = 0.0
    w_eff = None
    rows = []
    while True:
        ts = H.task_str(task)
        if not (ts[:2] == "FG" or ts == "NEW_X" or ts == "START"):
            break
        a = time.perf_counter()
        s(n, m, x, l, u, nbd, f, g, 0.0, 0.0, wa, iwa, task, -1, csave, lsave, isave, dsave)
        t_in += time.perf_counter() - a
        ts = H.task_str(task)
        if ts[:2] == "FG":
            f[0] = fg(x, g)
        elif ts[:5] == "NEW_X":
            it = int(isave[29])
            ne, nl, nseg = int(isave[40]), int(n + 1 - isave[39]), int(isave[32])
            if t_mark is None:
                if it >= W0 and (not is_burst(1, ne, nl, n) or it >= W0 + 10):
                    t_mark, w_eff, t_last = t_in, it, t_in
            else:
                rows.append((t_in - t_last, is_burst(nseg, ne, nl, n)))
                t_last = t_in
                if len(rows) >= steps:
                    break
                if budget_s is not None and time.perf_counter() - t_start > budget_s and len(rows) >= 5:
                    break
    if t_mark is None or not rows:
        raise RuntimeError("CPU baseline ended before the timed region: " + H.task_str(task))
    k = len(rows)
    st = [r[0] for r in rows if not r[1]]
    bu = [r[0] for r in rows if r[1]]
    return {"spi": (t_in - t_mark) / k, "k": k, "warmup_effective": w_eff,
            "steady": {"iterations": len(st), "s_per_step": (sum(st) / len(st)) if st else None},
            "burst": {"iterations": len(bu), "s_per_step": (sum(bu) / len(bu)) if bu else None},
            "wall_s": time.perf_counter() - t_start}


def reference_arm(a):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    world = max(1, a.gpus)
    wl = WORKLOADS[a.workload]
    if a.workload == "driver3_f32":
        raise SystemExit("--impl reference: the REAL32 workload is timed by the b200 arm's cpu_baseline only")
    strong = a.scaling == "strong" or world == 1
    n_global = a.n if strong else a.n * world
    n_local = -(-n_global // world)
    cfg = base_config(a.workload, n_global, n_local, a.m, world, a.scaling if world > 1 else "single", l_odd=wl["l_odd"] or L_ODD)
    full = world == 1
    n_run = n_global if full else a.cpu_n
    r = cpu_run(n_run, a.m, a.warmup, a.steps, a.workload, budget_s=a.ref_budget_s, l_odd=wl["l_odd"] or L_ODD)
    spi = r["spi"] * (n_global / n_run)
    v = 1.0 / spi
    sample = ("CPU oracle port of src/lbfgsb.f90 (g++ -O3 -funroll-loops, serial like the reference; no Fortran compiler in "
              "the image), time inside setulb only (f/g excluded), %s, %d timed iterations after %d warm-up (%.0f s wall)" % (
                  ("the full n=%d" % n_global) if full else
                  ("n=%d sample of the same problem, scaled linearly to n=%d (N > 1: bounded sample)" % (n_run, n_global)),
                  r["k"], r["warmup_effective"], r["wall_s"]))
    out = {
        "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": a.gpus, "steps": r["k"],
        "warmup": a.warmup, "warmup_effective": r["warmup_effective"], "ms_per_step": spi * 1e3, "higher_is_better": True,
        "scaling": "strong" if strong else "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": cfg,
        "run": {"measured_n": n_run, "full_n": full, "steady": r["steady"], "burst": r["burst"], "host_cores": os.cpu_count()},
        "cpu_baseline": {"value": v, "unit": UNIT, "cores": 1, "kind": "port", "sample": sample},
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(out))


# ---------------------------------------------------------------------------------------------
# clocks
# ---------------------------------------------------------------------------------------------
class ClockSampler(threading.Thread):
    def __init__(self, index):
        super().__init__(daemon=True)
        self.index = index
        self.samples = []
        self.reasons = set()
        self.max_mhz = None
        self.stop_flag = False
        self.ok = False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception:  # noqa: BLE001
            self.nv = None

    def run(self):
        if not self.ok:
            return
        nv = self.nv
        names = {
            getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8): "hw_slowdown",
            getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4): "sw_power_cap",
        }
        while not self.stop_flag:
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:  # noqa: BLE001
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, nm in names.items():
                    if r & bit:
                        self.reasons.add(nm)
            except Exception:  # noqa: BLE001
                pass
            time.sleep(0.01)

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": 0}
        return {"sm_mhz": float(np.median(self.samples)), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.samples)}


# ---------------------------------------------------------------------------------------------
# algorithmic bytes per launch of each kernel family (DESIGN.md "Kernels"): every distinct input
# element read once, every output written once, w = bytes per real, ints 4, state byte 1.
# ---------------------------------------------------------------------------------------------
def family_bytes(n, col, nfree, nmv, w=8):
    upd = n * (3 * w + 2 * w) + 2 * (col - 1) * w * n
    cls = n * (4 * w + 8) + n * (2 * w + 4) + 2 * col * w * nmv
    fgram = n * 1 + 2 * col * w * n
    cwv = n + nfree * 4 * w + 2 * col * w * nfree
    return {
        # fused passes: the algorithmic bytes of the two routines they replace (each routine's own inputs
        # and outputs once, SURVEY.md section 8(a)); the fusion reads the shared streams only once
        "update_classify": upd + cls,
        "subsm_lsinit": n * (1 + 3 * w + w) + nfree * (4 * w + 4 + w) + 2 * col * w * nfree + n * (3 * w + 3 * w + 2 * w + 4),
        "formk_cmprlb": fgram + cwv,
        "ls_trial": n * (5 * w + 4),                                   # gd (2w) + projgr (4w+4) sharing g
        "update": upd,                                                 # g,r,d in; s,y out; col-1 older pairs
        "cauchy_classify": cls,
        "gcp_freev": n * (3 * w + 4 + 2),
        "formk_gram": fgram,
        "cmprlb_wv": cwv,
        "subsm_step": n * (1 + 3 * w + w) + nfree * (4 * w + 4 + w) + 2 * col * w * nfree,
        "ls_init": n * (3 * w + 3 * w + 2 * w + 4),
        "ls_step": n * 2 * w,
        "projgr": n * (4 * w + 4),
    }


def canonical_bytes_per_iteration(n, col, nfree, nmv, nb, w=8):
    """SURVEY.md section 8(a): n(35w+40) + nf(12w+20) + nb(w+4) + 2col*w*(2n + nmv + 3nf)."""
    return n * (35 * w + 40) + nfree * (12 * w + 20) + nb * (w + 4) + 2 * col * w * (2 * n + nmv + 3 * nfree)


def load_peaks():
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:  # noqa: BLE001
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    src = "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback 6650 GB/s (B200_PROFILING.md)"
    return peak, src


def ncu_traffic(family, n, dtype, m):
    """DRAM bytes per launch of a kernel family from the committed ncu capture (profiles/ncu_traffic.json); entries are
    keyed `family` (real64, m <= 10) or `family@f32m20`; None when no capture at this n exists."""
    try:
        tj = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json")))
    except Exception:  # noqa: BLE001
        return None
    key = family if np.dtype(dtype) == np.float64 else "%s@f32m%d" % (family, 20 if m > 10 else (10 if m > 5 else 5))
    ent = tj.get(key)
    if ent and int(ent.get("n", 0)) == n:
        return ent["dram_bytes_per_launch"]
    return None


# ---------------------------------------------------------------------------------------------
# one workload on the device(s)
# ---------------------------------------------------------------------------------------------
class Ctx:
    """torch / distributed context of this process."""

    def __init__(self):
        import torch
        import torch.distributed as dist
        self.torch, self.dist = torch, dist
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        if not torch.cuda.is_available():
            raise SystemExit("bench.py needs a CUDA device (lbfgsb_b200 has no CPU path)")
        torch.cuda.set_device(self.local)
        self.dev = torch.device("cuda", self.local)
        if self.world > 1:
            dist.init_process_group("nccl", device_id=self.dev)
        # the engine works on this stream (never the null stream: 0 would make the engine create a private one)
        self.stream = torch.cuda.Stream(device=self.dev)
        self.comm = None
        if self.world > 1:
            from lbfgsb_b200 import sharded
            self.comm = sharded.nccl_comm_for_engine(self.rank, self.world, dist, self.dev)

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max_over_ranks(self, v):
        if self.world == 1:
            return float(v)
        t = self.torch.tensor([float(v)], dtype=self.torch.float64, device=self.dev)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t)


class DeviceSolve:
    """Problem data, workspace and objective of one workload on this rank's GPU."""

    def __init__(self, cx, kind, n_global, m, dtype, l_odd, plain_fg=False, sharded_run=None):
        import lbfgsb_b200
        from lbfgsb_b200 import sharded
        torch = cx.torch
        self.cx, self.kind, self.m = cx, kind, m
        self.dtype = np.dtype(dtype)
        tdt = torch.float64 if self.dtype == np.float64 else torch.float32
        world = cx.world if sharded_run is None else (cx.world if sharded_run else 1)
        rank = cx.rank if world > 1 else 0
        self.world, self.rank = world, rank
        lo, hi = sharded.shard_bounds(n_global, rank, world)
        n = hi - lo
        self.n, self.n_global, self.off = n, n_global, lo
        dev = cx.dev
        quad = kind == "quadratic"
        if quad:
            self.x = torch.full((n,), 0.5 * QUAD_SCALE, dtype=tdt, device=dev)
            self.l = torch.zeros(n, dtype=tdt, device=dev)
            self.u = torch.full((n,), QUAD_SCALE, dtype=tdt, device=dev)
        else:
            self.x = torch.full((n,), 3.0, dtype=tdt, device=dev)
            self.l = torch.full((n,), -100.0, dtype=tdt, device=dev)
            self.l[(lo % 2)::2] = l_odd          # odd 1-based variables are the even 0-based global indices
            self.u = torch.full((n,), 100.0, dtype=tdt, device=dev)
        self.nbd = torch.full((n,), 2, dtype=torch.int32, device=dev)
        self.g = torch.zeros_like(self.x)
        torch.cuda.synchronize()
        st = cx.stream.cuda_stream
        shard = (lo, n_global, cx.comm, rank, world) if world > 1 else None
        self.prob = lbfgsb_b200.DeviceProblem(n, m, self.dtype, stream=st, shard=shard)
        self.nfg = 0
        # The objective kernels run with their line-search epilogue (gd = g.d and max |proj g| formed while the gradient
        # is in registers; include/lbfgsb_b200.h "Objective with line-search epilogue") unless --plain-fg asks for the
        # plain ones.  The epilogue exists for real64.
        f64 = self.dtype == np.float64
        self.epilogue = f64 and not plain_fg
        epi = (self.l, self.u, self.nbd) if self.epilogue else (None, None, None)
        prob = self.prob
        if quad:
            fgk = lbfgsb_b200.QuadraticDevice(self.dtype, seed=QUAD_SEED, stream=st)
            if world > 1:
                fsh = sharded.ShardedQuadraticDevice(fgk, lo, rank, world, cx.dist, dev, engine=prob)
                fsh.bounds = epi if self.epilogue else None
                self._fg = lambda: fsh(self.x, self.g)
            elif f64:
                self._fg = lambda: prob.fused_fg(1, self.x, self.g, *epi, seed=QUAD_SEED)
            else:
                self._fg = lambda: fgk(self.x, self.g, offset=0)
        else:
            fgk = lbfgsb_b200.RosenbrockDevice(self.dtype, stream=st)
            if world > 1:
                fsh = sharded.ShardedRosenbrockDevice(fgk, rank, world, cx.dist, dev, engine=prob)
                fsh.bounds = epi if self.epilogue else None
                self._fg = lambda: fsh(self.x, self.g)
            elif f64:
                self._fg = lambda: prob.fused_fg(0, self.x, self.g, *epi)
            else:
                self._fg = lambda: fgk(self.x, self.g)
        self._keep = fgk

    def step_to(self, target_iter, factr=0.0, pgtol=0.0, on_newx=None):
        """Run until NEW_X with iter >= target_iter.  False when the solve ended first."""
        p = self.prob
        while True:
            p.setulb_dev(self.x, self.l, self.u, self.nbd, self.g, factr, pgtol)
            t = bytes(p.task[:5])
            if t[:2] == b"FG":
                self.nfg += 1
                p.f[0] = self._fg()
            elif t == b"NEW_X":
                if on_newx is not None:
                    on_newx()
                if p.isave[29] >= target_iter:
                    return True
            else:
                return False

    def counts(self):
        p = self.prob
        return dict(iter=int(p.isave[29]), nseg=int(p.isave[32]), nfree=int(p.isave[37]), nenter=int(p.isave[40]),
                    nleave=int(self.n_global + 1 - p.isave[39]), col=int(p.isave[27]), nfgv=int(p.isave[33]))

    def outputs(self):
        """x and g at dump_index(n_global), f, and the indices (as float64), as the solve stands; every rank of a
        sharded solve returns all of them."""
        torch, dev = self.cx.torch, self.cx.dev
        idx = dump_index(self.n_global)
        dst, src = (torch.from_numpy(a).to(dev) for a in shard_positions(idx, self.off, self.off + self.n))
        out = {}
        for name in ("x", "g"):
            v = getattr(self, name)
            s = torch.zeros(idx.size, dtype=v.dtype, device=dev)
            s[dst] = v[src]
            if self.world > 1:
                self.cx.dist.all_reduce(s)   # each index lies in one shard: the other ranks add zeros
            out[name] = s.cpu().numpy()
        out["f"] = self.prob.f.copy()
        out["index"] = idx.astype(np.float64)
        return out

    def close(self):
        self.prob.close()
        for k in ("x", "l", "u", "nbd", "g"):
            setattr(self, k, None)
        self.cx.torch.cuda.empty_cache()


def measure(cx, kind, n_global, m, dtype, l_odd, W, K, plain_fg=False, sharded_run=None, profile_k=None, want_clocks=True,
            want_outputs=False):
    """Warm-up, K timed iterations (CUDA events per iteration on the engine's stream), per-kernel-family pass.
    Returns the result dict of this workload (rank-independent fields are identical on every rank); with want_outputs,
    its "outputs" are DeviceSolve.outputs() after the last timed iteration."""
    torch = cx.torch
    ds = DeviceSolve(cx, kind, n_global, m, dtype, l_odd, plain_fg, sharded_run)
    prob = ds.prob
    w = ds.dtype.itemsize
    n = ds.n
    out = {}
    with torch.cuda.stream(cx.stream):
        cx.barrier()
        W0 = effective_warmup(W, m)
        if not ds.step_to(W0):
            raise SystemExit("solve ended during warm-up: " + prob.task_str())
        extra = 0
        while extra < 10:
            c = ds.counts()
            if not is_burst(1, c["nenter"], c["nleave"], n_global):
                break
            if not ds.step_to(c["iter"] + 1):
                raise SystemExit("solve ended during warm-up: " + prob.task_str())
            extra += 1
        w_eff = ds.counts()["iter"]
        clocks = ClockSampler(cx.local) if want_clocks else None
        if clocks:
            clocks.start()
        l0, s0 = prob.counters()
        f0 = ds.nfg
        evs = [torch.cuda.Event(enable_timing=True) for _ in range(K + 1)]
        rows = []

        def on_newx():
            evs[len(rows) + 1].record(cx.stream)
            rows.append(ds.counts())
        cx.barrier()
        evs[0].record(cx.stream)
        ok = ds.step_to(w_eff + K, on_newx=on_newx)
        cx.barrier()
        if clocks:
            clocks.stop_flag = True
        if not ok or len(rows) != K:
            raise SystemExit("solve ended inside the timed region after %d of %d steps: %s" % (len(rows), K, prob.task_str()))
        ms = cx.max_over_ranks(evs[0].elapsed_time(evs[K]))
        per = [evs[i].elapsed_time(evs[i + 1]) for i in range(K)]
        l1, s1 = prob.counters()
        if want_outputs:
            out["outputs"] = ds.outputs()
        fg_evals = ds.nfg - f0
        # our kernels per objective evaluation: the objective kernel + its final sum (+ 4 exchange kernels on a shard)
        fg_kernels = 2 if ds.world == 1 else 6
        launches = (l1 - l0) + fg_kernels * fg_evals
        value = K / (ms * 1e-3)
        burst = [is_burst(r["nseg"], r["nenter"], r["nleave"], n_global) for r in rows]
        st_ms = [t for t, b in zip(per, burst) if not b]
        bu_ms = [t for t, b in zip(per, burst) if b]
        cols = [r["col"] for r in rows]
        nfree = rows[-1]["nfree"]
        out.update({
            "value": value, "ms_per_step": ms / K, "steps": K, "warmup_effective": w_eff,
            "steady": {"iterations": len(st_ms), "ms_per_step": (sum(st_ms) / len(st_ms)) if st_ms else None,
                       "value": (1e3 * len(st_ms) / sum(st_ms)) if st_ms else None},
            "burst": {"iterations": len(bu_ms), "ms_per_step": (sum(bu_ms) / len(bu_ms)) if bu_ms else None,
                      "rule": "nseg > 1 or nenter + nleave > n/100"},
            "col_min_in_timed_region": min(cols), "col_max_in_timed_region": max(cols), "nfree": int(nfree),
            "nseg_max_in_timed_region": max(r["nseg"] for r in rows),
            "fg_evals_per_step": fg_evals / K, "gpu_launches": int(launches), "host_syncs_per_step": (s1 - s0) / K,
            "launches_per_step": launches / K,
        })
        if clocks:
            clocks.join(timeout=1.0)
            out["clocks"] = clocks.summary()

        # ---- per-kernel-family pass (CUDA events around every kernel, on the same stream) ----
        PK = profile_k if profile_k is not None else max(4, min(K, 8))
        col = rows[-1]["col"]
        prob.profile(True)
        prob.profile_reset()
        okp = ds.step_to(w_eff + K + PK)
        prof = prob.profile_read() if okp else {}
        prob.profile(False)
        peak, peak_src = load_peaks()
        fam_table, roof = {}, None
        if prof:
            st_free = nfree
            if ds.world > 1:           # local counts for the byte formulas (this rank's shard)
                st_free = int((prob.vector(7) <= 0).sum())
            fb = family_bytes(n, col, st_free, st_free, w)
            # passes that the engine folded into a neighbour in this run (their own launches did not happen or returned
            # at once): the neighbour is credited with the routine's algorithmic bytes
            if prof.get("gcp_freev", {"calls": 0})["calls"] == 0 or prof["gcp_freev"]["ms"] / max(prof["gcp_freev"]["calls"], 1) < 0.02:
                fb["formk_cmprlb"] += fb["gcp_freev"]      # cauchy's tail + freev inside k_formk_cmprlb (fuse_gf)
            fb["subsm_lsinit"] += fb["ls_step"]            # the stp = 1 trial point x = z is written by the subspace pass
            total_ms = sum(v["ms"] for v in prof.values())
            for name, v in prof.items():
                if v["calls"] == 0 or v["ms"] <= 0:
                    continue
                row = {"calls": int(v["calls"]), "ms_per_call": v["ms"] / v["calls"], "share": v["ms"] / total_ms}
                if name in fb:
                    gbs = fb[name] / (row["ms_per_call"] * 1e-3) / 1e9
                    if gbs > 2.5 * peak:
                        # launches that returned at once (the pass was folded into a fused kernel or its flag was off)
                        continue
                    row["bytes_per_call"] = fb[name]
                    row["gbs"] = gbs
                fam_table[name] = row
            cand = {k: v for k, v in fam_table.items() if "gbs" in v}
            if cand:
                top = max(cand, key=lambda k: cand[k]["share"])
                roof = {"bound": "hbm", "kernel": top, "achieved": cand[top]["gbs"], "peak": peak, "unit": "GB/s",
                        "frac": cand[top]["gbs"] / peak, "traffic": ncu_traffic(top, n, ds.dtype, m), "peak_source": peak_src,
                        "share_of_step": cand[top]["share"], "ms_per_launch": cand[top]["ms_per_call"],
                        "algorithmic_bytes_per_launch": cand[top]["bytes_per_call"]}
            # real DRAM traffic per iteration from the committed ncu captures (where one exists at this n)
            real = 0.0
            known = True
            for name, v in fam_table.items():
                if "gbs" not in v:
                    continue
                t = ncu_traffic(name, n, ds.dtype, m)
                if t is None:
                    known = False
                    break
                real += t * v["calls"] / PK
            if known and real > 0:
                fgb = 2 * w * n * out["fg_evals_per_step"] * (2.75 if ds.epilogue else 1.0)   # x in, g out (+ d, l, u, nbd)
                out["real_traffic_bytes_per_iteration"] = real + fgb
        nf_local = nfree // ds.world
        canon = canonical_bytes_per_iteration(n, col, nf_local, nf_local, 0, w)
        step_ms = out["steady"]["ms_per_step"] or out["ms_per_step"]
        iter_gbs = canon / (step_ms * 1e-3) / 1e9
        it_roof = {"canonical_bytes_per_iteration_per_gpu": canon, "canonical_gbs_per_gpu": iter_gbs,
                   "canonical_frac_of_peak": iter_gbs / peak, "peak": peak, "peak_source": peak_src,
                   "over": "steady iterations" if out["steady"]["ms_per_step"] else "all timed iterations",
                   "note": "the canonical numerator (SURVEY.md 8a) counts every routine's streams separately; fused passes "
                           "read shared streams once, so canonical_frac_of_peak can exceed 1 -- real_traffic_frac is the "
                           "physical fraction"}
        if "real_traffic_bytes_per_iteration" in out:
            rt = out.pop("real_traffic_bytes_per_iteration")
            it_roof["real_traffic_bytes_per_iteration_per_gpu"] = rt
            it_roof["real_traffic_gbs_per_gpu"] = rt / (step_ms * 1e-3) / 1e9
            it_roof["real_traffic_frac"] = it_roof["real_traffic_gbs_per_gpu"] / peak
        out["iteration_roofline"] = it_roof
        out["aggregate"] = {"variable_iterations_per_s": n_global * value,
                            "canonical_gbs_all_gpus": canon * ds.world * value / 1e9}
        if roof:
            out["roofline"] = roof
        if fam_table:
            out["kernel_families"] = fam_table
        out["task_after_profile_pass"] = prob.task_str()
        out["rank_exchange"] = {0: "none (single GPU)", 1: "ncclAllGather of the reduction records",
                                2: "reduction records stored into the peers' memory over NVLink (CUDA IPC), flags polled by "
                                   "the consuming kernel"}.get(prob.exchange_mode(), "?")
        out["fg"] = "device kernel, inside the timed region" + (
            "; it also forms the line-search sums g.d and max |proj g| (lbfgsb_problem_fused_f64), so the engine's own pass "
            "for them (k_ls_trial) is not launched" if ds.epilogue else "")
    ds.close()
    return out


def solve_to_convergence(cx, n, m, l_odd, factr, pgtol):
    """BASELINE.json configs[1]: the driver1 problem at n = 1e6, m = 5 solved to the reference's stopping test."""
    torch = cx.torch
    ds = DeviceSolve(cx, "rosenbrock", n, m, np.float64, l_odd, False, sharded_run=False)
    with torch.cuda.stream(cx.stream):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        ds.step_to(10 ** 9, factr=factr, pgtol=pgtol)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
    c = ds.counts()
    l, s = ds.prob.counters()
    out = {"workload": workload_name("rosenbrock", n, n, m, 1, "float64", l_odd), "baseline_config": "configs[1]",
           "factr": factr, "pgtol": pgtol, "iterations": c["iter"], "fg_evals": c["nfgv"], "task": ds.prob.task_str(),
           "f": float(ds.prob.f[0]), "seconds_to_solution": dt, "value": c["iter"] / dt, "unit": UNIT,
           "launches_per_iteration": l / max(c["iter"], 1), "host_syncs_per_iteration": s / max(c["iter"], 1)}
    ds.close()
    return out


def batched_rate(nprob=1000, n=25, m=5):
    """SURVEY.md section 8 f4: nprob copies of test/driver1.f90 (perturbed starting points) solved to the reference's
    stopping test by lbfgsb_batch_setulb_dev_f64, one CTA per problem; next to the CPU oracle on a 200-problem sample."""
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import batch_rate as BR
    g = BR.gpu_rate(nprob, n, m)
    c = BR.cpu_rate(200, n, m)
    return {"workload": "%d x driver1 (n=%d, m=%d, factr=1e7, pgtol=1e-5), perturbed x0" % (nprob, n, m), "baseline_config": "configs[0]",
            "metric": "problems_per_s", "value": g["problems_per_s"], "unit": "problems/s", "iterations_per_s": g["iterations_per_s"],
            "seconds": g["seconds"], "calls": g["calls"], "converged": g["converged"], "gpu_launches": 2 * g["calls"],
            "cpu_baseline": {"value": c["problems_per_s"], "unit": "problems/s", "cores": 1, "kind": "port",
                             "sample": "CPU oracle port, 200 of the problems one after the other through its driver loop"}}


def small_n_latency():
    """Where the fixed cost per setulb call decides the rate: ms per iteration, launches and host read-backs per iteration
    through the caller's loop (lbfgsb_setulb_dev_f64, objective with the line-search epilogue) and through the
    device-resident loop (lbfgsb_minimize_graph_dev_f64: one CUDA-graph launch and one read-back per step)."""
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import small_n_latency as SL
    out = []
    for n in (1000, 100000):
        out.append(SL.run(n, 10))
        out.append(SL.run_graph(n, 10))
    return out


def parity_check(cx, n_global=200_000, m=5, l_odd=1.0, iters=30):
    """N > 1: the sample problem sharded over the ranks and, on rank 0, on one GPU -- discrete trace and active-set hash
    equal at every iterate, f within 1e-10 (first 10 iterates) / 1e-6 (the logic of tests/mgpu_check.py)."""
    import mgpu_check as MC
    import lbfgsb_b200
    from lbfgsb_b200 import sharded
    torch, dist = cx.torch, cx.dist
    lo, hi = sharded.shard_bounds(n_global, cx.rank, cx.world)
    kern = lbfgsb_b200.RosenbrockDevice(np.float64)
    rows, task, _, _ = MC.solve(hi - lo, lo, n_global, m, l_odd, iters, (lo, n_global, cx.comm, cx.rank, cx.world),
                             lambda: sharded.ShardedRosenbrockDevice(kern, cx.rank, cx.world, dist, cx.dev), cx.dev,
                             cx.rank, cx.world, "rosenbrock")
    res = None
    if cx.rank == 0:
        ref, rtask, _, _ = MC.solve(n_global, 0, n_global, m, l_odd, iters, None, lambda: kern, cx.dev, 0, 1, "rosenbrock")
        ok, msg, worst = MC.compare(rows, task, ref, rtask)
        res = {"status": "ok" if ok else "FAIL", "n": n_global, "m": m, "iterates_compared": len(ref),
               "fields": "iter nfgv nseg nfree nact iword iback nenter col active-set-hash", "worst_rel_f": worst,
               "walks_nseg_gt_1": [r["nseg"] for r in ref if r["nseg"] > 1][:6]}
        if not ok:
            res["detail"] = msg[:400]
    torch.cuda.synchronize()
    return res


def main():
    a = parse()
    if a.impl == "reference":
        reference_arm(a)
        return
    # stdout carries exactly one JSON line: libraries that print there (NCCL's version banner) go to stderr
    sys.stdout.flush()
    saved_stdout = os.dup(1)
    os.dup2(2, 1)
    cx = Ctx()
    world, rank = cx.world, cx.rank
    wl = WORKLOADS[a.workload]
    dtype = wl["dtype"]
    l_odd = wl["l_odd"] if wl["l_odd"] is not None else L_ODD
    strong = (a.scaling == "strong") or world == 1
    n_global = a.n if strong else a.n * world
    n_local = -(-n_global // world)
    W, K = a.warmup, a.steps

    head = measure(cx, a.workload, n_global, a.m, dtype, l_odd, W, K, a.plain_fg, want_outputs=bool(a.dump_outputs))
    outputs = head.pop("outputs", None)
    if outputs is not None and rank == 0:
        write_outputs(a.dump_outputs, outputs)
    cfg = base_config(a.workload, n_global, n_local, a.m, world, ("strong" if strong else "weak") if world > 1 else "single",
                      dtype, l_odd)
    out = {
        "metric": METRIC, "value": head["value"], "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
        "warmup_effective": head["warmup_effective"], "ms_per_step": head["ms_per_step"], "higher_is_better": True,
        "scaling": "strong" if strong else "weak", "vs_baseline": None,
        "dtype": "f64" if np.dtype(dtype) == np.float64 else "f32", "data": "synthetic", "config": cfg,
        "gpu_launches": head["gpu_launches"], "clocks": head.get("clocks"),
    }
    for k in ("roofline", "iteration_roofline", "aggregate", "kernel_families"):
        if k in head:
            out[k] = head[k]
    out["run"] = {k: head[k] for k in ("steady", "burst", "col_min_in_timed_region", "col_max_in_timed_region", "nfree",
                                        "nseg_max_in_timed_region", "fg_evals_per_step", "launches_per_step",
                                        "host_syncs_per_step", "rank_exchange", "fg", "task_after_profile_pass")}
    if a.profile_out and rank == 0:
        with open(a.profile_out, "w") as fh:
            json.dump({"n": n_local, "m": a.m, "families": head.get("kernel_families"), "roofline": head.get("roofline")}, fh, indent=1)

    # ---- the other BASELINE.json configurations, in the same run ----
    extras = {}
    if not a.no_extra and a.workload == "rosenbrock":
        def slim(r, kind, ng, m, dt, lo, scaling):
            nl = -(-ng // world) if scaling != "single" else ng
            d = {"config": base_config(kind, ng, nl, m, world if scaling != "single" else 1, scaling, dt, lo),
                 "metric": METRIC, "unit": UNIT, "dtype": "f64" if np.dtype(dt) == np.float64 else "f32"}
            for k in ("value", "ms_per_step", "steps", "warmup_effective", "steady", "burst", "col_min_in_timed_region", "nfree",
                      "nseg_max_in_timed_region", "fg_evals_per_step", "launches_per_step", "roofline", "iteration_roofline",
                      "aggregate"):
                if k in r:
                    d[k] = r[k]
            return d
        try:
            if world == 1:
                q = WORKLOADS["quadratic"]
                r = measure(cx, "quadratic", q["n"], q["m"], q["dtype"], L_ODD, 12, min(K, 12), a.plain_fg, profile_k=4, want_clocks=False)
                extras["configs[3] quadratic, 1.25e8 per GPU"] = slim(r, "quadratic", q["n"], q["m"], q["dtype"], L_ODD, "single")
                d3 = WORKLOADS["driver3_f32"]
                r = measure(cx, "driver3_f32", d3["n"], d3["m"], d3["dtype"], d3["l_odd"], W, min(K, 12), True, profile_k=4, want_clocks=False)
                extras["configs[4] driver3-style n=4e8, m=20, REAL32"] = slim(r, "driver3_f32", d3["n"], d3["m"], d3["dtype"], d3["l_odd"], "single")
                extras["configs[1] n=1e6, m=5 to convergence"] = solve_to_convergence(cx, 1_000_000, 5, 1.0, 1.0e7, 1.0e-5)
                extras["configs[0] x 1000: batched small problems (one CTA per problem)"] = batched_rate()
                extras["small n: fixed cost per iteration (n=1e3, 1e5; caller loop vs lbfgsb_minimize_graph_dev_f64)"] = small_n_latency()
            else:
                other = "weak" if strong else "strong"
                ng = a.n * world if strong else a.n
                r = measure(cx, "rosenbrock", ng, a.m, dtype, l_odd, W, K, a.plain_fg, profile_k=4, want_clocks=False)
                extras["configs[2] %s series, n=%d" % (other, ng)] = slim(r, "rosenbrock", ng, a.m, dtype, l_odd, other)
                q = WORKLOADS["quadratic"]
                r = measure(cx, "quadratic", q["n"] * world, q["m"], q["dtype"], L_ODD, 12, min(K, 12), a.plain_fg, profile_k=4, want_clocks=False)
                extras["configs[3] quadratic weak series, n=%d" % (q["n"] * world)] = slim(r, "quadratic", q["n"] * world, q["m"], q["dtype"], L_ODD, "weak")
        except SystemExit as e:
            extras["error"] = str(e)
        except Exception as e:  # noqa: BLE001
            extras["error"] = "%s: %s" % (type(e).__name__, e)
    if extras:
        out["extra_configs"] = extras
    if world > 1 and not a.no_extra:
        try:
            out["parity"] = parity_check(cx)
        except Exception as e:  # noqa: BLE001
            out["parity"] = {"status": "error", "detail": "%s: %s" % (type(e).__name__, e)}

    # ---- e2e: HOST buffers ----
    if not a.no_e2e:
        try:
            out["e2e"] = e2e_host(cx, a.workload, n_global, a.m, W, K, l_odd)
        except Exception as e:  # noqa: BLE001
            out["e2e"] = {"value": None, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0,
                          "note": "failed: %s: %s" % (type(e).__name__, e)}
    if cx.comm:
        import lbfgsb_b200
        lbfgsb_b200.lib().lbfgsb_dev_nccl_destroy(cx.comm)
    if rank == 0 and world == 1 and not a.no_cpu and a.workload != "driver3_f32":
        try:
            r = cpu_run(a.cpu_n, a.m, W, min(K, 8), a.workload, l_odd=l_odd)
            v = 1.0 / (r["spi"] * n_global / a.cpu_n)
            out["cpu_baseline"] = {
                "value": v, "unit": UNIT, "cores": 1, "kind": "port",
                "sample": "CPU oracle port of src/lbfgsb.f90 (serial like the reference; no Fortran compiler in the "
                          "image), time inside setulb only, n=%d sample, %d iterations after %d warm-up, scaled "
                          "linearly to n=%d (`bench.py --impl reference` runs the full n); host has %d cores" % (
                              a.cpu_n, r["k"], r["warmup_effective"], n_global, os.cpu_count())}
        except Exception as e:  # noqa: BLE001
            out["cpu_baseline"] = {"value": None, "unit": UNIT, "cores": 1, "kind": "port", "sample": "failed: %s" % e}
    if world > 1:
        cx.dist.destroy_process_group()
    sys.stdout.flush()
    os.dup2(saved_stdout, 1)
    if rank == 0:
        print(json.dumps(out), flush=True)


def e2e_host(cx, kind, n_global, m, W, K, l_odd):
    """The same iterations with HOST x and g.  N = 1: through the C-ABI host twin lbfgsb_setulb_f64 (src/lbfgsb.f90:88-89
    argument for argument).  N > 1: through lbfgsb_b200.sharded.HostShard, the same staging around the sharded device
    variant.  Timed: the setulb calls only (they contain the H2D copy of g and the D2H copy of x); the caller's f/g runs
    on the device from a staged copy of x outside the timed region, as the metric excludes the user's f/g."""
    import harness as H
    import lbfgsb_b200
    from lbfgsb_b200 import sharded
    torch = cx.torch
    world, rank, dev = cx.world, cx.rank, cx.dev
    quad = kind == "quadratic"
    lo, hi = sharded.shard_bounds(n_global, rank, world)
    n = hi - lo
    xh = torch.full((n,), 0.5 * QUAD_SCALE if quad else 3.0, dtype=torch.float64).pin_memory()
    gh = torch.zeros(n, dtype=torch.float64).pin_memory()
    x, g = xh.numpy(), gh.numpy()
    if quad:
        l = np.zeros(n)
        u = np.full(n, QUAD_SCALE)
    else:
        l = np.full(n, -100.0)
        l[(lo % 2)::2] = l_odd
        u = np.full(n, 100.0)
    nbd = np.full(n, 2, np.int32)
    xs = torch.empty(n, dtype=torch.float64, device=dev)
    gs = torch.empty(n, dtype=torch.float64, device=dev)
    st = torch.cuda.current_stream().cuda_stream
    if quad:
        qk = lbfgsb_b200.QuadraticDevice(np.float64, seed=QUAD_SEED, stream=st)
        fg1 = (lambda xx, gg: qk(xx, gg, offset=0))
        fgs = sharded.ShardedQuadraticDevice(qk, lo, rank, world, cx.dist, dev) if world > 1 else None
    else:
        rk = lbfgsb_b200.RosenbrockDevice(np.float64, stream=st)
        fg1 = rk
        fgs = sharded.ShardedRosenbrockDevice(rk, rank, world, cx.dist, dev) if world > 1 else None
    task = H.make_task("START")
    csave = H.make_task("")
    lsave = np.zeros(4, np.int32)
    isave = np.zeros(44, np.int32)
    dsave = np.zeros(29)
    f = np.zeros(1)
    twin = None
    if world > 1:
        twin = sharded.HostShard(n, lo, n_global, m, cx.comm, rank, world)

        def call():
            twin.setulb(x, l, u, nbd, f, g, 0.0, 0.0, task, -1, csave, lsave, isave, dsave)
    else:
        def call():
            lbfgsb_b200.setulb(n, m, x, l, u, nbd, f, g, 0.0, 0.0, None, None, task, -1, csave, lsave, isave, dsave)
    W0 = effective_warmup(W, m)
    t_in, t0, it0, calls, c0 = 0.0, None, None, 0, 0
    try:
        while True:
            if world > 1:
                cx.barrier()   # the ranks enter the call together: the skew of the caller's own f/g staging is not setulb's time
            a = time.perf_counter()
            call()
            t_in += time.perf_counter() - a
            calls += 1
            ts = bytes(task[:5])
            if ts[:2] == b"FG":
                xs.copy_(xh, non_blocking=True)
                f[0] = fg1(xs, gs) if world == 1 else fgs(xs, gs)
                gh.copy_(gs)
                torch.cuda.synchronize()
            elif ts == b"NEW_X":
                it = int(isave[29])
                if it == W0:
                    if world > 1:
                        cx.barrier()
                    t0, it0, c0 = t_in, it, calls
                if it >= W0 + K:
                    break
            else:
                break
        if t0 is None or int(isave[29]) < W0 + K:
            return {"value": None, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0,
                    "note": "host-buffer solve ended early: " + H.task_str(task)}
        k = int(isave[29]) - it0
        ncalls = calls - c0
        sec = cx.max_over_ranks(t_in - t0)
        # per FG re-entry: g host->device; per call that moved x: x device->host (all ranks together)
        h2d = 8 * n_global * (ncalls - k) / k
        d2h = 8 * n_global * (ncalls - k) / k
        copy_ms = (h2d + d2h) / world / 55e9 * 1e3
        return {"value": k / sec, "unit": UNIT, "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                "ms_per_step": sec / k * 1e3, "warmup_effective": W0,
                "api": "lbfgsb_setulb_f64 (C-ABI host twin)" if world == 1 else "lbfgsb_b200.sharded.HostShard (sharded device variant + pinned staging)",
                "note": "time inside the setulb calls with pinned host x, g (copies included); f/g evaluated outside. "
                        "PCIe-bound: about %.1f of the %.1f ms per step are the serialised H2D copy of g and D2H copy of x "
                        "(%.2f GB each way per GPU at ~55 GB/s), inherent to host-resident x and g" % (
                            copy_ms, sec / k * 1e3, h2d / world / 1e9)}
    finally:
        if twin is not None:
            twin.close()
        else:
            lbfgsb_b200.lib().lbfgsb_host_release(isave.ctypes.data_as(__import__("ctypes").c_void_p))


if __name__ == "__main__":
    main()
