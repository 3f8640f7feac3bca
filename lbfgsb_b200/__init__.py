"""lbfgsb_b200 -- host-side mirror of the reference's `setulb` interface over the C ABI.

The product is the CUDA engine in csrc/ behind include/lbfgsb_b200.h.  This module is a thin
ctypes binding that plays the role of the Fortran module `lbfgsb_module`
(/root/reference/src/lbfgsb.f90:46-58): it exports

    setulb(n, m, x, l, u, nbd, f, g, factr, pgtol, wa, iwa, task, iprint, csave, lsave, isave, dsave)
        host arrays (numpy), same argument order and meaning as src/lbfgsb.f90:88-89;
    setulb_dev(handle, x, l, u, nbd, f, g, factr, pgtol, task, iprint, csave, lsave, isave, dsave)
        x, l, u, nbd, g are CUDA tensors (device pointers), the state arrays stay on the host.

There is no CPU path: importing works anywhere (so the symbol table can be checked), every
compute entry point needs a CUDA device and fails loudly without one or without the built
library.
"""
import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_ROOT = os.path.dirname(_HERE)
SO_PATH = os.path.join(_HERE, "liblbfgsb_b200.so")
_SOURCES = ["engine.cu", "common.cuh", "kernels_stream.cuh", "kernels_dense.cuh", "cauchy_walk.cuh", "kernels_tma.cuh",
            "tma_pipe.cuh", "cauchy_walk_dist.cuh", "batch.cuh", "host_print.h"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              # no fused multiply-add: the dense 2m x 2m algebra and dcsrch/dcstep must round like the
              # reference (gfortran x86-64 default has no FMA), see DESIGN.md "Numerics"
              "-fmad=false", "-Xcompiler", "-fPIC", "-shared"]

_LIB = None


class LbfgsbB200Error(RuntimeError):
    pass


def _stale():
    if not os.path.exists(SO_PATH):
        return True
    t = os.path.getmtime(SO_PATH)
    deps = [os.path.join(_HERE, "csrc", s) for s in _SOURCES]
    deps += [os.path.join(_ROOT, "include", h) for h in ("lbfgsb_b200.h", "lbfgsb_b200_shape.h")]
    return any(os.path.exists(p) and os.path.getmtime(p) > t for p in deps)


def build(force=False, verbose=False):
    """Compile csrc/engine.cu for sm_100a into lbfgsb_b200/liblbfgsb_b200.so (in-tree)."""
    if not (force or _stale()):
        return SO_PATH
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    cmd = [nvcc] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + \
          ["-o", SO_PATH, os.path.join(_HERE, "csrc", "engine.cu"), "-ldl"]
    subprocess.check_call(cmd)
    return SO_PATH


_REAL = {np.dtype(np.float64): ("f64", C.c_double), np.dtype(np.float32): ("f32", C.c_float)}


def lib():
    """The loaded C-ABI library.  Raises if it has not been built (no fallback of any kind)."""
    global _LIB
    if _LIB is None:
        if not os.path.exists(SO_PATH):
            raise LbfgsbB200Error(
                "lbfgsb_b200: %s is missing -- run `python -c 'import __graft_entry__ as g; g.build()'` "
                "(there is no CPU path)" % SO_PATH)
        L = C.CDLL(SO_PATH)
        L.lbfgsb_b200_last_error.restype = C.c_char_p
        L.lbfgsb_dev_create.restype = C.c_void_p
        L.lbfgsb_dev_create.argtypes = [C.c_int64, C.c_int32, C.c_int32, C.c_void_p]
        L.lbfgsb_dev_create_sharded.restype = C.c_void_p
        L.lbfgsb_dev_create_sharded.argtypes = [C.c_int64, C.c_int64, C.c_int64, C.c_int32, C.c_int32,
                                                C.c_void_p, C.c_void_p, C.c_int32, C.c_int32]
        L.lbfgsb_dev_destroy.argtypes = [C.c_void_p]
        L.lbfgsb_dev_set_iteration_file.argtypes = [C.c_void_p, C.c_char_p]
        L.lbfgsb_dev_checkpoint_write.argtypes = [C.c_void_p, C.c_char_p]
        L.lbfgsb_dev_checkpoint_read.argtypes = [C.c_void_p, C.c_char_p]
        L.lbfgsb_host_engine.restype = C.c_void_p
        L.lbfgsb_host_engine.argtypes = [C.c_void_p]
        L.lbfgsb_dev_vector.restype = C.c_void_p
        L.lbfgsb_dev_vector.argtypes = [C.c_void_p, C.c_int32]
        L.lbfgsb_dev_vector_copy.argtypes = [C.c_void_p, C.c_int32, C.c_void_p, C.c_int64]
        L.lbfgsb_dev_active_set_hash.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
        L.lbfgsb_dev_counters.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
        L.lbfgsb_dev_graph_stats.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
        L.lbfgsb_problem_rosenbrock_halo_f64.argtypes = [C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32,
                                                         C.c_void_p, C.c_void_p]
        L.lbfgsb_problem_quadratic_halo_f64.argtypes = [C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_uint64,
                                                        C.c_void_p, C.c_void_p]
        L.lbfgsb_dev_profile.argtypes = [C.c_void_p, C.c_int32]
        L.lbfgsb_dev_profile_reset.argtypes = [C.c_void_p]
        L.lbfgsb_dev_set_tie_limit.argtypes = [C.c_void_p, C.c_int64]
        L.lbfgsb_dev_set_tie_limit.restype = None
        L.lbfgsb_dev_tie_stats.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
        L.lbfgsb_dev_profile_read.argtypes = [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        L.lbfgsb_dev_nccl_init.restype = C.c_void_p
        L.lbfgsb_dev_nccl_init.argtypes = [C.c_void_p, C.c_int32, C.c_int32]
        L.lbfgsb_dev_nccl_destroy.argtypes = [C.c_void_p]
        L.lbfgsb_problem_scratch_bytes.restype = C.c_int64
        for sfx, cr in (("f64", C.c_double), ("f32", C.c_float)):
            getattr(L, "lbfgsb_setulb_" + sfx).restype = None
            getattr(L, "lbfgsb_setulb_dev_" + sfx).restype = None
            getattr(L, "lbfgsb_problem_rosenbrock_" + sfx).argtypes = [
                C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, cr, cr, C.c_void_p]
            getattr(L, "lbfgsb_problem_quadratic_" + sfx).argtypes = [
                C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_uint64, cr, cr, C.c_void_p]
        L.lbfgsb_problem_rosenbrock_halo_f64.argtypes = [C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32,
                                                         C.c_int32, C.c_void_p, C.c_void_p]
        L.lbfgsb_problem_quadratic_halo_f64.argtypes = [C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64,
                                                        C.c_uint64, C.c_void_p, C.c_void_p]
        for nm in ("lbfgsb_problem_fused_f64", "lbfgsb_problem_sharded_f64"):
            getattr(L, nm).argtypes = [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                       C.c_void_p, C.c_uint64]
        L.lbfgsb_dev_exchange_mode.argtypes = [C.c_void_p]
        L.lbfgsb_batch_create.restype = C.c_void_p
        L.lbfgsb_batch_create.argtypes = [C.c_int32, C.c_int64, C.c_int32, C.c_int32, C.c_void_p]
        L.lbfgsb_batch_destroy.argtypes = [C.c_void_p]
        L.lbfgsb_batch_counts.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        L.lbfgsb_batch_stream.restype = C.c_void_p
        L.lbfgsb_batch_stream.argtypes = [C.c_void_p]
        L.lbfgsb_batch_get_iwhere.restype = C.c_int
        L.lbfgsb_batch_get_iwhere.argtypes = [C.c_void_p, C.c_void_p]
        L.lbfgsb_batch_fg_mask.restype = C.c_void_p
        L.lbfgsb_batch_fg_mask.argtypes = [C.c_void_p]
        L.lbfgsb_batch_vector_copy.argtypes = [C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_int64]
        for sfx in ("f64", "f32"):
            getattr(L, "lbfgsb_batch_setulb_dev_" + sfx).restype = None
            getattr(L, "lbfgsb_batch_setulb_dev_" + sfx).argtypes = [C.c_void_p] * 14
            getattr(L, "lbfgsb_problem_rosenbrock_batch_" + sfx).argtypes = [C.c_int32, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p,
                                                                             C.c_void_p, C.c_void_p]
        _LIB = L
    return _LIB


def last_error():
    return lib().lbfgsb_b200_last_error().decode()


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def _check_task(task):
    s = bytes(task[:60]).decode(errors="replace")
    if s.startswith(("ERROR: CUDA", "ERROR: NO CUDA", "ERROR: INVALID LBFGSB", "ERROR: DEVICE POINTERS", "ERROR: SETULB CALLED")):
        raise LbfgsbB200Error(s.rstrip() + " -- " + last_error())


def setulb(n, m, x, l, u, nbd, f, g, factr, pgtol, wa, iwa, task, iprint, csave, lsave, isave, dsave,
           iteration_file=None):
    """Host twin of the reference's setulb (src/lbfgsb.f90:88-89); numpy arrays, updated in place.

    f is a 1-element array of x's dtype; task/csave are 60-byte uint8 arrays (blank padded);
    lsave int32[4]; isave int32[44]; dsave real[29].  wa / iwa are accepted for signature
    compatibility (the workspace lives on the device)."""
    sfx, cr = _REAL[x.dtype]
    fn = getattr(lib(), "lbfgsb_setulb_" + sfx)
    n32, m32, ip = C.c_int32(n), C.c_int32(m), C.c_int32(iprint)
    fa, pg = cr(factr), cr(pgtol)
    itf = iteration_file.encode() if iteration_file else None
    fn(C.byref(n32), C.byref(m32), _p(x), _p(l), _p(u), _p(nbd), _p(f), _p(g), C.byref(fa), C.byref(pg),
       _p(wa) if wa is not None else None, _p(iwa) if iwa is not None else None, _p(task), C.byref(ip),
       _p(csave), _p(lsave), _p(isave), _p(dsave), itf, C.c_int32(len(itf) if itf else 0))
    _check_task(task)


class HostSetulb:
    """Callable with the calling convention of tests/harness.py (same as oracle_py.OracleSetulb)."""

    def __init__(self, dtype=np.float64, iteration_file=None):
        self.dtype = np.dtype(dtype)
        self._isave = None
        self.iteration_file = iteration_file    # setulb's optional argument (src/lbfgsb.f90:243)

    def workspace(self, n, m):
        # the reference's sizes (src/lbfgsb.f90:146-148) are not needed: the state is on the device
        return np.zeros(1, dtype=self.dtype), np.zeros(1, dtype=np.int32)

    def __call__(self, n, m, x, l, u, nbd, f, g, factr, pgtol, wa, iwa, task, iprint, csave, lsave, isave, dsave):
        self._isave = isave
        setulb(n, m, x, l, u, nbd, f, g, factr, pgtol, wa, iwa, task, iprint, csave, lsave, isave, dsave,
               iteration_file=self.iteration_file)

    def engine(self):
        return lib().lbfgsb_host_engine(_p(self._isave))

    def active_set_hash(self, n, iwa):
        h, c = C.c_uint64(0), C.c_int64(0)
        e = self.engine()
        if not e:
            return None, None
        if lib().lbfgsb_dev_active_set_hash(e, C.byref(h), C.byref(c)) != 0:
            raise LbfgsbB200Error(last_error())
        return h.value, c.value

    def previous_x(self, n):
        t = np.zeros(n, dtype=self.dtype)
        fn = lib().lbfgsb_host_previous_x_f64 if self.dtype == np.float64 else lib().lbfgsb_host_previous_x_f32
        if fn(_p(self._isave), _p(t)) != 0:
            raise LbfgsbB200Error("no live problem bound to this isave")
        return t

    def release(self, isave):
        lib().lbfgsb_host_release(_p(isave))


class DeviceProblem:
    """Device-pointer variant (include/lbfgsb_b200.h section 2): the caller's x, g, l, u, nbd are CUDA
    tensors; f/g evaluation and the whole iteration stay on the GPU.  `stream` is a raw cudaStream_t
    (int) or None for the engine's private stream."""

    def __init__(self, n, m, dtype, stream=None, shard=None, iprint=-1, iteration_file=None):
        import torch
        self.torch = torch
        self.n, self.m = int(n), int(m)
        self.dtype = np.dtype(dtype)
        kind = 8 if self.dtype == np.float64 else 4
        if shard is None:
            self.h = lib().lbfgsb_dev_create(self.n, self.m, kind, stream)
        else:
            off, n_global, comm, rank, world = shard
            self.h = lib().lbfgsb_dev_create_sharded(self.n, off, n_global, self.m, kind, stream, comm, rank, world)
        if not self.h:
            raise LbfgsbB200Error("lbfgsb_dev_create failed: " + last_error())
        self.task = np.full(60, ord(" "), dtype=np.uint8)
        self.task[:5] = np.frombuffer(b"START", dtype=np.uint8)
        self.csave = np.full(60, ord(" "), dtype=np.uint8)
        self.lsave = np.zeros(4, dtype=np.int32)
        self.isave = np.zeros(44, dtype=np.int32)
        self.dsave = np.zeros(29, dtype=self.dtype)
        self.f = np.zeros(1, dtype=self.dtype)
        sfx, self._cr = _REAL[self.dtype]
        self._fn = getattr(lib(), "lbfgsb_setulb_dev_" + sfx)
        self._ip = C.c_int32(iprint)
        if iteration_file:
            lib().lbfgsb_dev_set_iteration_file(C.c_void_p(self.h), iteration_file.encode())

    def task_str(self):
        return bytes(self.task).decode().rstrip()

    def set_task(self, s):
        self.task[:] = ord(" ")
        b = s.encode()
        self.task[:len(b)] = np.frombuffer(b, dtype=np.uint8)

    def setulb_dev(self, x, l, u, nbd, g, factr, pgtol):
        # the marshalled argument list is kept for as long as the same buffers come back (the hot loop of a caller)
        key = (x.data_ptr(), l.data_ptr(), u.data_ptr(), nbd.data_ptr(), g.data_ptr(), factr, pgtol, self.f.ctypes.data,
               self.task.ctypes.data, self.csave.ctypes.data, self.lsave.ctypes.data, self.isave.ctypes.data,
               self.dsave.ctypes.data)
        if key != getattr(self, "_argkey", None):
            fa, pg = self._cr(factr), self._cr(pgtol)
            self._argkeep = (fa, pg)
            self._args = (C.c_void_p(self.h), C.c_void_p(key[0]), C.c_void_p(key[1]), C.c_void_p(key[2]), C.c_void_p(key[3]),
                          _p(self.f), C.c_void_p(key[4]), C.byref(fa), C.byref(pg), _p(self.task), C.byref(self._ip),
                          _p(self.csave), _p(self.lsave), _p(self.isave), _p(self.dsave))
            self._argkey = key
        self._fn(*self._args)
        if self.task[0] == 69:     # 'E': an ERROR task -- raise for the ones that mean the engine itself failed
            _check_task(self.task)

    def minimize(self, x, l, u, nbd, g, fg, factr, pgtol, max_iter=0, max_fg=0):
        """lbfgsb_minimize_dev_*: the library owns the task loop (include/lbfgsb_b200.h section 3).
        fg(x, g) -> f evaluates the objective at the tensor x into the tensor g.  Returns the C return code;
        self.task / self.f / self.isave / self.dsave hold the final state."""
        sfx, cr = _REAL[self.dtype]
        CB = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.POINTER(cr), C.c_void_p)

        def _cb(user, n, xp, gp, fout, stream):
            try:
                fout[0] = fg(x, g)
                return 0
            except Exception:  # noqa: BLE001
                return 1
        cb = CB(_cb)
        fn = getattr(lib(), "lbfgsb_minimize_dev_" + sfx)
        fn.restype = C.c_int
        fn.argtypes = [C.c_void_p] * 5 + [CB, C.c_void_p, cr, cr, C.c_int32, C.c_int32, C.c_int32] + [C.c_void_p] * 7
        rc = fn(C.c_void_p(self.h), C.c_void_p(x.data_ptr()), C.c_void_p(l.data_ptr()), C.c_void_p(u.data_ptr()),
                C.c_void_p(nbd.data_ptr()), cb, None, cr(factr), cr(pgtol), int(max_iter), int(max_fg), self._ip.value,
                _p(self.f), C.c_void_p(g.data_ptr()), _p(self.task), _p(self.csave), _p(self.lsave), _p(self.isave),
                _p(self.dsave))
        _check_task(self.task)
        return rc

    def minimize_graph(self, x, l, u, nbd, g, fg_enqueue, factr, pgtol, max_iter=0, max_fg=0):
        """lbfgsb_minimize_graph_dev_*: the task loop kept on the device, one CUDA-graph launch per iteration step.
        fg_enqueue(x_ptr, g_ptr, f_dev_ptr, stream) only enqueues the objective's kernels on `stream` (it is captured in a
        CUDA graph) and leaves f in device memory.  Returns the C return code."""
        sfx, cr = _REAL[self.dtype]
        CB = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p)

        def _cb(user, n, xp, gp, fdev, stream):
            try:
                fg_enqueue(xp, gp, fdev, stream)
                return 0
            except Exception:  # noqa: BLE001
                return 1
        cb = CB(_cb)
        fn = getattr(lib(), "lbfgsb_minimize_graph_dev_" + sfx)
        fn.restype = C.c_int
        fn.argtypes = [C.c_void_p] * 5 + [CB, C.c_void_p, cr, cr, C.c_int32, C.c_int32] + [C.c_void_p] * 7
        rc = fn(C.c_void_p(self.h), C.c_void_p(x.data_ptr()), C.c_void_p(l.data_ptr()), C.c_void_p(u.data_ptr()),
                C.c_void_p(nbd.data_ptr()), cb, None, cr(factr), cr(pgtol), int(max_iter), int(max_fg),
                _p(self.f), C.c_void_p(g.data_ptr()), _p(self.task), _p(self.csave), _p(self.lsave), _p(self.isave),
                _p(self.dsave))
        _check_task(self.task)
        return rc

    def graph_stats(self):
        """(steps that ran as one graph launch, engine kernels per such launch)."""
        a, b = C.c_int64(0), C.c_int64(0)
        lib().lbfgsb_dev_graph_stats(C.c_void_p(self.h), C.byref(a), C.byref(b))
        return a.value, b.value

    def checkpoint_write(self, path):
        if lib().lbfgsb_dev_checkpoint_write(C.c_void_p(self.h), path.encode()) != 0:
            raise LbfgsbB200Error("checkpoint write failed: " + last_error())

    def checkpoint_read(self, path):
        if lib().lbfgsb_dev_checkpoint_read(C.c_void_p(self.h), path.encode()) != 0:
            raise LbfgsbB200Error("checkpoint read failed: " + last_error())

    def active_set_hash(self):
        h, c = C.c_uint64(0), C.c_int64(0)
        if lib().lbfgsb_dev_active_set_hash(C.c_void_p(self.h), C.byref(h), C.byref(c)) != 0:
            raise LbfgsbB200Error(last_error())
        return h.value, c.value

    @staticmethod
    def _opt(t):
        return C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p(0)

    def fused_fg(self, kind, x, g, l=None, u=None, nbd=None, seed=0):
        """Sample objective (0 Rosenbrock, 1 quadratic) on this single-GPU workspace's stream.  With l, u, nbd the
        kernel also forms the line-search sums gd = g.d and max |proj g| (include/lbfgsb_b200.h:
        lbfgsb_problem_fused_f64), and the next setulb_dev call skips its own pass over g, d, x, l, u, nbd."""
        out = C.c_double(0.0)
        rc = lib().lbfgsb_problem_fused_f64(C.c_void_p(self.h), C.c_int32(kind), C.c_void_p(x.data_ptr()),
                                            C.c_void_p(g.data_ptr()), self._opt(l), self._opt(u), self._opt(nbd),
                                            C.byref(out), C.c_uint64(int(seed)))
        if rc != 0:
            raise LbfgsbB200Error("objective kernel failed (rc %d): %s" % (rc, last_error()))
        return out.value

    def sharded_fg(self, kind, x, g, l=None, u=None, nbd=None, seed=0):
        """Sample objective (0 Rosenbrock, 1 quadratic) of this rank's shard with halo and partial-f exchange over peer
        memory (include/lbfgsb_b200.h: lbfgsb_problem_sharded_f64); with l, u, nbd also the line-search sums, as
        fused_fg.  Returns f, or None when the workspace does not exchange over peer memory."""
        out = C.c_double(0.0)
        rc = lib().lbfgsb_problem_sharded_f64(C.c_void_p(self.h), C.c_int32(kind), C.c_void_p(x.data_ptr()),
                                              C.c_void_p(g.data_ptr()), self._opt(l), self._opt(u), self._opt(nbd),
                                              C.byref(out), C.c_uint64(int(seed)))
        if rc == 2:
            return None
        if rc != 0:
            raise LbfgsbB200Error("sharded objective failed: " + last_error())
        return out.value

    def exchange_mode(self):
        """0 single GPU, 1 records through ncclAllGather, 2 records stored into the peers' memory (NVLink)."""
        return int(lib().lbfgsb_dev_exchange_mode(C.c_void_p(self.h)))

    def counters(self):
        a, b = C.c_int64(0), C.c_int64(0)
        lib().lbfgsb_dev_counters(C.c_void_p(self.h), C.byref(a), C.byref(b))
        return a.value, b.value

    def set_tie_limit(self, max_breakpoints):
        """Heap replay of equal breakpoints at the exit of the Cauchy search (include/lbfgsb_b200.h); 0 = off."""
        lib().lbfgsb_dev_set_tie_limit(C.c_void_p(self.h), C.c_int64(int(max_breakpoints)))

    def tie_stats(self):
        """(heap replays done, exits inside a tie group that were not replayed)."""
        a, b = C.c_int64(0), C.c_int64(0)
        lib().lbfgsb_dev_tie_stats(C.c_void_p(self.h), C.byref(a), C.byref(b))
        return a.value, b.value

    def profile(self, on=True):
        lib().lbfgsb_dev_profile(C.c_void_p(self.h), 1 if on else 0)

    def profile_reset(self):
        lib().lbfgsb_dev_profile_reset(C.c_void_p(self.h))

    def profile_read(self):
        cap = 64
        names = C.create_string_buffer(32 * cap)
        ms = (C.c_double * cap)()
        by = (C.c_double * cap)()
        calls = (C.c_int64 * cap)()
        k = lib().lbfgsb_dev_profile_read(C.c_void_p(self.h), cap, names, ms, by, calls)
        out = {}
        for i in range(k):
            nm = names.raw[32 * i:32 * (i + 1)].split(b"\0")[0].decode()
            out[nm] = {"ms": ms[i], "bytes": by[i], "calls": calls[i]}
        return out

    def vector(self, which, count=None, dtype=None):
        """Copy of a work vector (diagnostics): 0 z, 1 r, 2 d, 3 t, 4 xp, 7 iwhere, 8 the previous gradient, all of n
        elements by default; 5 ws and 6 wy hold m columns of ldw = roundup(n, 32) reals (column j of the S/Y ring at
        j * ldw), so pass count = m * ldw for them.  A count beyond the vector's allocation raises."""
        torch = self.torch
        n = self.n if count is None else count
        tdt = {np.dtype(np.float64): torch.float64, np.dtype(np.float32): torch.float32}[self.dtype]
        if which == 7:
            tdt = torch.int32
        out = torch.empty(n, dtype=tdt, device="cuda")
        if lib().lbfgsb_dev_vector_copy(C.c_void_p(self.h), which, C.c_void_p(out.data_ptr()),
                                        C.c_int64(out.numel() * out.element_size())) != 0:
            raise LbfgsbB200Error("lbfgsb_dev_vector_copy failed")
        return out

    def close(self):
        if self.h:
            lib().lbfgsb_dev_destroy(C.c_void_p(self.h))
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class RosenbrockDevice:
    """f/g of the reference's sample problem (test/driver1.f90:274-289) evaluated on the device."""

    def __init__(self, dtype, stream=None):
        import torch
        self.dtype = np.dtype(dtype)
        self.scratch = torch.empty(int(lib().lbfgsb_problem_scratch_bytes()), dtype=torch.uint8, device="cuda")
        sfx, self._cr = _REAL[self.dtype]
        self._fn = getattr(lib(), "lbfgsb_problem_rosenbrock_" + sfx)
        self._f = np.zeros(1, dtype=self.dtype)
        self.stream = stream
        self._n = 0

    def __call__(self, x, g, first=1, last=1, xl=0.0, xr=0.0):
        self._n = x.numel()
        rc = self._fn(C.c_int64(x.numel()), C.c_void_p(x.data_ptr()), C.c_void_p(g.data_ptr()), _p(self._f),
                      C.c_void_p(self.stream), first, last, self._cr(xl), self._cr(xr), C.c_void_p(self.scratch.data_ptr()))
        if rc != 0:
            raise LbfgsbB200Error("rosenbrock kernel failed: " + last_error())
        return self._f[0]

    def enqueue(self, halo_dev):
        """An objective for DeviceProblem.minimize_graph (float64, whole problem on one GPU): kernels only, f stays on the
        device.  halo_dev: two zeros on the device (the neighbours' values of a shard; unused here)."""
        def fg(xp, gp, fdev, stream):
            rc = lib().lbfgsb_problem_rosenbrock_halo_f64(C.c_int64(self._n), C.c_void_p(xp), C.c_void_p(gp), C.c_void_p(fdev),
                                                          C.c_void_p(stream), 1, 1, C.c_void_p(halo_dev.data_ptr()),
                                                          C.c_void_p(self.scratch.data_ptr()))
            if rc != 0:
                raise LbfgsbB200Error("rosenbrock kernel failed")
        return fg

    def shard_async(self, x, g, first, last, halo_dev, f_part_dev):
        """Shard evaluation without a host round trip (float64): xl, xr from halo_dev[0..1], partial f -> f_part_dev."""
        rc = lib().lbfgsb_problem_rosenbrock_halo_f64(
            C.c_int64(x.numel()), C.c_void_p(x.data_ptr()), C.c_void_p(g.data_ptr()), C.c_void_p(f_part_dev.data_ptr()),
            C.c_void_p(self.stream), C.c_int32(first), C.c_int32(last), C.c_void_p(halo_dev.data_ptr()), C.c_void_p(self.scratch.data_ptr()))
        if rc != 0:
            raise LbfgsbB200Error("rosenbrock kernel failed")


class QuadraticDevice:
    """f/g of the bound-constrained convex quadratic of BASELINE.json configs[3] on the device
    (include/lbfgsb_b200.h: lbfgsb_problem_quadratic_*).  `offset` is the global index of x[0]."""

    def __init__(self, dtype, seed=0, stream=None):
        import torch
        self.dtype = np.dtype(dtype)
        self.seed = int(seed)
        self.scratch = torch.empty(int(lib().lbfgsb_problem_scratch_bytes()), dtype=torch.uint8, device="cuda")
        sfx, self._cr = _REAL[self.dtype]
        self._fn = getattr(lib(), "lbfgsb_problem_quadratic_" + sfx)
        self._f = np.zeros(1, dtype=self.dtype)
        self.stream = stream

    def __call__(self, x, g, offset=0, xl=0.0, xr=0.0):
        rc = self._fn(C.c_int64(x.numel()), C.c_void_p(x.data_ptr()), C.c_void_p(g.data_ptr()), _p(self._f),
                      C.c_void_p(self.stream), C.c_int64(offset), C.c_uint64(self.seed), self._cr(xl), self._cr(xr),
                      C.c_void_p(self.scratch.data_ptr()))
        if rc != 0:
            raise LbfgsbB200Error("quadratic kernel failed: " + last_error())
        return self._f[0]

    def shard_async(self, x, g, offset, halo_dev, f_part_dev):
        rc = lib().lbfgsb_problem_quadratic_halo_f64(
            C.c_int64(x.numel()), C.c_void_p(x.data_ptr()), C.c_void_p(g.data_ptr()), C.c_void_p(f_part_dev.data_ptr()),
            C.c_void_p(self.stream), C.c_int64(offset), C.c_uint64(self.seed), C.c_void_p(halo_dev.data_ptr()),
            C.c_void_p(self.scratch.data_ptr()))
        if rc != 0:
            raise LbfgsbB200Error("quadratic kernel failed")


class BatchProblem:
    """Batched small problems (include/lbfgsb_b200.h section 6): nprob independent problems of the same n and m, one
    CTA per problem, one call per reverse-communication step of the whole batch.  x, l, u, g are [nprob, n] CUDA tensors,
    nbd [nprob, n] int32, f a CUDA tensor [nprob]; task / csave / lsave / isave / dsave are per-problem host arrays with
    the reference's meaning (src/lbfgsb.f90:194-242)."""

    def __init__(self, nprob, n, m, dtype=np.float64, stream=None):
        self.nprob, self.n, self.m = int(nprob), int(n), int(m)
        self.dtype = np.dtype(dtype)
        kind = 8 if self.dtype == np.float64 else 4
        self.h = lib().lbfgsb_batch_create(self.nprob, self.n, self.m, kind, stream)
        if not self.h:
            raise LbfgsbB200Error("lbfgsb_batch_create failed: " + last_error())
        self.task = np.full((self.nprob, 60), ord(" "), dtype=np.uint8)
        self.task[:, :5] = np.frombuffer(b"START", dtype=np.uint8)
        self.csave = np.full((self.nprob, 60), ord(" "), dtype=np.uint8)
        self.lsave = np.zeros((self.nprob, 4), dtype=np.int32)
        self.isave = np.zeros((self.nprob, 44), dtype=np.int32)
        self.dsave = np.zeros((self.nprob, 29), dtype=self.dtype)
        sfx, self._cr = _REAL[self.dtype]
        self._fn = getattr(lib(), "lbfgsb_batch_setulb_dev_" + sfx)
        self._fg = getattr(lib(), "lbfgsb_problem_rosenbrock_batch_" + sfx)
        self.stream = lib().lbfgsb_batch_stream(C.c_void_p(self.h))
        self.fg_mask_ptr = lib().lbfgsb_batch_fg_mask(C.c_void_p(self.h))
        self._ext = None      # torch's view of the batch's stream, made at the first call

    def _after_torch(self):
        """Orders the batch's stream after the work enqueued so far on torch's current stream."""
        import torch
        if self._ext is None:
            self._ext = torch.cuda.ExternalStream(self.stream)
        self._ext.wait_stream(torch.cuda.current_stream())

    def task_str(self, p):
        return bytes(self.task[p]).decode().rstrip()

    def set_task(self, p, text):
        self.task[p, :] = ord(" ")
        b = text.encode()
        self.task[p, :len(b)] = np.frombuffer(b, dtype=np.uint8)

    def setulb_dev(self, x, l, u, nbd, f, g, factr, pgtol):
        """One call for the whole batch.  The batch's stream first waits for torch's current stream, so f and g written
        there by a torch objective are complete before the kernel reads them."""
        self._after_torch()
        fa, pg = self._cr(factr), self._cr(pgtol)
        self._fn(C.c_void_p(self.h), C.c_void_p(x.data_ptr()), C.c_void_p(l.data_ptr()), C.c_void_p(u.data_ptr()),
                 C.c_void_p(nbd.data_ptr()), C.c_void_p(f.data_ptr()), C.c_void_p(g.data_ptr()), C.byref(fa), C.byref(pg),
                 _p(self.task), _p(self.csave), _p(self.lsave), _p(self.isave), _p(self.dsave))
        if (self.task[:, 0] == 69).any():
            for p in range(self.nprob):
                _check_task(self.task[p])

    def iwhere(self):
        """iwhere of every problem ([nprob, n] int32 on the host): the reference's iwa(2n+1:3n) per problem."""
        out = np.empty((self.nprob, self.n), dtype=np.int32)
        if lib().lbfgsb_batch_get_iwhere(C.c_void_p(self.h), _p(out)) != 0:
            raise LbfgsbB200Error("lbfgsb_batch_get_iwhere failed")
        return out

    def vector(self, p, which, count=None):
        """Copy of problem p's slice of a work vector (diagnostics; codes of DeviceProblem.vector): n elements by
        default; ws (5) and wy (6) hold m columns of ldw = roundup(n, 32) reals, so pass count = m * ldw for them.
        A problem out of range or a count beyond the problem's slice raises."""
        import torch
        k = self.n if count is None else int(count)
        tdt = torch.int32 if which == 7 else {np.dtype(np.float64): torch.float64, np.dtype(np.float32): torch.float32}[self.dtype]
        out = torch.empty(k, dtype=tdt, device="cuda")
        self._after_torch()     # the copy runs on the batch's stream
        if lib().lbfgsb_batch_vector_copy(C.c_void_p(self.h), int(p), int(which), C.c_void_p(out.data_ptr()),
                                          C.c_int64(out.numel() * out.element_size())) != 0:
            raise LbfgsbB200Error("lbfgsb_batch_vector_copy failed: " + last_error())
        return out

    def counts(self):
        a, b, c = C.c_int32(0), C.c_int32(0), C.c_int32(0)
        lib().lbfgsb_batch_counts(C.c_void_p(self.h), C.byref(a), C.byref(b), C.byref(c))
        return a.value, b.value, c.value

    def rosenbrock_fg(self, x, g, f, all_problems=False):
        """Sample objective (test/driver1.f90:274-289) on the batch's stream, for the problems whose task asks for f and g
        (the batch's own device mask), or for every problem."""
        rc = self._fg(self.nprob, self.n, C.c_void_p(x.data_ptr()), C.c_void_p(g.data_ptr()), C.c_void_p(f.data_ptr()),
                      None if all_problems else C.c_void_p(self.fg_mask_ptr), C.c_void_p(self.stream))
        if rc != 0:
            raise LbfgsbB200Error("batched objective kernel failed")

    def solve(self, x, l, u, nbd, f, g, factr, pgtol, fg=None, max_iter=0, on_newx=None):
        """The task loop of test/driver1.f90:263-292 for the whole batch.  fg(x, g, f) evaluates every problem (default:
        the sample objective); max_iter > 0 stops a problem at that many iterations as driver2.f90:174-181 does."""
        fg = fg or (lambda xx, gg, ff: self.rosenbrock_fg(xx, gg, ff))
        calls = 0
        while True:
            self.setulb_dev(x, l, u, nbd, f, g, factr, pgtol)
            calls += 1
            nfg, nnew, _ = self.counts()
            if nfg == 0 and nnew == 0:
                return calls
            if nfg:
                fg(x, g, f)
            if nnew:
                if on_newx is not None:
                    on_newx(self)
                if max_iter > 0:
                    for p in np.nonzero((self.task[:, 0] == 78) & (self.isave[:, 29] >= max_iter))[0]:
                        self.set_task(int(p), "STOP: TOTAL NO. of ITERATIONS REACHED LIMIT")

    def close(self):
        if self.h:
            lib().lbfgsb_batch_destroy(C.c_void_p(self.h))
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
