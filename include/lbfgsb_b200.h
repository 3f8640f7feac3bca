/* lbfgsb_b200 -- C ABI of the B200-native L-BFGS-B iteration engine.
 *
 * Drop-in boundary for ONE path of jacobwilliams/lbfgsb: everything `mainlb`
 * does between two returns to the caller, behind the reference's own
 * reverse-communication entry point
 *
 *     subroutine setulb(n,m,x,l,u,Nbd,f,g,Factr,Pgtol,Wa,Iwa,Task,Iprint,
 *                       Csave,Lsave,Isave,Dsave,iteration_file)      src/lbfgsb.f90:88-89
 *
 * Same `task` protocol ('START' -> 'FG_START' -> 'FG_LNSRCH'* -> 'NEW_X' -> ... ->
 * 'CONVERGENCE: ...' | 'ABNORMAL_TERMINATION_IN_LNSRCH' | 'ERROR: ...'; user 'STOP...'),
 * same meaning of isave(22:44), dsave(1:29), lsave(1:4)   (src/lbfgsb.f90:194-242, :904-947).
 * All arguments are passed by reference, strings are blank-padded character(60),
 * logicals are 4-byte, so a Fortran `bind(C)` interface forwards 1:1
 * (see fortran/lbfgsb_b200_module.F90 and INTEGRATION.md).
 *
 * There is no CPU fallback: every entry point needs a CUDA device and fails with
 * task = 'ERROR: ...' / a non-zero return code when there is none.
 */
#ifndef LBFGSB_B200_H
#define LBFGSB_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define LBFGSB_B200_MMAX 20   /* largest history size m (reference recommends 3 <= m <= 20, src/lbfgsb.f90:95-97) */

typedef struct lbfgsb_dev lbfgsb_dev_t;   /* opaque device workspace: replaces wa/iwa (src/lbfgsb.f90:146-149) */

int lbfgsb_b200_version(void);
/* last error text of the calling thread's most recent failing call ("" if none) */
const char* lbfgsb_b200_last_error(void);

/* ---- (1) host twin of setulb: host arrays in, host arrays out -------------------------------
 * replaces: setulb, src/lbfgsb.f90:88-286 (REAL64 build) / the -DREAL32 build (lbfgsb_kinds_module.F90:29-37).
 * x,l,u,nbd are staged to the GPU at task='START'; g (and f) on every 'FG' re-entry; x is copied
 * back whenever the engine changed it.  wa/iwa are accepted for signature compatibility and are
 * not used as workspace (the state lives on the device); the handle is kept in isave(17:19),
 * which the reference leaves unused.  itfile/itfile_len = iteration_file (may be NULL/0).   */
void lbfgsb_setulb_f64(const int32_t* n, const int32_t* m, double* x, const double* l, const double* u,
                       const int32_t* nbd, double* f, double* g, const double* factr, const double* pgtol,
                       double* wa, int32_t* iwa, char* task, const int32_t* iprint, char* csave,
                       int32_t* lsave, int32_t* isave, double* dsave, const char* itfile, int32_t itfile_len);
void lbfgsb_setulb_f32(const int32_t* n, const int32_t* m, float* x, const float* l, const float* u,
                       const int32_t* nbd, float* f, float* g, const float* factr, const float* pgtol,
                       float* wa, int32_t* iwa, char* task, const int32_t* iprint, char* csave,
                       int32_t* lsave, int32_t* isave, float* dsave, const char* itfile, int32_t itfile_len);
/* frees the device workspace bound to this isave (needed when the caller leaves its loop on a
 * user 'STOP' without calling setulb again, as test/driver2.f90:174-190 does) */
void lbfgsb_host_release(int32_t* isave);
/* copies the previous iterate t (= wa(lt:lt+n-1), read by test/driver3.f90:173-175) to the host */
int lbfgsb_host_previous_x_f64(const int32_t* isave, double* t_out);
int lbfgsb_host_previous_x_f32(const int32_t* isave, float* t_out);
/* the device workspace behind a host-twin problem (NULL if none), for the diagnostics of section (4) */
lbfgsb_dev_t* lbfgsb_host_engine(const int32_t* isave);

/* ---- (2) device-pointer variant --------------------------------------------------------------
 * x, g, l, u, nbd are CUDA device pointers (16-byte aligned); f and the state arrays stay on the
 * host.  The caller's f/g evaluation and every O(n), O(mn) step of the iteration stay on the GPU.
 * real_kind: 8 (REAL64) or 4 (REAL32).  cuda_stream: a cudaStream_t (NULL = a private stream).
 * n is the number of variables held by this process.                                         */
lbfgsb_dev_t* lbfgsb_dev_create(int64_t n, int32_t m, int32_t real_kind, void* cuda_stream);
/* sharded over `world` GPUs by variable index (contiguous blocks): n_local variables starting at
 * global index `offset` of n_global; nccl_comm is an initialised ncclComm_t (see
 * lbfgsb_dev_nccl_unique_id / lbfgsb_dev_nccl_init).                                            */
lbfgsb_dev_t* lbfgsb_dev_create_sharded(int64_t n_local, int64_t offset, int64_t n_global, int32_t m,
                                        int32_t real_kind, void* cuda_stream, void* nccl_comm,
                                        int32_t rank, int32_t world);
void lbfgsb_dev_destroy(lbfgsb_dev_t* h);
/* name of the summary file written when iprint >= 1 (the optional `iteration_file` argument of setulb,
 * src/lbfgsb.f90:243; default 'iterate.dat').  Call before the START entry.                      */
void lbfgsb_dev_set_iteration_file(lbfgsb_dev_t* h, const char* name);
void lbfgsb_setulb_dev_f64(lbfgsb_dev_t* h, double* x_dev, const double* l_dev, const double* u_dev,
                           const int32_t* nbd_dev, double* f, double* g_dev, const double* factr,
                           const double* pgtol, char* task, const int32_t* iprint, char* csave,
                           int32_t* lsave, int32_t* isave, double* dsave);
void lbfgsb_setulb_dev_f32(lbfgsb_dev_t* h, float* x_dev, const float* l_dev, const float* u_dev,
                           const int32_t* nbd_dev, float* f, float* g_dev, const float* factr,
                           const float* pgtol, char* task, const int32_t* iprint, char* csave,
                           int32_t* lsave, int32_t* isave, float* dsave);

/* ---- (3) driver that owns the task loop (the reference's own @todo, src/lbfgsb.f90:36-37) -----------
 * The loop of test/driver1.f90:263-292 / driver2.f90:112-190 in C: calls fg whenever task(1:2) == 'FG',
 * stops like driver2 (:174-181) when the number of iterations reaches max_iter or the number of f/g
 * evaluations reaches max_fg (task = 'STOP: ...'; a limit <= 0 is no limit).  fg evaluates f and g at
 * x_dev on the given stream, stores f in *f_out (host) and returns 0 (non-zero aborts with
 * task = 'STOP: THE OBJECTIVE CALLBACK FAILED').  Returns 0 when the loop ended on CONVERGENCE or a STOP
 * limit, 1 on ABNORMAL_TERMINATION, 2 on ERROR.  task/csave/lsave/isave/dsave as in setulb. */
typedef int (*lbfgsb_fg_dev_f64)(void* user, int64_t n, const double* x_dev, double* g_dev, double* f_out, void* cuda_stream);
typedef int (*lbfgsb_fg_dev_f32)(void* user, int64_t n, const float* x_dev, float* g_dev, float* f_out, void* cuda_stream);
int lbfgsb_minimize_dev_f64(lbfgsb_dev_t* h, double* x_dev, const double* l_dev, const double* u_dev, const int32_t* nbd_dev,
                            lbfgsb_fg_dev_f64 fg, void* user, double factr, double pgtol, int32_t max_iter, int32_t max_fg,
                            int32_t iprint, double* f, double* g_dev, char* task, char* csave, int32_t* lsave, int32_t* isave,
                            double* dsave);
int lbfgsb_minimize_dev_f32(lbfgsb_dev_t* h, float* x_dev, const float* l_dev, const float* u_dev, const int32_t* nbd_dev,
                            lbfgsb_fg_dev_f32 fg, void* user, float factr, float pgtol, int32_t max_iter, int32_t max_fg,
                            int32_t iprint, float* f, float* g_dev, char* task, char* csave, int32_t* lsave, int32_t* isave,
                            float* dsave);

/* The same loop kept on the device.  fg only ENQUEUES work on cuda_stream (kernel launches, no synchronisation, no host
 * read-back: it is captured in a CUDA graph) and leaves f in *f_dev (device memory).  One iteration step -- the objective,
 * the FG_LNSRCH entry of setulb, the NEW_X entry -- is then one graph launch and one read-back of the state header
 * (src/lbfgsb.f90:36-37 @todo; the reverse-communication contract :884-890, :770-787 is kept on the device: each entry
 * kernel opens its setulb call only if `task` in the state block asks for it).  START / FG_START, the STOP of a limit and
 * every branch off the common path (breakpoint walk, entering/leaving variables, backtrack, restarts) go through setulb as
 * in lbfgsb_minimize_dev_*; the results are bit-identical to that loop.  Single-GPU workspaces with bounds; otherwise the
 * loop runs call by call with f read back from *f_dev.  No text output (iprint < 0).  Return value as lbfgsb_minimize_dev_*. */
typedef int (*lbfgsb_fg_enqueue_f64)(void* user, int64_t n, const double* x_dev, double* g_dev, double* f_dev, void* cuda_stream);
typedef int (*lbfgsb_fg_enqueue_f32)(void* user, int64_t n, const float* x_dev, float* g_dev, float* f_dev, void* cuda_stream);
int lbfgsb_minimize_graph_dev_f64(lbfgsb_dev_t* h, double* x_dev, const double* l_dev, const double* u_dev, const int32_t* nbd_dev,
                                  lbfgsb_fg_enqueue_f64 fg, void* user, double factr, double pgtol, int32_t max_iter, int32_t max_fg,
                                  double* f, double* g_dev, char* task, char* csave, int32_t* lsave, int32_t* isave, double* dsave);
int lbfgsb_minimize_graph_dev_f32(lbfgsb_dev_t* h, float* x_dev, const float* l_dev, const float* u_dev, const int32_t* nbd_dev,
                                  lbfgsb_fg_enqueue_f32 fg, void* user, float factr, float pgtol, int32_t max_iter, int32_t max_fg,
                                  float* f, float* g_dev, char* task, char* csave, int32_t* lsave, int32_t* isave, float* dsave);
/* how many steps ran as a graph launch since the workspace was created, and how many kernels one such launch holds
 * (the engine's; the objective's come on top) */
int lbfgsb_dev_graph_stats(lbfgsb_dev_t* h, int64_t* graph_steps, int64_t* launches_per_step);

/* ---- (4) checkpoint / resume of the device workspace ----------------------------------------------
 * The reference keeps its whole state in the caller's wa/iwa/isave/dsave/lsave/task/csave, so a caller can
 * checkpoint by saving those arrays (and test/driver3.f90:152-182 reads `t` out of wa).  Here wa/iwa live on
 * the device: these two calls write / read them (S, Y, the five work vectors, iwhere, the free-set flags
 * and the state block) to / from a file, in chunks through pinned memory.  To resume: create a workspace of
 * the same n, m, real_kind (and shard), read the file, restore your own x, g, f, task, csave, lsave, isave,
 * dsave, and continue calling setulb_dev.  Call them between two setulb calls.  Return 0 on success.   */
int lbfgsb_dev_checkpoint_write(lbfgsb_dev_t* h, const char* path);
int lbfgsb_dev_checkpoint_read(lbfgsb_dev_t* h, const char* path);

/* NCCL plumbing for the sharded variant (128-byte unique id made on rank 0, broadcast by the caller) */
int lbfgsb_dev_nccl_unique_id(void* id128);
void* lbfgsb_dev_nccl_init(const void* id128, int32_t rank, int32_t world);
void lbfgsb_dev_nccl_destroy(void* comm);

/* ---- diagnostics used by the parity tests and the benchmark -------------------------------- */
/* 64-bit identity of the active set {i : iwhere(i) > 0} (freev, src/lbfgsb.f90:2047) and its size */
int lbfgsb_dev_active_set_hash(lbfgsb_dev_t* h, uint64_t* hash, int64_t* count);
/* device pointer of a work vector: 0 z, 1 r, 2 d, 3 t, 4 xp, 5 ws, 6 wy, 7 iwhere, 8 previous gradient */
void* lbfgsb_dev_vector(lbfgsb_dev_t* h, int32_t which);
/* device-to-device copy of `bytes` bytes of that work vector into dst_dev (after the engine's stream drained); returns 1
   without copying when `bytes` exceeds the vector's allocation: m * ldw reals for 5 and 6 (ldw = n rounded up to a
   multiple of 32), ldw int32 for 7, ldw reals otherwise */
int lbfgsb_dev_vector_copy(lbfgsb_dev_t* h, int32_t which, void* dst_dev, int64_t bytes);
/* how the per-rank reduction records travel on a sharded workspace: 0 single GPU, 1 ncclAllGather, 2 stores into the
 * peers' memory over NVLink (CUDA IPC; default when every rank can map every peer, LBFGSB_B200_P2P=0 switches it off) */
int lbfgsb_dev_exchange_mode(lbfgsb_dev_t* h);
/* counters since creation: kernels launched, host syncs, device ms per kernel family (see DESIGN.md) */
int lbfgsb_dev_counters(lbfgsb_dev_t* h, int64_t* launches, int64_t* syncs);
/* per-kernel timing: when enabled every streaming kernel is bracketed by CUDA events on the
 * engine's stream; names/ms/bytes/calls are returned for up to `cap` kernel families          */
void lbfgsb_dev_profile(lbfgsb_dev_t* h, int32_t enable);
int lbfgsb_dev_profile_read(lbfgsb_dev_t* h, int32_t cap, char* names /* cap*32 */, double* ms, double* bytes,
                            int64_t* calls);
void lbfgsb_dev_profile_reset(lbfgsb_dev_t* h);
/* Equal breakpoints at the exit of the generalized-Cauchy-point search (src/lbfgsb.f90:1416 inside a group of
 * equal t): which members of the group end up fixed depends on the order in which they are popped, and the
 * reference pops them in the order of its heap (hpsolb, :2079-2157).  The engine then replays that heap (single-GPU
 * workspaces): by one device thread for calls with up to 16 384 breakpoints, on the engine's host thread from a copy of
 * the breakpoint list beyond that (tens of nanoseconds per heap operation, as the reference pays on every walk), up to
 * `max_breakpoints` breakpoints per call (default 2^28, environment LBFGSB_B200_TIE_LIMIT; 0 switches the replay
 * off).  Beyond the limit such a group is taken in variable order and the event is counted; sharded workspaces always
 * use (t, global index) order.  The batched small-problem path (section 6) pops the reference's heap itself.
 * tie_stats: replays done, exits inside a tie group that were not replayed (since START).            */
void lbfgsb_dev_set_tie_limit(lbfgsb_dev_t* h, int64_t max_breakpoints);
int lbfgsb_dev_tie_stats(lbfgsb_dev_t* h, int64_t* replays, int64_t* not_replayed);

/* ---- sample problem of the reference drivers, evaluated on the device -----------------------
 * test/driver1.f90:274-289: f = 4[ 1/4 (x1-1)^2 + sum_{i>=2} (x_i - x_{i-1}^2)^2 ] and its gradient.
 * xl / xr are the neighbours' boundary values on a shard (ignored when first / last).          */
int lbfgsb_problem_rosenbrock_f64(int64_t n, const double* x_dev, double* g_dev, double* f_out, void* cuda_stream,
                                  int32_t first, int32_t last, double xl, double xr, void* scratch_dev);
int lbfgsb_problem_rosenbrock_f32(int64_t n, const float* x_dev, float* g_dev, float* f_out, void* cuda_stream,
                                  int32_t first, int32_t last, float xl, float xr, void* scratch_dev);
int64_t lbfgsb_problem_scratch_bytes(void);
/* shard variants without a host round trip: xl, xr are read from halo_dev[0..1], the shard's part of f is left
 * in f_part_dev[0] (device), nothing is synchronised -- the caller all-reduces f_part_dev on the same stream */
int lbfgsb_problem_rosenbrock_halo_f64(int64_t n, const double* x_dev, double* g_dev, double* f_part_dev, void* cuda_stream,
                                       int32_t first, int32_t last, const double* halo_dev, void* scratch_dev);
/* Objective with line-search epilogue (SURVEY section 8(f) f4).  While the gradient of a trial point is still in
 * registers, the objective kernel also forms gd = g.d (lnsrlb, src/lbfgsb.f90:2244) and max |proj g| (projgr :2610-2620)
 * in the engine's fixed reduction shape (include/lbfgsb_b200_shape.h) and leaves the block partials where the engine's
 * own pass (k_ls_trial) would; the next lbfgsb_setulb_dev call on the workspace skips that pass (44 bytes per variable).
 * Same products in the same order: results are bit-identical.  Pass l, u, nbd (device pointers, as given to setulb) to
 * get the epilogue, NULL to leave it out.  kind 0: Rosenbrock, 1: quadratic (seed).  Evaluated on the workspace's
 * stream; f is read back once.  Returns 0, 1 on a CUDA failure, 2 when the workspace is of the wrong kind.
 * (The built-in objectives use the caller-side hook below, lbfgsb_dev_trial_sums / _commit.)
 *   lbfgsb_problem_fused_f64   -- single-GPU workspace
 *   lbfgsb_problem_sharded_f64 -- sharded workspace whose ranks exchange over peer memory (lbfgsb_dev_exchange_mode == 2):
 *     halo values and the per-rank parts of f travel as stores into the neighbours' / peers' memory; f is summed in rank
 *     order (identical on every rank).  Returns 2 otherwise (use the *_halo_* variants with your own collectives).   */
/* The same hook for a caller's own gradient kernel.  lbfgsb_dev_trial_sums gives the search direction d and the two
 * arrays of `grid` block partials; the kernel must walk the variables in the fixed shape of lbfgsb_b200_shape.h
 * (`grid` blocks of `block` threads, tiles of block*vec*unroll variables: thread t owns the `vec` variables at
 * t*vec + k*block*vec, k = 0..unroll-1, of a tile), add g_i*d_i into one
 * accumulator per thread in that order, combine lanes by xor-butterfly and warps serially (block_sum_store in
 * lbfgsb_b200/csrc/common.cuh), store the block's sum in gd_part_dev[blockIdx.x] and the block's maximum of
 * |proj g|_i (projgr :2611-2619) in pg_part_dev[blockIdx.x]; then call lbfgsb_dev_trial_sums_commit before the next
 * setulb_dev (task FG_LNSRCH).  Without the commit the engine computes the sums itself.                              */
typedef struct {
    const void* d_dev;      /* search direction of the current line search, n reals                       */
    void* gd_part_dev;      /* [grid] block partials of sum g_i d_i                                        */
    void* pg_part_dev;      /* [grid] block partials of max |proj g|_i                                     */
    int64_t n;
    int32_t grid, block, unroll, real_kind;
    int32_t vec, reserved;
} lbfgsb_trial_sums_t;
int lbfgsb_dev_trial_sums(lbfgsb_dev_t* h, lbfgsb_trial_sums_t* out);
void lbfgsb_dev_trial_sums_commit(lbfgsb_dev_t* h);
int lbfgsb_problem_fused_f64(lbfgsb_dev_t* h, int32_t kind, const double* x_dev, double* g_dev, const double* l_dev,
                             const double* u_dev, const int32_t* nbd_dev, double* f_out, uint64_t seed);
int lbfgsb_problem_sharded_f64(lbfgsb_dev_t* h, int32_t kind, const double* x_dev, double* g_dev, const double* l_dev,
                               const double* u_dev, const int32_t* nbd_dev, double* f_out, uint64_t seed);
int lbfgsb_problem_quadratic_halo_f64(int64_t n, const double* x_dev, double* g_dev, double* f_part_dev, void* cuda_stream,
                                      int64_t index_offset, uint64_t seed, const double* halo_dev, void* scratch_dev);

/* ---- bound-constrained convex quadratic (BASELINE.json configs[3]; SURVEY.md section 8(d) "Config 4") ----
 * f = 1/2 x'Ax - b'x,  A = tridiag(-1, 2 + delta_i, -1),
 * delta_i = 0.1 + hi32(splitmix64(2 i + 2 seed'))/2^32,  b_i = 2 hi32(splitmix64(2 i + 1 + 2 seed'))/2^32 - 1,
 * seed' = seed * 0x9E3779B97F4A7C15 (mod 2^64), i = global 0-based index = index_offset + local index.
 * g = Ax - b.  On a shard the caller passes the neighbours' boundary values xl / xr (0 at the ends of
 * the chain) and adds the partial f over the ranks.  There is no reference file for this objective: the
 * reference ships only the Rosenbrock drivers; this is the weak-scaling workload the north star names. */
int lbfgsb_problem_quadratic_f64(int64_t n, const double* x_dev, double* g_dev, double* f_out, void* cuda_stream,
                                 int64_t index_offset, uint64_t seed, double xl, double xr, void* scratch_dev);
int lbfgsb_problem_quadratic_f32(int64_t n, const float* x_dev, float* g_dev, float* f_out, void* cuda_stream,
                                 int64_t index_offset, uint64_t seed, float xl, float xr, void* scratch_dev);

/* ---- (6) batched small problems (SURVEY.md section 8 f4) ----------------------------------------------
 * The reference keeps no state between calls (src/lbfgsb.f90:52-56): a caller with many small boxes runs many
 * independent copies of the task loop of test/driver1.f90:263-292.  A batch holds nprob problems of the same
 * n and m; ONE call advances every problem from its own task to its next return point of mainlb, one CTA per
 * problem (n <= 65 536 real64 / 131 072 real32 variables).  Same protocol per problem: task and csave are
 * [nprob][60] blank-padded, lsave [nprob][4], isave [nprob][44], dsave [nprob][29] (host arrays, same meaning as
 * in setulb); x, l, u, g are [nprob][n] device arrays, nbd [nprob][n] device int32, and f is a DEVICE array
 * [nprob] (the caller's batched objective kernel writes it; no host round trip for f).  Problems whose task is a
 * terminal one ('CONVERGENCE...', 'ABNORMAL...', 'ERROR...', 'STOP...') are left alone, so the caller simply keeps
 * calling until lbfgsb_batch_counts reports no 'FG' and no 'NEW_X' task.  'STOP' with task(7:9)='CPU' restores the
 * previous iterate of that problem (:565-571).  Equal breakpoints are taken in hpsolb's order (the Cauchy search of
 * a small problem is the reference's own sequential loop, :1378-1497).
 * A call works on the batch's stream (lbfgsb_batch_stream) and reads f_dev and g_dev there: the caller must order
 * that stream after the writes of f and g (an event recorded after the objective and waited on by the batch's
 * stream, or the objective enqueued on that stream itself).  The call synchronises the stream before it returns. */
typedef struct lbfgsb_batch lbfgsb_batch_t;
lbfgsb_batch_t* lbfgsb_batch_create(int32_t nprob, int64_t n, int32_t m, int32_t real_kind, void* cuda_stream);
void lbfgsb_batch_destroy(lbfgsb_batch_t* h);
void lbfgsb_batch_setulb_dev_f64(lbfgsb_batch_t* h, double* x_dev, const double* l_dev, const double* u_dev, const int32_t* nbd_dev,
                                 double* f_dev, double* g_dev, const double* factr, const double* pgtol, char* task, char* csave,
                                 int32_t* lsave, int32_t* isave, double* dsave);
void lbfgsb_batch_setulb_dev_f32(lbfgsb_batch_t* h, float* x_dev, const float* l_dev, const float* u_dev, const int32_t* nbd_dev,
                                 float* f_dev, float* g_dev, const float* factr, const float* pgtol, char* task, char* csave,
                                 int32_t* lsave, int32_t* isave, float* dsave);
/* after a call: how many problems ask for f and g, how many returned 'NEW_X', how many are finished */
int lbfgsb_batch_counts(lbfgsb_batch_t* h, int32_t* n_fg, int32_t* n_newx, int32_t* n_done);
void* lbfgsb_batch_stream(lbfgsb_batch_t* h);   /* the cudaStream_t the batch works on */
/* device int32 [nprob], refreshed by every call: 1 where the problem's task now asks for f and g */
void* lbfgsb_batch_fg_mask(lbfgsb_batch_t* h);
/* iwhere of every problem copied to the host, int32 [nprob][n] -- what the reference keeps in iwa(2n+1:3n)
 * (src/lbfgsb.f90:258; codes -3, -1, 0, 1, 2, 3 of cauchy :1203-1213).  Returns 0 on success. */
int lbfgsb_batch_get_iwhere(lbfgsb_batch_t* h, int32_t* iwhere_host);
/* diagnostics: copy `bytes` of one problem's work vector to dst_dev (device), with the `which` codes of
 * lbfgsb_dev_vector_copy (0 z, 1 r, 2 d, 3 t, 4 xp, 7 iwhere, 8 the previous gradient: ldw = roundup(n, 32) elements;
 * 5 ws, 6 wy: m columns of ldw reals, column j of the S/Y ring at j * ldw).  Returns nonzero for a problem out of
 * range, an unknown code or a byte count beyond that problem's slice. */
int lbfgsb_batch_vector_copy(lbfgsb_batch_t* h, int32_t problem, int32_t which, void* dst_dev, int64_t bytes);
/* the sample objective (test/driver1.f90:274-289) for a batch: problem p from x_dev[p][.] into g_dev[p][.], f_dev[p];
 * mask_dev (may be NULL): int32 [nprob], problems with 0 are skipped */
int lbfgsb_problem_rosenbrock_batch_f64(int32_t nprob, int64_t n, const double* x_dev, double* g_dev, double* f_dev,
                                        const int32_t* mask_dev, void* cuda_stream);
int lbfgsb_problem_rosenbrock_batch_f32(int32_t nprob, int64_t n, const float* x_dev, float* g_dev, float* f_dev,
                                        const int32_t* mask_dev, void* cuda_stream);

/* ---- single-kernel entry points for the per-routine parity tests (device pointers) ---------- */
int lbfgsb_test_projgr_f64(int64_t n, const double* l, const double* u, const int32_t* nbd, const double* x,
                           const double* g, double* sbgnrm_out);
int lbfgsb_test_sum_f64(int64_t n, const double* a, const double* b, double* out);      /* fixed-shape sum of a*b */
int lbfgsb_test_sum_f32(int64_t n, const float* a, const float* b, float* out);
int lbfgsb_test_sort_f64(int64_t n, const double* t_dev, int32_t* order_out_dev, double* sorted_out_dev);
/* hpsolb (:2079-2157) replayed on the device: heap built over t(1..n), popped n times; order_out = iorder of the pops */
/* host-only: the engine's host-thread heap replay (long breakpoint lists, sharded workspaces) on t_host[nb] (> 0, variable
 * order): the variables whose breakpoint equals tk in the reference's order (:1384-1397, hpsolb :2079-2157) */
int lbfgsb_test_host_heap_group_f64(int64_t nb, const double* t_host, double tk, int32_t* group_out, int64_t* group_count);
int lbfgsb_test_heap_order_f64(int64_t n, const double* t_dev, int32_t* order_out_dev);
/* formk's entering/leaving corrections (src/lbfgsb.f90:1801-1851) on their own.  ws_dev, wy_dev: m columns of ldw reals;
 * state_dev: one byte per variable, bit 0 = free now, bit 1 = free before (rows with the two bits different are listed);
 * out_host: six [20 x 20] column-major sums over the listed rows -- entering rows: Wy_i Wy_j, Ws_i Ws_j (both for j <= i),
 * Ws_i Wy_j, then the same three for leaving rows; i, j = position in the ring counted from `head` (1-based column). */
int lbfgsb_test_formk_delta_f64(int64_t n, int32_t m, int32_t col, int32_t head, int64_t ldw, const double* ws_dev,
                                const double* wy_dev, const unsigned char* state_dev, double* out_host);
int lbfgsb_test_formk_delta_f32(int64_t n, int32_t m, int32_t col, int32_t head, int64_t ldw, const float* ws_dev,
                                const float* wy_dev, const unsigned char* state_dev, float* out_host);
int lbfgsb_test_dense_f64(int32_t op, int32_t m, int32_t col, double theta, double* a, double* b, double* c,
                          int32_t* info);   /* op 0 dpofa(a,lda=m,n=col) 1 dtrsl job01 2 dtrsl job11 3 bmv 4 formt (one thread);
                                               10-14 the same by one warp, as the scalar kernels run them; 15 formk's dense
                                               tail (:1853-1906): a = wn1 (2m x 2m), b = sy, c = wn (out) */
int lbfgsb_test_dcsrch_f64(double f, double g, double* stp, double stpmax, int32_t* task, int32_t* isave2,
                           double* dsave13);

#ifdef __cplusplus
}
#endif
#endif
