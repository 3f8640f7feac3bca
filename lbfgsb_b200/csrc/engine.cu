// Host side of the B200 L-BFGS-B engine: device workspace, the kernel pipeline
// enqueued for each `task` entry of the reverse-communication protocol
// (src/lbfgsb.f90:552-577), and the C ABI of include/lbfgsb_b200.h.
//
// One status read-back per return to the caller (plus one after the Cauchy
// classify pass when bounds are present, to size the breakpoint walk).  All
// data-dependent branches of mainlb are taken on the device (kernels_dense.cuh).
#include <cuda_runtime.h>
#include <dlfcn.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <mutex>
#include <string>
#include <unordered_set>
#include <vector>

#include "../../include/lbfgsb_b200.h"
#include "cauchy_walk.cuh"
#include "kernels_tma.cuh"
#include "cauchy_walk_dist.cuh"
#include "batch.cuh"
#include "host_print.h"
#include <algorithm>

// ---------------------------------------------------------------------------
// errors
// ---------------------------------------------------------------------------
static thread_local std::string g_last_error;
static void set_error(const char* fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    g_last_error = buf;
}
#define CK(call)                                                                             \
    do {                                                                                     \
        cudaError_t _e = (call);                                                             \
        if (_e != cudaSuccess) {                                                             \
            set_error("CUDA error %s at %s:%d (%s)", cudaGetErrorString(_e), __FILE__, __LINE__, #call); \
            return false;                                                                    \
        }                                                                                    \
    } while (0)

// ---------------------------------------------------------------------------
// NCCL through dlopen (the process may already hold torch's bundled libnccl.so.2)
// ---------------------------------------------------------------------------
typedef struct ncclComm* ncclComm_t;
typedef struct { char internal[128]; } ncclUniqueId;
struct NcclApi {
    int (*GetUniqueId)(ncclUniqueId*);
    int (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int);
    int (*CommDestroy)(ncclComm_t);
    int (*AllGather)(const void*, void*, size_t, int, ncclComm_t, cudaStream_t);
    int (*Send)(const void*, size_t, int, int, ncclComm_t, cudaStream_t);
    int (*Recv)(void*, size_t, int, int, ncclComm_t, cudaStream_t);
    int (*GroupStart)();
    int (*GroupEnd)();
    const char* (*GetErrorString)(int);
    bool ok;
};
static NcclApi* nccl_api() {
    static NcclApi api;
    static bool tried = false;
    if (!tried) {
        tried = true;
        api.ok = false;
        void* h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
        if (!h) h = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
        if (h) {
            api.GetUniqueId = (int (*)(ncclUniqueId*))dlsym(h, "ncclGetUniqueId");
            api.CommInitRank = (int (*)(ncclComm_t*, int, ncclUniqueId, int))dlsym(h, "ncclCommInitRank");
            api.CommDestroy = (int (*)(ncclComm_t))dlsym(h, "ncclCommDestroy");
            api.AllGather = (int (*)(const void*, void*, size_t, int, ncclComm_t, cudaStream_t))dlsym(h, "ncclAllGather");
            api.GetErrorString = (const char* (*)(int))dlsym(h, "ncclGetErrorString");
            api.Send = (int (*)(const void*, size_t, int, int, ncclComm_t, cudaStream_t))dlsym(h, "ncclSend");
            api.Recv = (int (*)(void*, size_t, int, int, ncclComm_t, cudaStream_t))dlsym(h, "ncclRecv");
            api.GroupStart = (int (*)())dlsym(h, "ncclGroupStart");
            api.GroupEnd = (int (*)())dlsym(h, "ncclGroupEnd");
            api.ok = api.GetUniqueId && api.CommInitRank && api.CommDestroy && api.AllGather && api.Send && api.Recv &&
                     api.GroupStart && api.GroupEnd;
        }
    }
    return &api;
}

#define LB_TIE_DEVICE_MAX 16384   // breakpoints of a call up to which the heap replay runs on the device (one thread)

// ---------------------------------------------------------------------------
// kernel families (profiling / launch accounting)
// ---------------------------------------------------------------------------
enum Fam {
    F_ERRCLB, F_ACTIVE, F_PROJGR, F_CLASSIFY, F_GCP_FREEV, F_FORMK_GRAM, F_FORMK_DELTA, F_CMPRLB_WV,
    F_SUBSM_STEP, F_BACKTRACK, F_LS_INIT, F_LS_STEP, F_LS_TRIAL, F_UPDATE, F_RESTORE, F_WALK_COMPACT,
    F_WALK_SORT, F_WALK_SCAN, F_WALK_FIX, F_SCALAR, F_HASH, F_UPDATE_CLASSIFY, F_FORMK_CMPRLB, F_SUBSM_LSINIT, F_COUNT
};
static const char* fam_name[F_COUNT] = {
    "errclb", "active", "projgr", "cauchy_classify", "gcp_freev", "formk_gram", "formk_delta", "cmprlb_wv",
    "subsm_step", "backtrack", "ls_init", "ls_step", "ls_trial", "update", "restore", "walk_compact",
    "walk_sort", "walk_scan", "walk_fix", "scalar", "hash", "update_classify", "formk_cmprlb", "subsm_lsinit"};

// The scalar header of the state block straight into the host's pinned mirror, then a sequence word: the host waits
// for that word instead of enqueueing a copy and synchronising the stream (a shorter round trip per setulb call).
// The sequence number lives on the device, so that a captured CUDA graph publishes with the same fixed arguments.
__global__ void __launch_bounds__(256) k_publish(const unsigned* src, unsigned* dst_host, int words, volatile unsigned long long* flag_host,
                                                 unsigned long long* counter) {
    for (int q = threadIdx.x; q < words; q += blockDim.x) dst_host[q] = src[q];
    __threadfence_system();
    __syncthreads();
    if (threadIdx.x == 0) { const unsigned long long v = *counter + 1; *counter = v; *flag_host = v; }
}

struct EngineBase {
    virtual ~EngineBase() {}
    int real_kind;
    lbprint::Ctx pr;     // the reference's text output (host_print.h)
};

template <typename T>
struct Engine : EngineBase {
    i64 n = 0, n_global = 0, offset = 0;
    int m = 0, mt = 0;
    bool fused = false;              // the cross-routine fused passes are in use (kernels_tma.cuh: fused_passes_ok)
    cudaStream_t stream = 0;
    bool own_stream = false;
    Wk<T> w;
    WalkBuf<T> wb;
    DevState<T>* s_dev = nullptr;
    DevState<T>* s_host = nullptr;   // pinned mirror (scalar header only is copied)
    size_t header_bytes = 0;
    int* tile_counts = nullptr; i64* tile_offsets = nullptr; i64 ntiles = 0;
    int* rs_counts = nullptr;
    SortCtl* ctl_el = nullptr;
    SortCtl* ctl_host = nullptr;     // pinned
    T* tmpAB = nullptr; T* tmpF = nullptr; unsigned long long* jmin = nullptr;
    T* fd_parts = nullptr; T* delta = nullptr; T* delta_all = nullptr; T* delta_sum = nullptr;
    std::vector<void*> allocs;
    // sharding
    int R = 1, rank = 0;
    ncclComm_t comm = nullptr;
    Red<T>* rec_local = nullptr; Red<T>* rec_all = nullptr;
    // sharded breakpoint walk (cauchy_walk_dist.cuh)
    unsigned long long* samp_local = nullptr; unsigned long long* samp_all = nullptr; unsigned long long* spl_dev = nullptr;
    DwCtl* dctl = nullptr; i64* pos_all = nullptr; SortCtl* ctl_d = nullptr;
    RoundRec* rr_local = nullptr; RoundRec* rr_all = nullptr;
    WalkCarry<T>* carry_local = nullptr; WalkCarry<T>* carry_all = nullptr;
    struct DynBuf { void* p = nullptr; size_t cap = 0; };
    DynBuf dw_send, dw_recv, dw_k0, dw_k1, dw_v0, dw_v1;
    // accounting
    i64 launches = 0, syncs = 0, tie_replays = 0;
    bool profile = false;
    bool debug_launch = (getenv("LBFGSB_B200_DEBUG_LAUNCH") != nullptr);
    struct Ev { int fam; cudaEvent_t a, b; };
    std::vector<Ev> pending;
    std::vector<cudaEvent_t> pool;
    double fam_ms[F_COUNT]; i64 fam_calls[F_COUNT];
    bool x_changed = false, g_changed = false;
    // breakpoint walks tend to come in runs of iterations: after an iteration that needed one, cauchy's per-variable pass of
    // the next iteration also stores every breakpoint and xcp = x (Wk::bp_hint), and the walk's first pass reads 8 bytes
    // per variable instead of recomputing them from x, g, l, u, nbd, iwhere
    bool walked_prev = false, walked_now = false, body_ran = false, bp_hint_ok = true, walk_gf_ok = true;
    bool started = false;            // this workspace has seen task = 'START' (or a checkpoint of a started run)

    // records over peer memory (kernels_dense.cuh: P2PBuf)
    bool p2p = false;
    P2PBuf<T>* p2p_local = nullptr;
    Peers peers, peers_delta;
    std::vector<void*> ipc_opened;
    bool trial_ready = false;   // the caller's objective kernel already left k_ls_trial's partials in w.part (TrialSums)
    unsigned long long site_seq = 0, delta_seq = 0, fg_seq = 0;
    T* fg_scratch = nullptr; T* fg_out = nullptr; T* fg_host = nullptr;
    int cur_slot = 0;
    bool site_pending = false;   // a producer was launched and its consumer not yet: the next dist() carries wait = 1
    Dist<T> dist() {
        Dist<T> d; d.R = R; d.all = rec_all;
        d.p2p = p2p ? p2p_local : nullptr; d.slot = cur_slot; d.seq = site_seq; d.dseq = delta_seq;
        d.wait = site_pending ? 1 : 0; site_pending = false;
        return d;
    }
    // Exchange CUDA IPC handles of the P2PBuf and of delta_all through the engine's communicator and map the peers'
    // buffers.  Any failure on any rank leaves every rank on the ncclAllGather path.
    bool setup_p2p() {
        if (const char* e = getenv("LBFGSB_B200_P2P")) { if (e[0] == '0') return true; }
        struct Pack { cudaIpcMemHandle_t hb, hd; int ok; int pad[3]; };
        Pack mine; memset(&mine, 0, sizeof mine);
        mine.ok = 1;
        if (cudaMalloc((void**)&p2p_local, sizeof(P2PBuf<T>)) != cudaSuccess) { p2p_local = nullptr; mine.ok = 0; cudaGetLastError(); }
        if (mine.ok) {
            allocs.push_back(p2p_local);
            cudaMemset(p2p_local, 0, sizeof(P2PBuf<T>));
            if (cudaIpcGetMemHandle(&mine.hb, p2p_local) != cudaSuccess || cudaIpcGetMemHandle(&mine.hd, delta_all) != cudaSuccess) {
                mine.ok = 0; cudaGetLastError();
            }
        }
        Pack* dsend = nullptr; Pack* drecv = nullptr;
        if (!dalloc(&dsend, sizeof(Pack)) || !dalloc(&drecv, sizeof(Pack) * R)) return false;
        CK(cudaMemcpy(dsend, &mine, sizeof mine, cudaMemcpyHostToDevice));
        if (!allgather(dsend, drecv, sizeof(Pack))) return false;
        std::vector<Pack> all(R);
        CK(cudaMemcpyAsync(all.data(), drecv, sizeof(Pack) * R, cudaMemcpyDeviceToHost, stream));
        CK(cudaStreamSynchronize(stream));
        bool ok = true;
        for (int q = 0; q < R; ++q) ok = ok && all[q].ok;
        memset(&peers, 0, sizeof peers); memset(&peers_delta, 0, sizeof peers_delta);
        int myok = ok ? 1 : 0;
        if (ok) {
            for (int q = 0; q < R && myok; ++q) {
                if (q == rank) { peers.p[q] = p2p_local; peers_delta.p[q] = delta_all; continue; }
                void *pb = nullptr, *pd = nullptr;
                if (cudaIpcOpenMemHandle(&pb, all[q].hb, cudaIpcMemLazyEnablePeerAccess) != cudaSuccess) { myok = 0; cudaGetLastError(); break; }
                ipc_opened.push_back(pb);
                if (cudaIpcOpenMemHandle(&pd, all[q].hd, cudaIpcMemLazyEnablePeerAccess) != cudaSuccess) { myok = 0; cudaGetLastError(); break; }
                ipc_opened.push_back(pd);
                peers.p[q] = pb; peers_delta.p[q] = pd;
            }
        }
        // second round: every rank must have mapped every peer
        int* dflag = nullptr; int* dflags = nullptr;
        if (!dalloc(&dflag, sizeof(int)) || !dalloc(&dflags, sizeof(int) * R)) return false;
        CK(cudaMemcpy(dflag, &myok, sizeof(int), cudaMemcpyHostToDevice));
        if (!allgather(dflag, dflags, sizeof(int))) return false;
        std::vector<int> oks(R);
        CK(cudaMemcpyAsync(oks.data(), dflags, sizeof(int) * R, cudaMemcpyDeviceToHost, stream));
        CK(cudaStreamSynchronize(stream));
        p2p = true;
        for (int q = 0; q < R; ++q) p2p = p2p && oks[q];
        return true;
    }

    template <typename P> bool dalloc(P** p, size_t bytes) {
        void* q = nullptr;
        if (bytes == 0) bytes = 16;
        cudaError_t e = cudaMalloc(&q, bytes);
        if (e != cudaSuccess) { set_error("cudaMalloc(%zu) failed: %s", bytes, cudaGetErrorString(e)); return false; }
        allocs.push_back(q);
        *p = (P*)q;
        return true;
    }

    bool init(i64 n_, i64 off_, i64 ng_, int m_, cudaStream_t st, ncclComm_t cm, int rank_, int world_) {
        n = n_; offset = off_; n_global = ng_; m = m_; R = world_; rank = rank_; comm = cm;
        real_kind = (int)sizeof(T);
        mt = (m <= 5) ? 5 : (m <= 10 ? 10 : 20);
        fused = (mt == 5 ? fused_passes_ok<T, 5>() : (mt == 10 ? fused_passes_ok<T, 10>() : fused_passes_ok<T, 20>()));
        if (const char* e = getenv("LBFGSB_B200_NO_FUSION")) { if (e[0] == '1') fused = false; }
        fast = fused;   // the fast NEW_X pipeline is built from the fused passes
        if (const char* e = getenv("LBFGSB_B200_NO_FAST")) { if (e[0] == '1') fast = false; }
        if (const char* e = getenv("LBFGSB_B200_NO_BP_HINT")) { if (e[0] == '1') { bp_hint_ok = false; walk_gf_ok = false; } }
        if (!(mt == 5 ? set_smem_attrs<5>() : (mt == 10 ? set_smem_attrs<10>() : set_smem_attrs<20>()))) return false;
        for (int q = 0; q < F_COUNT; ++q) { fam_ms[q] = 0; fam_calls[q] = 0; }
        if (st) stream = st;
        else { CK(cudaStreamCreateWithFlags(&stream, cudaStreamNonBlocking)); own_stream = true; }
        memset(&w, 0, sizeof w);
        w.n = n; w.m = m; w.off = offset;
        w.ldw = (n + 31) / 32 * 32;
        const size_t vb = (size_t)w.ldw * sizeof(T);
        if (!dalloc(&w.ws, vb * m) || !dalloc(&w.wy, vb * m)) return false;
        if (!dalloc(&w.z, vb) || !dalloc(&w.r, vb) || !dalloc(&w.d, vb) || !dalloc(&w.t, vb) || !dalloc(&w.xp, vb) || !dalloc(&w.gold, vb)) return false;
        if (!dalloc(&w.iwhere, (size_t)w.ldw * 4) || !dalloc(&w.state, (size_t)w.ldw)) return false;
        if (!dalloc(&w.part, sizeof(T) * LB_KMAX * LBFGSB_GRID) || !dalloc(&w.ipart, sizeof(i64) * LB_IMAX * LBFGSB_GRID)) return false;
        if (!dalloc(&w.part2, sizeof(T) * LB_KMAX * LBFGSB_GRID) || !dalloc(&w.ipart2, sizeof(i64) * LB_IMAX * LBFGSB_GRID)) return false;
        if (!dalloc(&s_dev, sizeof(DevState<T>)) || !dalloc(&pub_counter, 8) || !dalloc(&f_dev, sizeof(T))) return false;
        CK(cudaMemsetAsync(s_dev, 0, sizeof(DevState<T>), stream));
        CK(cudaMemsetAsync(pub_counter, 0, 8, stream));
        {
            i64 lim = (i64)1 << 28;   // heap replay of tied breakpoints at the exit: up to 2.7e8 breakpoints by default
                                      // (on the device up to LB_TIE_DEVICE_MAX, beyond that on the engine's host thread)
            if (R > 1) lim = (i64)1 << 26;   // sharded: every rank holds the whole breakpoint list of the call during a replay
            if (const char* e = getenv("LBFGSB_B200_TIE_LIMIT")) lim = atoll(e);
            CK(cudaMemcpyAsync(&s_dev->tie_limit, &lim, sizeof lim, cudaMemcpyHostToDevice, stream));
        }
        CK(cudaMemsetAsync(w.ws, 0, vb * m, stream));
        CK(cudaMemsetAsync(w.wy, 0, vb * m, stream));
        w.s = s_dev;
        CK(cudaHostAlloc((void**)&s_host, sizeof(DevState<T>) + 64, cudaHostAllocMapped));
        memset(s_host, 0, sizeof(DevState<T>) + 64);
        pub_flag = (volatile unsigned long long*)((char*)s_host + ((sizeof(DevState<T>) + 7) / 8) * 8);
        CK(cudaMallocHost((void**)&ctl_host, sizeof(SortCtl)));
        header_bytes = offsetof(DevState<T>, sy);
        // walk / compaction buffers
        const i64 tile = (i64)LBFGSB_BLOCK * Real<T>::VEC * Real<T>::UNROLL;
        ntiles = (n + tile - 1) / tile;
        if (!dalloc(&tile_counts, sizeof(int) * (size_t)(ntiles + 1)) || !dalloc(&tile_offsets, sizeof(i64) * (size_t)(ntiles + 1))) return false;
        if (!dalloc(&rs_counts, sizeof(int) * 256 * LB_RS_GRID)) return false;
        typedef typename Real<T>::key_t K;
        memset(&wb, 0, sizeof wb);
        if (!dalloc(&wb.k0, sizeof(K) * (size_t)w.ldw) || !dalloc(&wb.k1, sizeof(K) * (size_t)w.ldw)) return false;
        if (!dalloc(&wb.v0, 4 * (size_t)w.ldw) || !dalloc(&wb.v1, 4 * (size_t)w.ldw)) return false;
        if (!dalloc(&wb.ctl, sizeof(SortCtl)) || !dalloc(&ctl_el, sizeof(SortCtl))) return false;
        i64 cap = n < (i64)(1 << 22) ? n : (i64)(1 << 22);   // 4M breakpoints per chunk
        cap = (cap + LB_WB - 1) / LB_WB * LB_WB;
        wb.cap = cap;
        const size_t cb = (size_t)cap * sizeof(T);
        if (!dalloc(&wb.wj, cb * 2 * m) || !dalloc(&wb.vj, cb * 2 * m)) return false;
        if (!dalloc(&wb.delta, cb) || !dalloc(&wb.zeta, cb) || !dalloc(&wb.omega, cb) || !dalloc(&wb.g2, cb) ||
            !dalloc(&wb.g1, cb) || !dalloc(&wb.f1a, cb) || !dalloc(&wb.f2a, cb)) return false;
        const i64 nblk = cap / LB_WB;
        if (!dalloc(&wb.blkA, sizeof(T) * (size_t)nblk * 2 * LB_MMAX) || !dalloc(&wb.blkB, sizeof(T) * (size_t)nblk * 2 * LB_MMAX)) return false;
        if (!dalloc(&wb.blk_a, sizeof(T) * (size_t)nblk) || !dalloc(&wb.blk_b, sizeof(T) * (size_t)nblk) || !dalloc(&wb.blkH, sizeof(T) * (size_t)nblk)) return false;
        if (!dalloc(&tmpAB, sizeof(T) * 4 * LB_MMAX) || !dalloc(&tmpF, sizeof(T) * 2) || !dalloc(&jmin, 8)) return false;
        if (!dalloc(&fd_parts, sizeof(T) * (size_t)LB_FD_GRID * 6 * LB_MMAX * LB_MMAX) || !dalloc(&delta, sizeof(T) * 6 * LB_MMAX * LB_MMAX)) return false;
        CK(cudaMemsetAsync(delta, 0, sizeof(T) * 6 * LB_MMAX * LB_MMAX, stream));
        if (!dalloc(&rr_local, sizeof(RoundRec)) || !dalloc(&rr_all, sizeof(RoundRec) * (R > 1 ? R : 1))) return false;
        if (R > 1) {
            if (R > LB_MAXR) { set_error("at most %d ranks", LB_MAXR); return false; }
            if (!dalloc(&rec_local, sizeof(Red<T>)) || !dalloc(&rec_all, sizeof(Red<T>) * R)) return false;
            const size_t sb = sizeof(unsigned long long) * (2 * LB_DW_SAMPLES + 1);
            if (!dalloc(&samp_local, sb) || !dalloc(&samp_all, sb * R) || !dalloc(&spl_dev, 16 * LB_MAXR)) return false;
            if (!dalloc(&dctl, sizeof(DwCtl)) || !dalloc(&pos_all, sizeof(i64) * (LB_MAXR + 1) * R) || !dalloc(&ctl_d, sizeof(SortCtl))) return false;
            if (!dalloc(&carry_local, sizeof(WalkCarry<T>)) || !dalloc(&carry_all, sizeof(WalkCarry<T>) * R)) return false;
            if (!dalloc(&delta_all, sizeof(T) * 6 * LB_MMAX * LB_MMAX * R) || !dalloc(&delta_sum, sizeof(T) * 6 * LB_MMAX * LB_MMAX)) return false;
        }
        CK(cudaStreamSynchronize(stream));
        if (R > 1 && !setup_p2p()) return false;
        return true;
    }

    ~Engine() {
        for (void* p : ipc_opened) cudaIpcCloseMemHandle(p);
        for (void* p : allocs) cudaFree(p);
        if (iter_graph) cudaGraphExecDestroy(iter_graph);
        for (DynBuf* d : {&dw_send, &dw_recv, &dw_k0, &dw_k1, &dw_v0, &dw_v1, &tie_k, &tie_v, &tie_kall, &tie_vall}) if (d->p) cudaFree(d->p);
        if (fg_host) cudaFreeHost(fg_host);
        if (s_host) cudaFreeHost(s_host);
        if (ctl_host) cudaFreeHost(ctl_host);
        for (auto e : pool) cudaEventDestroy(e);
        for (auto& p : pending) { cudaEventDestroy(p.a); cudaEventDestroy(p.b); }
        if (own_stream && stream) cudaStreamDestroy(stream);
    }

    // ---- phase timers dsave(7:9) = cachyt, sbtime, lnscht (src/lbfgsb.f90:616-637, 655-713, 723-777) -------------
    // CUDA events on the engine's stream at the phase boundaries of a call, resolved after the call's last read-back.
    // On the fused paths a phase is the group of kernels that carries it: "cauchy" = the S/Y update + per-variable
    // pass + its scalar kernel (+ walk), "subspace" = the formk/cmprlb pass through the subspace pass (which also
    // forms lnsrlb's first-entry sums), "line search" = the scalar kernels of lnsrlb/dcsrch and the trial-point passes.
    enum { PH_CAUCHY = 0, PH_SUBSPACE = 1, PH_LNSRCH = 2, PH_END = 3 };
    struct Mark { int ph; cudaEvent_t e; };
    std::vector<Mark> marks;
    double ph_time[3] = {0, 0, 0};
    void phase(int ph) {
        Mark mk; mk.ph = ph; mk.e = get_event();
        cudaEventRecord(mk.e, stream);
        marks.push_back(mk);
    }
    void resolve_phases() {
        if (!marks.empty()) cudaEventSynchronize(marks.back().e);
        for (size_t i = 0; i + 1 < marks.size(); ++i) {
            if (marks[i].ph == PH_END) continue;
            float ms = 0;
            if (cudaEventElapsedTime(&ms, marks[i].e, marks[i + 1].e) == cudaSuccess) ph_time[marks[i].ph] += (double)ms * 1e-3;
        }
        for (auto& mk : marks) pool.push_back(mk.e);
        marks.clear();
    }

    // ---- launch helpers ----------------------------------------------------
    cudaEvent_t get_event() {
        if (!pool.empty()) { cudaEvent_t e = pool.back(); pool.pop_back(); return e; }
        cudaEvent_t e; cudaEventCreate(&e); return e;
    }
    void begin(int fam) {
        if (profile) { Ev ev; ev.fam = fam; ev.a = get_event(); ev.b = get_event(); cudaEventRecord(ev.a, stream); pending.push_back(ev); }
    }
    void end(int fam, int nlaunch = 1) {
        launches += nlaunch;
        if (debug_launch) {   // LBFGSB_B200_DEBUG_LAUNCH=1: name the kernel family whose launch failed
            cudaError_t e = cudaPeekAtLastError();
            if (e != cudaSuccess) fprintf(stderr, "lbfgsb_b200: launch of family '%s' failed: %s\n", fam_name[fam], cudaGetErrorString(e));
        }
        if (profile) cudaEventRecord(pending.back().b, stream);
        else fam_calls[fam] += 1;
    }
    // the timed launches from index `from` on returned at once (the fast pipeline paused in front of them): not counted
    void drop_events_from(size_t from) {
        while (pending.size() > from) { pool.push_back(pending.back().a); pool.push_back(pending.back().b); pending.pop_back(); }
    }
    void resolve_events() {
        if (!pending.empty()) cudaEventSynchronize(pending.back().b);
        for (auto& p : pending) {
            float ms = 0;
            cudaEventElapsedTime(&ms, p.a, p.b);
            fam_ms[p.fam] += ms; fam_calls[p.fam] += 1;
            pool.push_back(p.a); pool.push_back(p.b);
        }
        pending.clear();
    }
    // state read-back: k_publish (enqueued here or captured in the iteration graph) + a wait on the pinned sequence word.
    // Every k_publish that runs is waited for once, so the device counter and pub_expected advance together.
    volatile unsigned long long* pub_flag = nullptr;
    unsigned long long* pub_counter = nullptr;
    unsigned long long pub_expected = 0;
    void enqueue_publish() {
        k_publish<<<1, 256, 0, stream>>>((const unsigned*)s_dev, (unsigned*)s_host, (int)(header_bytes / 4), pub_flag, pub_counter);
    }
    bool wait_published() {
        pub_expected++;
        unsigned spins = 0;
        while (*pub_flag != pub_expected) {
            if ((++spins & 0x3fff) == 0) {   // a faulted kernel never publishes: ask the stream now and then
                cudaError_t q = cudaStreamQuery(stream);
                if (q != cudaSuccess && q != cudaErrorNotReady) { set_error("CUDA error %s while waiting for the state block", cudaGetErrorString(q)); return false; }
                if (q == cudaSuccess && *pub_flag != pub_expected) { set_error("the state block was not published (internal error)"); return false; }
            }
        }
        syncs++;
        return true;
    }
    bool sync_state(bool resolve = true) {
        enqueue_publish(); launches++;
        if (!wait_published()) return false;
        if (profile && resolve) resolve_events();
        if (s_host->p2p_timeout) { set_error("a peer rank's reduction record did not arrive (sharded run over peer memory)"); return false; }
        return true;
    }
    // finish + all-gather of a reduction site on sharded runs
    bool site(const SiteSpec& sp) {
        if (R <= 1) return true;
        site_pending = true;
        if (p2p) {
            site_seq++; cur_slot = (int)(site_seq & 1ULL);
            k_rank_finish_p2p<T><<<1, LB_SCALAR_THREADS, 0, stream>>>(w, sp, peers, R, rank, cur_slot, site_seq);
            launches++;
            return true;
        }
        k_rank_finish<T><<<1, LB_SCALAR_THREADS, 0, stream>>>(w, sp, rec_local);
        launches++;
        int rc = nccl_api()->AllGather(rec_local, rec_all, sizeof(Red<T>), 0 /*ncclChar*/, comm, stream);
        if (rc != 0) { set_error("ncclAllGather failed: %d", rc); return false; }
        return true;
    }
    // the same for a merged record of the fast pipeline (kernels_dense.cuh: MSite)
    bool site_m(const MSite& ms) {
        if (R <= 1) return true;
        site_pending = true;
        if (p2p) { site_seq++; cur_slot = (int)(site_seq & 1ULL); }
        k_rank_finish_m<T><<<1, LB_SCALAR_THREADS, 0, stream>>>(w, ms, rec_local, peers, R, rank, cur_slot, site_seq, p2p ? 1 : 0);
        launches++;
        if (!p2p) {
            int rc = nccl_api()->AllGather(rec_local, rec_all, sizeof(Red<T>), 0 /*ncclChar*/, comm, stream);
            if (rc != 0) { set_error("ncclAllGather failed: %d", rc); return false; }
        }
        return true;
    }
#define LG LBFGSB_GRID, LBFGSB_BLOCK, 0, stream
#define LS 1, LB_SCALAR_THREADS, 0, stream
#define MTCALL(kern, smemfn, ...)                                                                          \
    do {                                                                                                   \
        if (mt == 5) kern<T, 5><<<LBFGSB_GRID, LB_TMA_THREADS, smemfn<T, 5>(), stream>>>(__VA_ARGS__);        \
        else if (mt == 10) kern<T, 10><<<LBFGSB_GRID, LB_TMA_THREADS, smemfn<T, 10>(), stream>>>(__VA_ARGS__); \
        else kern<T, 20><<<LBFGSB_GRID, LB_TMA_THREADS, smemfn<T, 20>(), stream>>>(__VA_ARGS__);              \
    } while (0)

    // fused passes exist only for the (T, MT) pairs whose accumulators fit in registers
    template <int MT> void launch_update_classify() {
        if constexpr (fused_passes_ok<T, MT>()) k_update_classify<T, MT><<<LBFGSB_GRID, LB_TMA_THREADS, smem_update_classify<T, MT>(), stream>>>(w);
    }
    template <int MT> void launch_formk_cmprlb() {
        if constexpr (fused_passes_ok<T, MT>()) k_formk_cmprlb<T, MT, 0><<<LBFGSB_GRID, LB_TMA_THREADS, smem_formk_cmprlb<T, MT>(), stream>>>(w);
    }
    template <int MT> void launch_formk_cmprlb_gf() {
        if constexpr (fused_passes_ok<T, MT>()) k_formk_cmprlb<T, MT, 1><<<LBFGSB_GRID, LB_TMA_THREADS, smem_formk_cmprlb<T, MT>(), stream>>>(w);
    }
    template <int MT> void launch_formk_cmprlb_gf2() {
        if constexpr (fused_passes_ok<T, MT>()) k_formk_cmprlb<T, MT, 2><<<LBFGSB_GRID, LB_TMA_THREADS, smem_formk_cmprlb<T, MT>(), stream>>>(w);
    }
    template <int MT> void launch_subsm_lsinit() {
        if constexpr (fused_passes_ok<T, MT>()) k_subsm_lsinit<T, MT, 0><<<LBFGSB_GRID, LB_TMA_THREADS, smem_subsm<T, MT>(), stream>>>(w);
    }
    template <int MT> void launch_subsm_dir() {
        if constexpr (fused_passes_ok<T, MT>()) k_subsm_lsinit<T, MT, 1><<<LBFGSB_GRID, LB_TMA_THREADS, smem_subsm<T, MT>(), stream>>>(w);
    }
#define MTFUSED(fn) do { if (mt == 5) fn<5>(); else if (mt == 10) fn<10>(); else fn<20>(); } while (0)

    // the TMA-staged kernels need more than the default 48 KB of dynamic shared memory
    template <int MT> bool set_smem_attrs() {
        CK(cudaFuncSetAttribute(k_update<T, MT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_update<T, MT>()));
        CK(cudaFuncSetAttribute(k_cauchy_classify<T, MT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_classify<T, MT>()));
        CK(cudaFuncSetAttribute(k_formk_gram<T, MT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_formk<T, MT>()));
        CK(cudaFuncSetAttribute(k_cmprlb_wv<T, MT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_cmprlb<T, MT>()));
        CK(cudaFuncSetAttribute(k_subsm_step<T, MT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_subsm<T, MT>()));
        if constexpr (fused_passes_ok<T, MT>()) {
            CK(cudaFuncSetAttribute(k_update_classify<T, MT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_update_classify<T, MT>()));
            CK(cudaFuncSetAttribute(k_formk_cmprlb<T, MT, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_formk_cmprlb<T, MT>()));
            CK(cudaFuncSetAttribute(k_formk_cmprlb<T, MT, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_formk_cmprlb<T, MT>()));
            CK(cudaFuncSetAttribute(k_formk_cmprlb<T, MT, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_formk_cmprlb<T, MT>()));
            CK(cudaFuncSetAttribute(k_subsm_lsinit<T, MT, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_subsm<T, MT>()));
            CK(cudaFuncSetAttribute(k_subsm_lsinit<T, MT, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_subsm<T, MT>()));
        }
        return true;
    }

    // ---- the breakpoint walk, in rounds over increasing ranges of t (cauchy_walk.cuh) -------
    static unsigned long long key_of(T t) {
        typename Real<T>::key_t k;
        memcpy(&k, &t, sizeof k);
        return (unsigned long long)k;
    }
    // One round over the breakpoints with keys in rg.  Returns 0: go on with the next range, 1: the search is
    // closed, 2: the exit fell inside a group of equal breakpoints and the round must be redone in heap order,
    // -1: error.
    int run_round(const BpRange& rg, bool first = false) {
        begin(F_WALK_COMPACT);
        // the first round of a cauchy call also writes d, xcp = x and every variable's breakpoint (cauchy_walk.cuh)
        if (first) k_bp_count<T, true><<<LG>>>(w, rg, tile_counts);
        else k_bp_count<T, false><<<LG>>>(w, rg, tile_counts);
        k_walk_round_local<T><<<1, 1024, 0, stream>>>(w, tile_counts, tile_offsets, ntiles, wb.ctl, rr_local);
        end(F_WALK_COMPACT, 2);
        if (R > 1 && !allgather(rr_local, rr_all, sizeof(RoundRec))) return -1;
        k_walk_round_begin<T><<<1, 32, 0, stream>>>(w, R > 1 ? rr_all : rr_local, R, n_global); launches++;
        if (!sync_state()) return -1;
        if (s_host->walk_closed) return 1;
        if (s_host->walk_rcount > 0) {
            begin(F_WALK_COMPACT); k_bp_write<T><<<LG>>>(w, rg, tile_counts, tile_offsets, wb.k0, wb.v0); end(F_WALK_COMPACT);
            begin(F_WALK_SORT); enqueue_sort(wb.k0, wb.k1, wb.v0, wb.v1, wb.ctl, s_host->walk_lcount); end(F_WALK_SORT, 0);
            if (R > 1) { if (!round_scan_sharded()) return -1; }
            else if (!round_scan_single(s_host->walk_lcount)) return -1;
            if (!sync_state()) return -1;
            if (s_host->walk_closed) return 1;
            if (s_host->tie_redo) return 2;
        }
        return 0;
    }
    // The exit fell inside the group of breakpoints equal to tie_key (single GPU): the round is redone up to
    // that group, then the group runs as a round of its own in the reference's heap order (cauchy_walk.cuh
    // "heap replay").  Returns like run_round.
    int tie_replay(const BpRange& rg) {
        if (R > 1) return tie_replay_sharded(rg);
        const unsigned long long tk = s_host->tie_key;
        k_tie_restore<T><<<1, 32, 0, stream>>>(w); launches++;
        if (tk > 0) {
            BpRange ra = rg; ra.hi = tk - 1;
            if (!(ra.lo_valid && ra.hi <= ra.lo)) {
                const int st = run_round(ra);
                if (st < 0) return -1;
                if (st != 0) { set_error("heap replay: the round below the tie group did not pass (internal error)"); return -1; }
            }
        }
        begin(F_WALK_COMPACT);
        k_flag_count<T, 2><<<LG>>>(w, tile_counts);
        k_tile_scan<T><<<1, 1024, 0, stream>>>(w, 2, tile_counts, tile_offsets, ntiles, wb.ctl);
        k_flag_write<T, 2><<<LG>>>(w, tile_counts, tile_offsets, wb.k0, wb.v0);
        end(F_WALK_COMPACT, 3);
        if (s_host->nbreak <= LB_TIE_DEVICE_MAX) {
            begin(F_WALK_SORT); k_heap_replay<T><<<1, 1024, 0, stream>>>(w, wb); end(F_WALK_SORT);
        } else if (!heap_replay_on_host(tk)) return -1;
        if (!sync_state()) return -1;
        tie_replays++;
        if (s_host->walk_lcount <= 0) { set_error("heap replay: empty tie group (internal error)"); return -1; }
        if (!round_scan_single(s_host->walk_lcount)) return -1;
        if (!sync_state()) return -1;
        return s_host->walk_closed ? 1 : 0;
    }
    // The same on a sharded workspace.  The heap's history involves every breakpoint of the call, so every rank gathers
    // all of them -- (t, global index), in variable order, exactly the reference's t / iorder arrays (:1305-1322) -- and
    // pops the same heap on its host thread; the members of the group, in pop order, then form a round of their own whose
    // sort keys are their positions in that order (tie_round = 2, walk_t_of): the sample sort, the exchange of the
    // records and the scans in rank order run unchanged, and every rank fixes those of its own members that were passed.
    DynBuf tie_k, tie_v, tie_kall, tie_vall;
    int tie_replay_sharded(const BpRange& rg) {
        typedef typename Real<T>::key_t K;
        const unsigned long long tk = s_host->tie_key;
        if (n_global >= 2147483647LL) { set_error("heap replay on a sharded workspace needs n < 2^31"); return -1; }
        k_tie_restore<T><<<1, 32, 0, stream>>>(w); launches++;
        if (tk > 0) {
            BpRange ra = rg; ra.hi = tk - 1;
            if (!(ra.lo_valid && ra.hi <= ra.lo)) {
                const int st = run_round(ra);
                if (st < 0) return -1;
                if (st != 0) { set_error("heap replay: the round below the tie group did not pass (internal error)"); return -1; }
            }
        }
        // this rank's breakpoints of the call, passed ones included, in variable order
        begin(F_WALK_COMPACT);
        k_flag_count<T, 2><<<LG>>>(w, tile_counts);
        k_tile_scan<T><<<1, 1024, 0, stream>>>(w, 2, tile_counts, tile_offsets, ntiles, wb.ctl);
        k_flag_write<T, 2><<<LG>>>(w, tile_counts, tile_offsets, wb.k0, wb.v0);
        end(F_WALK_COMPACT, 3);
        SortCtl hc;
        CK(cudaMemcpyAsync(&hc, wb.ctl, sizeof hc, cudaMemcpyDeviceToHost, stream));
        CK(cudaStreamSynchronize(stream)); syncs++;
        // counts and shard offsets of all ranks
        RoundRec mine; mine.count = hc.count; mine.rem = offset; mine.kmin = 0; mine.pad = 0;
        CK(cudaMemcpyAsync(rr_local, &mine, sizeof mine, cudaMemcpyHostToDevice, stream));
        if (!allgather(rr_local, rr_all, sizeof(RoundRec))) return -1;
        std::vector<RoundRec> recs((size_t)R);
        CK(cudaMemcpyAsync(recs.data(), rr_all, sizeof(RoundRec) * R, cudaMemcpyDeviceToHost, stream));
        CK(cudaStreamSynchronize(stream)); syncs++;
        i64 maxc = 0, nb = 0;
        for (int q = 0; q < R; ++q) { if (recs[q].count > maxc) maxc = recs[q].count; nb += recs[q].count; }
        if (nb <= 0) { set_error("heap replay: no breakpoints (internal error)"); return -1; }
        if (!ensure(tie_k, sizeof(K) * (size_t)maxc) || !ensure(tie_v, 4 * (size_t)maxc) ||
            !ensure(tie_kall, sizeof(K) * (size_t)maxc * R) || !ensure(tie_vall, 4 * (size_t)maxc * R)) return -1;
        CK(cudaMemcpyAsync(tie_k.p, wb.k0, sizeof(K) * (size_t)hc.count, cudaMemcpyDeviceToDevice, stream));
        CK(cudaMemcpyAsync(tie_v.p, wb.v0, 4 * (size_t)hc.count, cudaMemcpyDeviceToDevice, stream));
        if (!allgather(tie_k.p, tie_kall.p, sizeof(K) * (size_t)maxc) || !allgather(tie_v.p, tie_vall.p, 4 * (size_t)maxc)) return -1;
        std::vector<K> hk((size_t)nb); std::vector<int> hv((size_t)nb);
        {
            i64 o = 0;
            for (int q = 0; q < R; ++q) {
                const i64 c = recs[q].count;
                if (c > 0) {
                    CK(cudaMemcpyAsync(hk.data() + o, (K*)tie_kall.p + (size_t)q * maxc, sizeof(K) * (size_t)c, cudaMemcpyDeviceToHost, stream));
                    CK(cudaMemcpyAsync(hv.data() + o, (int*)tie_vall.p + (size_t)q * maxc, 4 * (size_t)c, cudaMemcpyDeviceToHost, stream));
                }
                o += c;
            }
            CK(cudaStreamSynchronize(stream)); syncs++;
            o = 0;
            for (int q = 0; q < R; ++q) {   // local -> global variable index (0-based); rem carries the shard offset
                for (i64 i = 0; i < recs[q].count; ++i) hv[(size_t)(o + i)] += (int)recs[q].rem;
                o += recs[q].count;
            }
        }
        std::vector<K> gk; std::vector<int> gv;
        heap_group_order((K)tk, hk, hv, (int)s_host->ibkmin, gk, gv);
        // this rank's members: key = position in the pop order, value = local variable
        std::vector<K> lk; std::vector<int> lv;
        const i64 g = (i64)gv.size();
        // REAL32: the position travels as a real in the exchanged record, exact below 2^24 -- a larger group is taken in
        // variable order (what happens beyond the replay limit)
        if (sizeof(T) == 4 && g >= ((i64)1 << 24)) std::sort(gv.begin(), gv.end());
        for (i64 ppos = 0; ppos < g; ++ppos) {
            const i64 gi = gv[(size_t)ppos];
            if (gi >= offset && gi < offset + n) { lk.push_back((K)ppos); lv.push_back((int)(gi - offset)); }
        }
        const i64 cnt = (i64)lk.size();
        if (cnt > 0) {
            CK(cudaMemcpyAsync(wb.k1, lk.data(), sizeof(K) * (size_t)cnt, cudaMemcpyHostToDevice, stream));
            CK(cudaMemcpyAsync(wb.v1, lv.data(), sizeof(int) * (size_t)cnt, cudaMemcpyHostToDevice, stream));
        }
        k_heap_replay_commit<T><<<1, 32, 0, stream>>>(w, wb, cnt, g, 2); launches++;
        CK(cudaStreamSynchronize(stream));   // lk, lv are locals
        if (!sync_state()) return -1;
        tie_replays++;
        if (g <= 0) { set_error("heap replay: empty tie group (internal error)"); return -1; }
        if (!round_scan_sharded()) return -1;
        if (!sync_state()) return -1;
        return s_host->walk_closed ? 1 : 0;
    }
    // hpsolb's pop order of the group of breakpoints equal to tk: hk / hv hold every breakpoint of the cauchy call in variable
    // order (destroyed), vmin the variable of the first minimum (taken before the heap exists, :1384-1397)
    template <typename K>
    static void heap_group_order(K tk, std::vector<K>& hk, std::vector<int>& hv, int vmin, std::vector<K>& gk, std::vector<int>& gv) {
        const i64 nb = (i64)hk.size();
        i64 spos = -1;
        for (i64 i = 0; i < nb; ++i) if (hv[(size_t)i] == vmin) spos = i;
        if (spos >= 0 && hk[(size_t)spos] == tk) { gk.push_back(tk); gv.push_back(vmin); }
        K* t = hk.data() - 1; int* io = hv.data() - 1;   // 1-based
        const i64 ib = spos + 1;
        if (ib >= 1 && ib != nb) { t[ib] = t[nb]; io[ib] = io[nb]; }   // :1394-1397
        i64 nleft = nb - 1;
        heap_build<K>(t, io, nleft);
        while (nleft > 0) {
            K out; int var;
            heap_pop<K>(t, io, nleft, out, var);
            nleft--;
            if (out > tk) break;
            if (out == tk) { gk.push_back(out); gv.push_back(var); }
        }
    }
    // hpsolb's pop order of the group of breakpoints equal to tk, on the host (cauchy_walk.cuh "heap replay"): wb.k0 / wb.v0
    // hold every breakpoint of this cauchy call in variable order.  The reference pays the same sequential heap.
    bool heap_replay_on_host(unsigned long long tk64) {
        typedef typename Real<T>::key_t K;
        SortCtl hc;
        CK(cudaMemcpyAsync(&hc, wb.ctl, sizeof hc, cudaMemcpyDeviceToHost, stream));
        CK(cudaStreamSynchronize(stream)); syncs++;
        const i64 nb = hc.count;
        if (nb <= 0) { set_error("heap replay: no breakpoints (internal error)"); return false; }
        std::vector<K> hk((size_t)nb); std::vector<int> hv((size_t)nb);
        CK(cudaMemcpyAsync(hk.data(), wb.k0, sizeof(K) * (size_t)nb, cudaMemcpyDeviceToHost, stream));
        CK(cudaMemcpyAsync(hv.data(), wb.v0, sizeof(int) * (size_t)nb, cudaMemcpyDeviceToHost, stream));
        CK(cudaStreamSynchronize(stream));
        std::vector<K> gk; std::vector<int> gv;
        heap_group_order((K)tk64, hk, hv, (int)(s_host->ibkmin - offset), gk, gv);
        const i64 cnt = (i64)gk.size();
        if (cnt > 0) {
            CK(cudaMemcpyAsync(wb.k1, gk.data(), sizeof(K) * (size_t)cnt, cudaMemcpyHostToDevice, stream));
            CK(cudaMemcpyAsync(wb.v1, gv.data(), sizeof(int) * (size_t)cnt, cudaMemcpyHostToDevice, stream));
        }
        k_heap_replay_commit<T><<<1, 32, 0, stream>>>(w, wb, cnt, cnt, 1); launches++;
        CK(cudaStreamSynchronize(stream));   // gk, gv are locals
        return true;
    }
    // ---- the breakpoint walk, in rounds over increasing ranges of t (cauchy_walk.cuh) -------
    bool enqueue_walk_rounds() {
        const T dtm0 = s_host->dtm;          // minimiser of the first segment (s_cauchy); dtm0 >= bkmin here
        unsigned long long his[3];
        int nr = 0;
        if (dtm0 > (T)0 && dtm0 < (T)INFINITY) {
            const T t1 = (T)2 * dtm0, t2 = (T)16 * dtm0;
            if (t1 < (T)INFINITY) his[nr++] = key_of(t1);
            if (t2 < (T)INFINITY) his[nr++] = key_of(t2);
        }
        his[nr++] = 0xffffffffffffffffULL;
        BpRange rg; rg.lo = 0; rg.lo_valid = 0; rg.hi = 0;
        bool first = true;
        for (int r = 0; r < nr;) {
            rg.hi = his[r];
            if (rg.lo_valid && rg.hi <= rg.lo) { ++r; continue; }
            int st = run_round(rg, first && !w.bp_hint);
            first = false;
            if (st < 0) return false;
            if (st == 1) break;
            if (st == 2) {
                const unsigned long long tk = s_host->tie_key;
                st = tie_replay(rg);
                if (st < 0) return false;
                if (st == 1) break;
                rg.lo = tk; rg.lo_valid = 1;   // the whole group was passed: the rest of this range follows
                continue;
            }
            rg.lo = rg.hi; rg.lo_valid = 1; ++r;
        }
        if (!s_host->walk_closed) { set_error("the breakpoint walk did not close (internal error)"); return false; }
        return true;
    }
    // scans of one round's sorted list on a single GPU
    bool round_scan_single(i64 count) {
        begin(F_WALK_SCAN);
        for (i64 start = 0; start < count; start += wb.cap) {
            const i64 len = (count - start < wb.cap) ? (count - start) : wb.cap;
            const i64 nblk = (len + LB_WB - 1) / LB_WB;
            CK(cudaMemsetAsync(jmin, 0xff, 8, stream));
            k_walk_gather<T><<<(unsigned)nblk, LB_WB, 0, stream>>>(w, wb, start, len);
            k_walk_scan_vec<T><<<1, 1024, 0, stream>>>(w, wb, nblk, tmpAB);
            k_walk_dots<T><<<(unsigned)nblk, LB_WB, 0, stream>>>(w, wb, start, len);
            k_walk_scan_f2<T><<<1, 32, 0, stream>>>(w, wb, nblk, tmpF);
            k_walk_f2<T><<<(unsigned)nblk, LB_WB, 0, stream>>>(w, wb, start, len);
            k_walk_scan_f1<T><<<1, 32, 0, stream>>>(w, wb, nblk, tmpF);
            k_walk_test<T><<<(unsigned)nblk, LB_WB, 0, stream>>>(w, wb, start, len, jmin);
            k_walk_chunk_end<T><<<1, 32, 0, stream>>>(w, wb, start, len, tmpAB, tmpF, jmin);
            launches += 8;
        }
        k_walk_round_end<T><<<1, LB_WB, 0, stream>>>(w, wb, n_global, R == 1 ? 1 : 0);
        end(F_WALK_SCAN, 1);
        begin(F_WALK_FIX);
        k_walk_fix<T><<<LBFGSB_GRID, 256, 0, stream>>>(w, wb);
        end(F_WALK_FIX);
        return true;
    }

    // ---- the breakpoint walk on a sharded problem (cauchy_walk_dist.cuh) -----
    bool ensure(DynBuf& d, size_t bytes) {
        if (bytes == 0) bytes = 16;
        if (d.cap >= bytes) return true;
        if (d.p) cudaFree(d.p);
        d.p = nullptr; d.cap = 0;
        const size_t want = bytes + bytes / 8;
        cudaError_t e = cudaMalloc(&d.p, want);
        if (e != cudaSuccess) { set_error("cudaMalloc(%zu) failed in the sharded breakpoint walk: %s", want, cudaGetErrorString(e)); return false; }
        d.cap = want;
        return true;
    }
    bool allgather(const void* src, void* dst, size_t bytes) {
        int rc = nccl_api()->AllGather(src, dst, bytes, 0 /*ncclChar*/, comm, stream);
        if (rc != 0) { set_error("ncclAllGather failed: %d", rc); return false; }
        return true;
    }
    // `count` = number of items (what ctl->count holds on the device): sizes the grid
    static int sort_blocks(i64 count) {
        i64 nb = (count + 2 * LB_RS_TILE - 1) / (2 * LB_RS_TILE);
        return (int)(nb < 1 ? 1 : (nb > LB_RS_GRID ? LB_RS_GRID : nb));
    }
    void enqueue_sort(typename Real<T>::key_t* k0, typename Real<T>::key_t* k1, int* v0, int* v1, SortCtl* ctl, i64 count) {
        typedef typename Real<T>::key_t K;
        if (count <= LB_SMALL_SORT_MAX) {   // (count = ctl->count: the callers pass what the device holds)
            k_small_sort<K><<<1, 1024, 0, stream>>>(k0, k1, v0, v1, ctl); launches++;
            return;
        }
        const int nblk = sort_blocks(count);
        for (int pass = 0; pass < (int)sizeof(K); ++pass) {
            k_rs_hist<K><<<nblk, 256, 0, stream>>>(k0, k1, ctl, pass * 8, rs_counts);
            k_rs_scan<<<1, 1024, 0, stream>>>(rs_counts, ctl, nblk);
            k_rs_scatter<K><<<nblk, 256, 0, stream>>>(k0, k1, v0, v1, ctl, pass * 8, rs_counts);
            k_rs_flip<<<1, 32, 0, stream>>>(ctl);
            launches += 4;
        }
    }
    // a small round on a sharded problem (cauchy_walk_dist.cuh "Small rounds"): every rank scans the whole gathered list
    bool round_scan_gathered(i64 total) {
        typedef typename Real<T>::key_t K;
        const int col = s_host->col;
        const int rs = 3 + 2 * col;
        const i64 cap = (total + 63) / 64 * 64;   // >= every rank's count of the round
        if (!ensure(dw_send, sizeof(T) * (size_t)cap * rs) || !ensure(dw_recv, sizeof(T) * (size_t)cap * rs * R)) return false;
        if (!ensure(dw_k0, sizeof(K) * (size_t)total) || !ensure(dw_k1, sizeof(K) * (size_t)total) ||
            !ensure(dw_v0, 4 * (size_t)total) || !ensure(dw_v1, 4 * (size_t)total)) return false;
        begin(F_WALK_SCAN);
        k_rw_count<T><<<1, 32, 0, stream>>>(w, wb, rr_local); launches++;
        if (!allgather(rr_local, rr_all, sizeof(RoundRec))) return false;
        T* send = (T*)dw_send.p; T* recv = (T*)dw_recv.p;
        k_dw_pack<T><<<LBFGSB_GRID, 256, 0, stream>>>(w, wb, send, rs); launches++;
        if (!allgather(send, recv, sizeof(T) * (size_t)cap * rs)) return false;
        WalkBuf<T> wd = wb;
        wd.k0 = (K*)dw_k0.p; wd.k1 = (K*)dw_k1.p; wd.v0 = (int*)dw_v0.p; wd.v1 = (int*)dw_v1.p; wd.ctl = ctl_d;
        k_rw_keys<T><<<32, 256, 0, stream>>>(recv, rs, cap, rr_all, R, wd.k0, wd.v0, ctl_d); launches++;
        enqueue_sort(wd.k0, wd.k1, wd.v0, wd.v1, ctl_d, total);
        for (i64 start = 0; start < total; start += wd.cap) {
            const i64 len = (total - start < wd.cap) ? (total - start) : wd.cap;
            const i64 nblk = (len + LB_WB - 1) / LB_WB;
            CK(cudaMemsetAsync(jmin, 0xff, 8, stream));
            k_dw_gather<T><<<(unsigned)nblk, LB_WB, 0, stream>>>(w, wd, recv, rs, start, len);
            k_walk_scan_vec<T><<<1, 1024, 0, stream>>>(w, wd, nblk, tmpAB);
            k_walk_dots<T><<<(unsigned)nblk, LB_WB, 0, stream>>>(w, wd, start, len);
            k_walk_scan_f2<T><<<1, 32, 0, stream>>>(w, wd, nblk, tmpF);
            k_walk_f2<T><<<(unsigned)nblk, LB_WB, 0, stream>>>(w, wd, start, len);
            k_walk_scan_f1<T><<<1, 32, 0, stream>>>(w, wd, nblk, tmpF);
            k_walk_test<T><<<(unsigned)nblk, LB_WB, 0, stream>>>(w, wd, start, len, jmin);
            k_walk_chunk_end<T><<<1, 32, 0, stream>>>(w, wd, start, len, tmpAB, tmpF, jmin);
            launches += 8;
        }
        k_walk_round_end<T><<<1, LB_WB, 0, stream>>>(w, wd, n_global, 1);
        end(F_WALK_SCAN, 1);
        begin(F_WALK_FIX);
        k_rw_fix<T><<<64, 256, 0, stream>>>(w, wb, wd, cap, rank);
        end(F_WALK_FIX);
        return true;
    }
    // one round on a sharded problem: this rank's breakpoints of the round are sorted in wb
    bool round_scan_sharded() {
        typedef typename Real<T>::key_t K;
        if (s_host->walk_rcount > 0 && s_host->walk_rcount <= LB_RW_MAX) return round_scan_gathered(s_host->walk_rcount);
        const int S = LB_DW_SAMPLES;
        // 2. splitters from regular samples
        begin(F_WALK_SCAN);
        k_dw_sample<T><<<1, 64, 0, stream>>>(w, wb, samp_local); launches++;
        const size_t sbytes = sizeof(unsigned long long) * (2 * S + 1);
        if (!allgather(samp_local, samp_all, sbytes)) return false;
        std::vector<unsigned long long> hs((size_t)(2 * S + 1) * R);
        CK(cudaMemcpyAsync(hs.data(), samp_all, sbytes * R, cudaMemcpyDeviceToHost, stream));
        CK(cudaStreamSynchronize(stream)); syncs++;
        std::vector<std::pair<unsigned long long, i64>> smp;
        for (int q = 0; q < R; ++q)
            for (int i = 0; i < S; ++i) smp.push_back({hs[(size_t)q * (2 * S + 1) + i], (i64)hs[(size_t)q * (2 * S + 1) + S + i]});
        std::sort(smp.begin(), smp.end());
        std::vector<unsigned long long> spl(2 * (R - 1));
        for (int q = 1; q < R; ++q) { spl[q - 1] = smp[(size_t)q * S].first; spl[(R - 1) + (q - 1)] = (unsigned long long)smp[(size_t)q * S].second; }
        CK(cudaMemcpyAsync(spl_dev, spl.data(), sizeof(unsigned long long) * 2 * (R - 1), cudaMemcpyHostToDevice, stream));
        k_dw_partition<T><<<1, 32, 0, stream>>>(w, wb, R, spl_dev, dctl); launches++;
        if (!allgather(dctl->pos, pos_all, sizeof(i64) * (LB_MAXR + 1))) return false;
        std::vector<i64> hp((size_t)(LB_MAXR + 1) * R);
        CK(cudaMemcpyAsync(hp.data(), pos_all, sizeof(i64) * (LB_MAXR + 1) * R, cudaMemcpyDeviceToHost, stream));
        CK(cudaStreamSynchronize(stream)); syncs++;
        // 3. exchange plan: cnt(q -> r) = pos_q[r+1] - pos_q[r]
        auto cnt = [&](int q, int r) { return hp[(size_t)q * (LB_MAXR + 1) + r + 1] - hp[(size_t)q * (LB_MAXR + 1) + r]; };
        DwCtl hc; memset(&hc, 0, sizeof hc);
        for (int r = 0; r <= R; ++r) hc.pos[r] = hp[(size_t)rank * (LB_MAXR + 1) + r];
        i64 nrecv = 0;
        for (int q = 0; q < R; ++q) { hc.roff[q] = nrecv; nrecv += cnt(q, rank); }
        hc.roff[R] = nrecv;
        i64 nb_glob = 0, goff = 0;
        for (int r = 0; r < R; ++r) {
            i64 t = 0;
            for (int q = 0; q < R; ++q) t += cnt(q, r);
            if (r < rank) goff += t;
            nb_glob += t;
        }
        hc.goff = goff; hc.nb_glob = nb_glob;
        if (nrecv > 2147483647LL) { set_error("a rank would receive more than 2^31 breakpoints"); return false; }
        const i64 nb_loc = hc.pos[R];
        const int col = s_host->col;
        const int rs = 3 + 2 * col;
        if (!ensure(dw_send, sizeof(T) * (size_t)nb_loc * rs) || !ensure(dw_recv, sizeof(T) * (size_t)nrecv * rs)) return false;
        if (!ensure(dw_k0, sizeof(K) * (size_t)nrecv) || !ensure(dw_k1, sizeof(K) * (size_t)nrecv) ||
            !ensure(dw_v0, 4 * (size_t)nrecv) || !ensure(dw_v1, 4 * (size_t)nrecv)) return false;
        CK(cudaMemcpyAsync(dctl, &hc, sizeof hc, cudaMemcpyHostToDevice, stream));
        CK(cudaStreamSynchronize(stream));   // hc is a stack object
        T* send = (T*)dw_send.p; T* recv = (T*)dw_recv.p;
        k_dw_pack<T><<<LBFGSB_GRID, 256, 0, stream>>>(w, wb, send, rs); launches++;
        nccl_api()->GroupStart();
        for (int q = 0; q < R; ++q) {
            const i64 sc = cnt(rank, q), rc = cnt(q, rank);
            if (q == rank) {
                if (sc > 0) CK(cudaMemcpyAsync(recv + hc.roff[q] * rs, send + hc.pos[q] * rs, sizeof(T) * (size_t)sc * rs, cudaMemcpyDeviceToDevice, stream));
                continue;
            }
            if (sc > 0) nccl_api()->Send(send + hc.pos[q] * rs, sizeof(T) * (size_t)sc * rs, 0, q, comm, stream);
            if (rc > 0) nccl_api()->Recv(recv + hc.roff[q] * rs, sizeof(T) * (size_t)rc * rs, 0, q, comm, stream);
        }
        int grc = nccl_api()->GroupEnd();
        if (grc != 0) { set_error("nccl send/recv group failed: %d", grc); return false; }
        // 4. this rank's key range in global order
        WalkBuf<T> wd = wb;
        wd.k0 = (K*)dw_k0.p; wd.k1 = (K*)dw_k1.p; wd.v0 = (int*)dw_v0.p; wd.v1 = (int*)dw_v1.p; wd.ctl = ctl_d;
        k_dw_keys<T><<<LBFGSB_GRID, 256, 0, stream>>>(recv, rs, nrecv, wd.k0, wd.v0, ctl_d); launches++;
        enqueue_sort(wd.k0, wd.k1, wd.v0, wd.v1, ctl_d, nrecv);
        // 5. scans in rank order, carries handed from rank to rank
        for (int turn = 0; turn < R; ++turn) {
            if (turn == rank) {
                for (i64 start = 0; start < nrecv; start += wd.cap) {
                    const i64 len = (nrecv - start < wd.cap) ? (nrecv - start) : wd.cap;
                    const i64 nblk = (len + LB_WB - 1) / LB_WB;
                    CK(cudaMemsetAsync(jmin, 0xff, 8, stream));
                    k_dw_gather<T><<<(unsigned)nblk, LB_WB, 0, stream>>>(w, wd, recv, rs, start, len);
                    k_walk_scan_vec<T><<<1, 1024, 0, stream>>>(w, wd, nblk, tmpAB);
                    k_walk_dots<T><<<(unsigned)nblk, LB_WB, 0, stream>>>(w, wd, start, len);
                    k_walk_scan_f2<T><<<1, 32, 0, stream>>>(w, wd, nblk, tmpF);
                    k_walk_f2<T><<<(unsigned)nblk, LB_WB, 0, stream>>>(w, wd, start, len);
                    k_walk_scan_f1<T><<<1, 32, 0, stream>>>(w, wd, nblk, tmpF);
                    k_walk_test<T><<<(unsigned)nblk, LB_WB, 0, stream>>>(w, wd, start, len, jmin);
                    k_walk_chunk_end<T><<<1, 32, 0, stream>>>(w, wd, start, len, tmpAB, tmpF, jmin);
                    launches += 8;
                }
                k_dw_fixcount<T><<<LBFGSB_GRID, 256, 0, stream>>>(w, wd, R, dctl); launches++;
            }
            k_dw_turn_end<T><<<1, LB_WB, 0, stream>>>(w, wd, dctl, wd.cap, turn == rank ? 1 : 0, R, carry_local); launches++;
            if (!allgather(carry_local, carry_all, sizeof(WalkCarry<T>))) return false;
            k_dw_adopt<T><<<1, 32, 0, stream>>>(w, carry_all, turn, R, rank, dctl, n_global); launches++;
        }
        end(F_WALK_SCAN, 0);
        // 6. fix the local variables that precede the exit
        begin(F_WALK_FIX);
        k_dw_fix<T><<<LBFGSB_GRID, 256, 0, stream>>>(w, wb, dctl);
        end(F_WALK_FIX);
        return true;
    }

    // ---- prelims + first lnsrlb (:601-773): the general pipeline -------------------------------
    // `from` = where to enter: PAUSE_NONE for the whole body, or the stage at which the fast pipeline paused
    // (common.cuh PAUSE_*; the device state is then exactly what this sequence would have produced up to there,
    // and s_host is current).
    bool enqueue_body(int from = PAUSE_NONE) {
        body_ran = true;
        for (;;) {
            bool gf = false;   // cauchy's tail and freev run inside k_formk_cmprlb (decided by s_cauchy)
            bool gf2 = false;  // ... after a breakpoint walk (s_walk_gf)
            if (from <= PAUSE_CLASSIFY) {
                phase(PH_CAUCHY);
                begin(F_CLASSIFY); MTCALL(k_cauchy_classify, smem_classify, w); end(F_CLASSIFY);
                if (!site(site_cauchy(mt))) return false;
                begin(F_SCALAR); s_cauchy<T><<<LS>>>(w, dist(), mt, fused ? 1 : 0); end(F_SCALAR);
            }
            if (from <= PAUSE_WALK) {
                if (s_host->cnstnd) {
                    if (from != PAUSE_WALK && !sync_state()) return false;
                    if (s_host->go && s_host->in_body && s_host->need_walk) {
                        walked_now = true;
                        if (!enqueue_walk_rounds()) return false;   // (its first count pass writes xcp and the breakpoints)
                        // the walk has closed: a = M c, and the cauchy tail + freev move into k_formk_cmprlb (fuse_gf = 2) --
                        // unless that product fails, which the host does not wait to learn: both variants are enqueued
                        if (fused && walk_gf_ok) { begin(F_SCALAR); s_walk_gf<T><<<LS>>>(w, 1); end(F_SCALAR); gf2 = true; }
                    }
                    gf = fused && s_host->go && s_host->in_body && s_host->fuse_gf;
                }
            }
            if (from <= PAUSE_GCP_FREEV) {
                phase(PH_SUBSPACE);
                if (!gf) {
                    begin(F_GCP_FREEV); k_gcp_freev<T><<<LG>>>(w); end(F_GCP_FREEV);   // (returns at once under fuse_gf = 2)
                    if (!site(site_freev())) return false;
                }
                begin(F_SCALAR); s_freev<T><<<LS>>>(w, dist(), n_global, 0); end(F_SCALAR);
                if (fused) {
                    begin(F_FORMK_CMPRLB);
                    if (gf) MTFUSED(launch_formk_cmprlb_gf);
                    else { if (gf2) { MTFUSED(launch_formk_cmprlb_gf2); launches++; } MTFUSED(launch_formk_cmprlb); }
                    end(F_FORMK_CMPRLB);
                }
                else { begin(F_FORMK_GRAM); MTCALL(k_formk_gram, smem_formk, w); end(F_FORMK_GRAM); }
                if (gf || gf2) {
                    if (!site(site_freev())) return false;
                    begin(F_SCALAR); s_freev<T><<<LS>>>(w, dist(), n_global, 1); end(F_SCALAR);
                }
            }
            if (from <= PAUSE_DELTA) {
                if (from == PAUSE_DELTA) phase(PH_SUBSPACE);
                begin(F_FORMK_DELTA);
                k_el_count<T><<<LG>>>(w, tile_counts);
                k_tile_scan<T><<<1, 1024, 0, stream>>>(w, 1, tile_counts, tile_offsets, ntiles, ctl_el);
                k_flag_write<T, 1><<<LG>>>(w, tile_counts, tile_offsets, wb.k0, wb.v0);
                k_formk_delta<T><<<fd_grid<T>(), 256, 0, stream>>>(w, wb.v0, ctl_el, fd_parts);
                k_formk_delta_final<T><<<(6 * LB_MMAX * LB_MMAX + 255) / 256, 256, 0, stream>>>(w, fd_parts, fd_grid<T>(), delta);
                end(F_FORMK_DELTA, 5);
                if (!site(site_formk(mt))) return false;
                if (R > 1) {
                    if (p2p) { delta_seq++; k_delta_push<T><<<1, 256, 0, stream>>>(w, delta, peers_delta, peers, R, rank, delta_seq); launches++; }
                    else if (!allgather(delta, delta_all, sizeof(T) * 6 * LB_MMAX * LB_MMAX)) return false;
                }
                begin(F_SCALAR); s_formk_dense<T><<<LS>>>(w, dist(), mt, R > 1 ? delta_all : delta, delta_sum); end(F_SCALAR);
                if (!fused) { begin(F_CMPRLB_WV); MTCALL(k_cmprlb_wv, smem_cmprlb, w); end(F_CMPRLB_WV); }
                if (!site(site_wv(mt))) return false;
                begin(F_SCALAR); s_subsm_dense<T><<<LS>>>(w, dist(), mt, fused ? 1 : 0); end(F_SCALAR);
                if (fused) { begin(F_SUBSM_LSINIT); MTFUSED(launch_subsm_lsinit); end(F_SUBSM_LSINIT); }
                else { begin(F_SUBSM_STEP); MTCALL(k_subsm_step, smem_subsm, w); end(F_SUBSM_STEP); }
                if (!site(site_subsm())) return false;
                begin(F_SCALAR); s_subsm_post<T><<<LS>>>(w, dist(), fused ? 1 : 0); end(F_SCALAR);
            }
            if (from <= PAUSE_BACKTRACK) {
                if (from == PAUSE_BACKTRACK) phase(PH_SUBSPACE);
                begin(F_BACKTRACK);
                if (fused) { MTFUSED(launch_subsm_dir); launches++; }   // direction for the backtrack after a speculative step
                k_bt_alpha<T><<<LG>>>(w);
                if (!site(site_bt())) return false;
                s_bt<T><<<LS>>>(w, dist(), offset);
                k_bt_apply<T><<<LG>>>(w);
                end(F_BACKTRACK, 3);
            }
            phase(PH_LNSRCH);
            begin(F_LS_INIT); k_ls_init<T><<<LG>>>(w); end(F_LS_INIT);
            if (!site(site_lsinit())) return false;
            begin(F_SCALAR); s_ls_init<T><<<LS>>>(w, dist()); end(F_SCALAR);
            begin(F_LS_STEP); k_ls_step<T><<<LG>>>(w); end(F_LS_STEP);
            phase(PH_END);
            if (!sync_state()) return false;
            if (s_host->do_step) x_changed = true;
            if (!s_host->restart) break;
            // "refresh the lbfgs memory and restart the iteration": run the prelims again
            begin(F_SCALAR); s_restart_body<T><<<1, 32, 0, stream>>>(w); end(F_SCALAR);
            from = PAUSE_NONE;
        }
        return true;
    }

    // ---- NEW_X entry, fast pipeline (kernels_dense.cuh "Fast pipeline") ---------------------------------
    // Three streaming passes and four scalar kernels with one host read-back at the end; any branch off the
    // common path pauses the sequence on the device and the general pipeline takes over at that stage.
    bool fast = false;
    bool fast_newx(T f) {
        begin(F_SCALAR); f_head<T><<<1, 32, 0, stream>>>(w, f, 1); end(F_SCALAR);
        phase(PH_CAUCHY);
        begin(F_UPDATE_CLASSIFY); MTFUSED(launch_update_classify); end(F_UPDATE_CLASSIFY);
        if (!site_m(msite_ucf(mt))) return false;
        begin(F_SCALAR); f_ucf<T><<<LS>>>(w, dist(), mt); end(F_SCALAR);
        const size_t ev_ucf = pending.size();
        phase(PH_SUBSPACE);
        begin(F_FORMK_CMPRLB); MTFUSED(launch_formk_cmprlb_gf); end(F_FORMK_CMPRLB);
        if (!site_m(msite_mid(mt))) return false;
        begin(F_SCALAR); f_mid<T><<<LS>>>(w, dist(), mt, n_global); end(F_SCALAR);
        const size_t ev_mid = pending.size();
        begin(F_SUBSM_LSINIT); MTFUSED(launch_subsm_lsinit); end(F_SUBSM_LSINIT);
        if (!site_m(msite_tail())) return false;
        phase(PH_LNSRCH);
        begin(F_SCALAR); f_tail<T><<<LS>>>(w, dist()); end(F_SCALAR);
        phase(PH_END);
        if (!sync_state(false)) return false;
        if (profile) {
            const int ps = s_host->pause;
            if (ps == PAUSE_CLASSIFY || ps == PAUSE_WALK || ps == PAUSE_GCP_FREEV) drop_events_from(ev_ucf);
            else if (ps == PAUSE_DELTA || ps == PAUSE_LSINIT) drop_events_from(ev_mid);
            resolve_events();
        }
        return finish_call(false);
    }
    i64 fast_pauses = 0;

    // The rest of a setulb call after its last read-back, from the state header in s_host: the general pipeline from
    // where the fast one paused, the restored iterate, the body again after a restart, or lnsrlb's pending trial point.
    // `stepped`: k_ls_step was already enqueued behind the read-back (the iteration graph) and took the step or unstep.
    bool finish_call(bool stepped) {
        if (s_host->pause != PAUSE_NONE) {
            const int from = s_host->pause;
            fast_pauses++;
            s_resume<T><<<1, 32, 0, stream>>>(w); launches++;
            return enqueue_body(from);
        }
        if (s_host->do_restore) {
            begin(F_RESTORE); k_restore<T><<<LG>>>(w); end(F_RESTORE);
            CK(cudaStreamSynchronize(stream));
            if (profile) resolve_events();
            x_changed = true; g_changed = true;
        }
        if (s_host->restart) {
            // lnsrlb met an ascent direction at its first entry (:2247-2253) after the subspace pass had stepped
            // speculatively: x = t again before the iteration restarts (s_restart_body clears the flag)
            if (s_host->do_unstep && !stepped) { begin(F_LS_STEP); k_ls_step<T><<<LG>>>(w); end(F_LS_STEP); }
            begin(F_SCALAR); s_restart_body<T><<<1, 32, 0, stream>>>(w); end(F_SCALAR);
            return enqueue_body();
        }
        if (stepped) return true;
        // lnsrlb's trial point: nothing to do when the subspace pass already stepped
        if (s_host->do_unstep || (s_host->do_step && !s_host->step_done)) {
            begin(F_LS_STEP); k_ls_step<T><<<LG>>>(w); end(F_LS_STEP);
            CK(cudaStreamSynchronize(stream));
            if (profile) resolve_events();
        }
        if (s_host->do_step) x_changed = true;
        return true;
    }

    // ---- device-resident iteration: the caller's loop as one CUDA graph per step (kernels_dense.cuh g_ls_trial / g_head) ----
    // Graph = [objective kernels -> g, f_dev] [k_ls_trial, g_ls_trial: FG_LNSRCH entry] [g_head .. f_tail: NEW_X entry, fast
    // pipeline] [k_ls_step: the next trial point] [k_publish].  One launch and one read-back per step; whatever the fast
    // pipeline does not cover (pause, restart, restore) is finished by the general pipeline on the host, as in call().
    cudaGraphExec_t iter_graph = nullptr;
    T* f_dev = nullptr;   // f of the objective callback of minimize_graph
    i64 graph_launches_per_step = 0, graph_steps = 0;
    template <typename FGE>
    bool build_iter_graph(FGE fg, void* user, int max_iter, int max_fg) {
        if (iter_graph) { cudaGraphExecDestroy(iter_graph); iter_graph = nullptr; }
        w.bp_hint = 0;
        cudaGraph_t graph = nullptr;
        CK(cudaStreamBeginCapture(stream, cudaStreamCaptureModeRelaxed));
        int rc = fg(user, n, w.x, w.g, f_dev, (void*)stream);
        k_ls_trial<T><<<LG>>>(w);
        g_ls_trial<T><<<LS>>>(w, dist(), f_dev);
        g_head<T><<<1, 32, 0, stream>>>(w, 1, max_iter, max_fg);
        MTFUSED(launch_update_classify);
        f_ucf<T><<<LS>>>(w, dist(), mt);
        MTFUSED(launch_formk_cmprlb_gf);
        f_mid<T><<<LS>>>(w, dist(), mt, n_global);
        MTFUSED(launch_subsm_lsinit);
        f_tail<T><<<LS>>>(w, dist());
        k_ls_step<T><<<LG>>>(w);
        enqueue_publish();
        graph_launches_per_step = 11;
        cudaError_t ce = cudaStreamEndCapture(stream, &graph);
        if (rc != 0 || ce != cudaSuccess || !graph) {
            if (graph) cudaGraphDestroy(graph);
            cudaGetLastError();
            set_error("the objective callback could not be captured in a CUDA graph (%s)", rc != 0 ? "callback failed" : cudaGetErrorString(ce));
            return false;
        }
        ce = cudaGraphInstantiate(&iter_graph, graph, 0);
        cudaGraphDestroy(graph);
        if (ce != cudaSuccess) { set_error("cudaGraphInstantiate failed: %s", cudaGetErrorString(ce)); iter_graph = nullptr; return false; }
        return true;
    }
    // one step of the device-resident loop; the state block is current in s_host afterwards
    bool graph_step() {
        CK(cudaGraphLaunch(iter_graph, stream));
        launches += graph_launches_per_step; graph_steps++;
        if (!wait_published()) return false;
        // what call() does after its read-back, for the call that ran last inside the graph
        for (auto& mk : marks) pool.push_back(mk.e);
        marks.clear();
        walked_now = false; body_ran = false;
        if (!finish_call(true)) return false;
        resolve_phases();
        return check_launch();
    }

    bool check_launch() {
        cudaError_t e = cudaGetLastError();
        if (e != cudaSuccess) { set_error("kernel launch failed: %s", cudaGetErrorString(e)); return false; }
        return true;
    }

    // ---- one setulb call (device pointers) ----------------------------------
    // entry: 0 START, 1 FG_START, 2 FG_LNSRCH, 3 NEW_X, 4 STOP (cpu restore flag in aux), 5 other
    bool call(int entry, int aux, T* x, const T* l, const T* u, const int* nbd, T* f, T* g, T factr, T pgtol) {
        w.x = x; w.l = l; w.u = u; w.nbd = nbd; w.g = g;
        w.bp_hint = (entry == 3 && walked_prev && bp_hint_ok) ? 1 : 0;
        walked_now = false; body_ran = false;
        x_changed = false; g_changed = false;
        for (auto& mk : marks) pool.push_back(mk.e);
        marks.clear();
        const bool ts_ready = trial_ready;   // valid only for the call that follows the objective evaluation
        trial_ready = false;
        if (entry == 0) {
            started = true;
            ph_time[0] = ph_time[1] = ph_time[2] = 0;
            int host_err = 0;
            if (factr < (T)0) host_err = TK_ERR_FACTR;
            s_start<T><<<1, 32, 0, stream>>>(w, factr, pgtol, host_err); launches++;
            begin(F_ERRCLB); k_errclb<T><<<LG>>>(w); end(F_ERRCLB);
            if (!site(site_errclb())) return false;
            s_errclb<T><<<LS>>>(w, dist(), offset); launches++;
            begin(F_ACTIVE); k_active<T><<<LG>>>(w); end(F_ACTIVE);
            if (!site(site_active())) return false;
            s_active<T><<<LS>>>(w, dist()); launches++;
            if (!sync_state()) return false;
            x_changed = true;
            return check_launch();
        }
        if (entry == 4) {   // user STOP (:565-572)
            if (aux) {
                CK(cudaMemcpyAsync(x, w.t, sizeof(T) * n, cudaMemcpyDeviceToDevice, stream));
                CK(cudaMemcpyAsync(g, w.gold, sizeof(T) * n, cudaMemcpyDeviceToDevice, stream));
                CK(cudaStreamSynchronize(stream));
                *f = s_host->fold;
                s_host->f = s_host->fold;
                x_changed = true; g_changed = true;
            }
            s_host->task = TK_STOP;
            return true;
        }
        if (entry == 5) {   // any other task: start() (:573-575)
            s_host->task = TK_FG_START;
            return true;
        }
        if (entry == 1) {
            s_call_begin<T><<<1, 32, 0, stream>>>(w, *f, entry); launches++;
            begin(F_PROJGR); k_projgr<T><<<LG>>>(w); end(F_PROJGR);
            if (!site(site_projgr())) return false;
            begin(F_SCALAR); s_fg_start<T><<<LS>>>(w, dist()); end(F_SCALAR);
            if (!enqueue_body()) return false;
        } else if (entry == 2) {
            // the scalar kernel opens the call itself (call_begin = 1); the trial point, or the restored iterate,
            // is written after the state came back, and only when there is something to write
            phase(PH_LNSRCH);
            if (!ts_ready) { begin(F_LS_TRIAL); k_ls_trial<T><<<LG>>>(w); end(F_LS_TRIAL); }
            if (!site(site_lstrial())) return false;
            begin(F_SCALAR); s_ls_trial<T><<<LS>>>(w, dist(), 1, *f); end(F_SCALAR);
            phase(PH_END);
            if (!sync_state() || !finish_call(false)) return false;
        } else if (fast && s_host->cnstnd) {   // NEW_X, fast pipeline
            if (!fast_newx(*f)) return false;
        } else {   // NEW_X
            s_call_begin<T><<<1, 32, 0, stream>>>(w, *f, entry); launches++;
            begin(F_SCALAR); s_newx_tests<T><<<1, 32, 0, stream>>>(w, fused ? 1 : 0); end(F_SCALAR);
            if (fused) { begin(F_UPDATE_CLASSIFY); MTFUSED(launch_update_classify); end(F_UPDATE_CLASSIFY); }
            begin(F_UPDATE); MTCALL(k_update, smem_update, w); end(F_UPDATE);
            if (!site(site_update(mt))) return false;
            begin(F_SCALAR); s_update_dense<T><<<LS>>>(w, dist(), mt); end(F_SCALAR);
            if (!enqueue_body()) return false;
        }
        *f = s_host->f;
        if (body_ran) walked_prev = walked_now;
        resolve_phases();
        return check_launch();
    }

    // ---- checkpoint / resume (include/lbfgsb_b200.h section 4) --------------------------------
    struct CkHeader { char magic[8]; i64 n, ldw, n_global, offset; int m, real_kind, R, rank; i64 state_bytes; };
    bool checkpoint_io(const char* path, bool write) {
        CK(cudaStreamSynchronize(stream));
        // written under a temporary name and renamed on success: a failure never truncates the previous checkpoint
        const std::string tmp = std::string(path) + ".tmp";
        FILE* fp = fopen(write ? tmp.c_str() : path, write ? "wb" : "rb");
        if (!fp) { set_error("cannot open checkpoint file %s", write ? tmp.c_str() : path); return false; }
        CkHeader hd; memset(&hd, 0, sizeof hd);
        memcpy(hd.magic, "LBB2CKP2", 8);
        hd.n = n; hd.ldw = w.ldw; hd.n_global = n_global; hd.offset = offset; hd.m = m; hd.real_kind = (int)sizeof(T); hd.R = R; hd.rank = rank;
        hd.state_bytes = (i64)sizeof(DevState<T>);
        bool ok = true;
        if (write) ok = fwrite(&hd, sizeof hd, 1, fp) == 1;
        else {
            CkHeader in;
            ok = fread(&in, sizeof in, 1, fp) == 1 && memcmp(in.magic, hd.magic, 8) == 0 && in.n == hd.n && in.ldw == hd.ldw &&
                 in.n_global == hd.n_global && in.offset == hd.offset && in.m == hd.m && in.real_kind == hd.real_kind &&
                 in.R == hd.R && in.rank == hd.rank && in.state_bytes == hd.state_bytes;
            if (!ok) set_error("checkpoint %s does not match this workspace (n, m, real kind or shard differ)", path);
        }
        // the heap-replay limit is a property of this workspace (lbfgsb_dev_set_tie_limit / LBFGSB_B200_TIE_LIMIT), not of
        // the run that wrote the checkpoint
        i64 my_tie_limit = 0;
        if (ok && !write) ok = cudaMemcpy(&my_tie_limit, &s_dev->tie_limit, sizeof my_tie_limit, cudaMemcpyDeviceToHost) == cudaSuccess;
        const size_t CH = (size_t)64 << 20;
        void* stage = nullptr;
        if (ok && cudaMallocHost(&stage, CH) != cudaSuccess) { set_error("cudaMallocHost failed"); ok = false; }
        auto xfer = [&](void* dptr, size_t bytes) {
            for (size_t o = 0; ok && o < bytes; o += CH) {
                const size_t c = bytes - o < CH ? bytes - o : CH;
                if (write) {
                    ok = cudaMemcpy(stage, (char*)dptr + o, c, cudaMemcpyDeviceToHost) == cudaSuccess && fwrite(stage, 1, c, fp) == c;
                } else {
                    ok = fread(stage, 1, c, fp) == c && cudaMemcpy((char*)dptr + o, stage, c, cudaMemcpyHostToDevice) == cudaSuccess;
                }
            }
        };
        const size_t vb = (size_t)w.ldw * sizeof(T);
        xfer(s_dev, sizeof(DevState<T>));
        xfer(w.ws, vb * m); xfer(w.wy, vb * m);
        xfer(w.z, vb); xfer(w.r, vb); xfer(w.d, vb); xfer(w.t, vb); xfer(w.xp, vb); xfer(w.gold, vb);
        xfer(w.iwhere, (size_t)w.ldw * 4); xfer(w.state, (size_t)w.ldw);
        if (stage) cudaFreeHost(stage);
        if (ok && !write) ok = cudaMemcpy(&s_dev->tie_limit, &my_tie_limit, sizeof my_tie_limit, cudaMemcpyHostToDevice) == cudaSuccess;
        if (ok && !write) ok = cudaMemcpy(s_host, s_dev, header_bytes, cudaMemcpyDeviceToHost) == cudaSuccess;
        if (ok && !write) started = true;
        if (write && ok) ok = fflush(fp) == 0;
        if (fclose(fp) != 0) ok = false;
        if (write) {
            if (ok) ok = rename(tmp.c_str(), path) == 0;
            else remove(tmp.c_str());
        }
        if (!ok && g_last_error.empty()) set_error("checkpoint %s failed on %s", write ? "write" : "read", path);
        return ok;
    }

    bool active_hash(uint64_t* hash, i64* count) {
        begin(F_HASH); k_active_hash<T><<<LG>>>(w, offset); end(F_HASH);
        // finish on the host: 2 x GRID integers
        std::vector<i64> hp(2 * LBFGSB_GRID);
        CK(cudaMemcpyAsync(hp.data(), w.ipart, sizeof(i64) * 2 * LBFGSB_GRID, cudaMemcpyDeviceToHost, stream));
        CK(cudaStreamSynchronize(stream));
        uint64_t h = 0; i64 c = 0;
        for (int b = 0; b < LBFGSB_GRID; ++b) { h += (uint64_t)hp[b]; c += hp[LBFGSB_GRID + b]; }
        *hash = h; *count = c;
        return true;
    }
};

// ---------------------------------------------------------------------------
// task strings
// ---------------------------------------------------------------------------
static void put60(char* s, const char* lit) {
    size_t k = strlen(lit);
    if (k > 60) k = 60;
    memcpy(s, lit, k);
    for (size_t i = k; i < 60; ++i) s[i] = ' ';
}
static bool pre60(const char* s, const char* lit) { return memcmp(s, lit, strlen(lit)) == 0; }
static bool eq60(const char* s, const char* lit) {
    size_t k = strlen(lit);
    if (memcmp(s, lit, k) != 0) return false;
    for (size_t i = k; i < 60; ++i) if (s[i] != ' ') return false;
    return true;
}
static const char* task_text(int code) {
    switch (code) {
        case TK_FG_START: return "FG_START";
        case TK_FG_LNSRCH: return "FG_LNSRCH";
        case TK_NEW_X: return "NEW_X";
        case TK_CONV_PG: return "CONVERGENCE: NORM_OF_PROJECTED_GRADIENT_<=_PGTOL";
        case TK_CONV_F: return "CONVERGENCE: REL_REDUCTION_OF_F_<=_FACTR*EPSMCH";
        case TK_ABNORMAL: return "ABNORMAL_TERMINATION_IN_LNSRCH";
        case TK_RESTART: return "RESTART_FROM_LNSRCH";
        case TK_ERR_N: return "ERROR: N <= 0";
        case TK_ERR_M: return "ERROR: M <= 0";
        case TK_ERR_FACTR: return "ERROR: FACTR < 0";
        case TK_ERR_NBD: return "ERROR: INVALID NBD";
        case TK_ERR_INFEAS: return "ERROR: NO FEASIBLE SOLUTION";
        default: return "START";
    }
}
static const char* csave_text(int code) {
    switch (code) {
        case CS_START: return "START";
        case CS_FG: return "FG";
        case CS_CONV: return "CONVERGENCE";
        case CS_WARN_ROUND: return "WARNING: ROUNDING ERRORS PREVENT PROGRESS";
        case CS_WARN_XTOL: return "WARNING: XTOL TEST SATISFIED";
        case CS_WARN_STPMAX: return "WARNING: STP = STPMAX";
        case CS_WARN_STPMIN: return "WARNING: STP = STPMIN";
        case CS_ERR_STP_LT_MIN: return "ERROR: STP < STPMIN";
        case CS_ERR_STP_GT_MAX: return "ERROR: STP > STPMAX";
        case CS_ERR_G_GE_0: return "ERROR: INITIAL G >= ZERO";
        case CS_ERR_FTOL: return "ERROR: FTOL < ZERO";
        case CS_ERR_GTOL: return "ERROR: GTOL < ZERO";
        case CS_ERR_XTOL: return "ERROR: XTOL < ZERO";
        case CS_ERR_STPMIN: return "ERROR: STPMIN < ZERO";
        case CS_ERR_STPMAX: return "ERROR: STPMAX < STPMIN";
        default: return "";
    }
}

// save_locals (:904-947): device mirror -> the caller's isave / dsave / lsave
template <typename T>
static void export_state_of(const DevState<T>* s, i64 ng, const double* ph_time, char* task, char* csave, int32_t* lsave, int32_t* isave,
                            T* dsave) {
    auto clamp32 = [](i64 v) { return (int32_t)(v > 2147483647LL ? 2147483647LL : v); };
    lsave[0] = s->prjctd; lsave[1] = s->cnstnd; lsave[2] = s->boxed; lsave[3] = s->updatd;
    isave[21] = clamp32(s->nintol);
    isave[23] = 0;                      // itfile: no Fortran unit on this path
    isave[24] = s->iback; isave[25] = s->nskip; isave[26] = s->head; isave[27] = s->col; isave[28] = s->itail;
    isave[29] = s->iter; isave[30] = s->iupdat;
    isave[32] = clamp32(s->nseg); isave[33] = s->nfgv; isave[34] = s->info; isave[35] = s->ifun; isave[36] = s->iword;
    isave[37] = clamp32(s->nfree); isave[38] = clamp32(s->nact);
    isave[39] = clamp32(ng + 1 - s->nleave);   // ileave
    isave[40] = clamp32(s->nenter);
    isave[42] = s->brackt; isave[43] = s->stage;
    dsave[0] = s->theta; dsave[1] = s->fold; dsave[2] = s->tol; dsave[3] = s->dnorm; dsave[4] = s->epsmch;
    dsave[5] = 0; dsave[9] = 0;   // cpu1, time1: host clock readings of the reference, not kept here
    dsave[6] = (T)ph_time[0]; dsave[7] = (T)ph_time[1]; dsave[8] = (T)ph_time[2];   // cachyt, sbtime, lnscht (seconds)
    dsave[10] = s->gd; dsave[11] = s->stpmx; dsave[12] = s->sbgnrm; dsave[13] = s->stp; dsave[14] = s->gdold; dsave[15] = s->dtd;
    for (int q = 0; q < 13; ++q) dsave[16 + q] = s->ls[q];
    put60(task, task_text(s->task));
    if (s->csave != CS_BLANK) put60(csave, csave_text(s->csave));
}
template <typename T>
static void export_state(const Engine<T>* e, char* task, char* csave, int32_t* lsave, int32_t* isave, T* dsave) {
    export_state_of<T>(e->s_host, e->n_global, e->ph_time, task, csave, lsave, isave, dsave);
}

// Text output of one setulb call (host_print.h), in the reference's order: the iterate-0 lines, the logged
// messages, then prn2lb on NEW_X or prn3lb on termination.
template <typename T>
static void print_after_call(Engine<T>* e, int entry, const T* x, const T* l, const T* u, const T* g, T f, const char* task) {
    lbprint::Ctx& c = e->pr;
    const DevState<T>* s = e->s_host;
    if (c.iprint < 0 && s->ev_n == 0) return;
    const i64 n = e->n;
    std::vector<T> hx, hg, hl, hu;
    auto fetch = [&](const T* dv, std::vector<T>& hv) -> const T* {
        hv.resize((size_t)n);
        if (cudaMemcpy(hv.data(), dv, sizeof(T) * (size_t)n, cudaMemcpyDeviceToHost) != cudaSuccess) return nullptr;
        return hv.data();
    };
    const bool term = pre60(task, "CONV") || pre60(task, "ABNO") || pre60(task, "ERROR") || pre60(task, "STOP");
    if (entry == 0) {
        if (!pre60(task, "ERROR")) {
            const bool vec = c.iprint > 100 && e->R == 1;
            lbprint::prn1lb<T>(c, e->n_global, e->m, (double)s->epsmch, s->prjctd != 0, s->cnstnd != 0, s->nbdd,
                               vec ? fetch(l, hl) : nullptr, vec ? fetch(u, hu) : nullptr, vec ? fetch(x, hx) : nullptr);
        }
    } else if (entry != 4) {
        if (entry == 1) lbprint::iterate0(c, 0, 1, (double)f, (double)s->sbgnrm);
        for (int k = 0; k < s->ev_n && k < LB_EVMAX; ++k) lbprint::event(c, s->ev_code[k], (double)s->ev_a[k], (double)s->ev_b[k]);
        if (s->task == TK_NEW_X) {
            const bool vec = c.iprint > 100 && e->R == 1;
            lbprint::prn2lb<T>(c, n, vec ? fetch(x, hx) : nullptr, vec ? fetch(g, hg) : nullptr, (double)s->f, s->iter, s->nfgv,
                               s->nact, (double)s->sbgnrm, s->nseg, s->iword, s->iback, (double)s->stp, (double)s->xstep);
        }
    }
    if (term && c.iprint >= 0) {
        const bool vec = c.iprint >= 100 && e->R == 1 && !pre60(task, "ERROR");
        lbprint::prn3lb<T>(c, e->n_global, vec ? fetch(x, hx) : nullptr, (double)f, task, s->info, s->iter, s->nfgv, s->nintol,
                           s->nskip, s->nact, (double)s->sbgnrm, c.elapsed(), s->nseg, s->iback, (double)s->stp, (double)s->xstep,
                           s->errk);
    }
    fflush(stdout);
    if (c.itf) fflush(c.itf);
}

template <typename T>
static void setulb_dev_impl(lbfgsb_dev_t* hh, T* x, const T* l, const T* u, const int32_t* nbd, T* f, T* g,
                            const T* factr, const T* pgtol, char* task, const int32_t* iprint, char* csave,
                            int32_t* lsave, int32_t* isave, T* dsave) {
    Engine<T>* e = (Engine<T>*)hh;
    if (!e || e->real_kind != (int)sizeof(T)) { put60(task, "ERROR: INVALID LBFGSB_B200 HANDLE"); set_error("invalid handle"); return; }
    e->pr.iprint = (iprint && e->rank == 0) ? *iprint : -1;   // on a sharded problem rank 0 prints
    int entry, aux = 0;
    if (eq60(task, "START")) entry = 0;
    else if (pre60(task, "FG_LN")) entry = 2;
    else if (pre60(task, "NEW_X")) entry = 3;
    else if (pre60(task, "FG_ST")) entry = 1;
    else if (pre60(task, "STOP")) { entry = 4; aux = (memcmp(task + 6, "CPU", 3) == 0); }
    else entry = 5;
    if (entry == 0) {
        // isave(1:16): sizes/offsets of the reference's wa partition (:250-265), informational here
        const i64 n = e->n_global, m = e->m;
        const i64 mn = m * n, m2 = m * m, m24 = 4 * m2;
        i64 v[16]; v[0] = mn; v[1] = m2; v[2] = m24; v[3] = 1; v[4] = v[3] + mn; v[5] = v[4] + mn; v[6] = v[5] + m2;
        v[7] = v[6] + m2; v[8] = v[7] + m2; v[9] = v[8] + m24; v[10] = v[9] + m24; v[11] = v[10] + n; v[12] = v[11] + n;
        v[13] = v[12] + n; v[14] = v[13] + n; v[15] = v[14] + n;
        for (int q = 0; q < 16; ++q) isave[q] = (v[q] <= 2147483647LL) ? (int32_t)v[q] : -1;
        e->pr.t0 = std::chrono::steady_clock::now();
        e->pr.word[0] = e->pr.word[1] = e->pr.word[2] = '-';
        e->pr.open_file();
    }
    e->x_changed = false; e->g_changed = false;   // (a plain STOP leaves x and g untouched, like the reference's finish())
    if (entry != 0 && !e->started) {
        // the reference would run on whatever the caller's isave/dsave hold; here the state is the workspace's, and a
        // workspace that never saw START has none (same answer as the host twin)
        put60(task, "ERROR: SETULB CALLED WITHOUT A VALID START");
        set_error("setulb_dev called with task other than START on a fresh workspace");
        return;
    }
    if (entry == 4 && !aux) { print_after_call<T>(e, 4, x, l, u, g, *f, task); return; }   // finish(): only prn3lb
    if ((((uintptr_t)x) | ((uintptr_t)l) | ((uintptr_t)u) | ((uintptr_t)nbd) | ((uintptr_t)g)) & 15) {
        set_error("x, l, u, nbd, g must be 16-byte aligned device pointers");
        put60(task, "ERROR: DEVICE POINTERS MUST BE 16-BYTE ALIGNED");
        return;
    }
    bool ok = e->call(entry, aux, x, l, u, nbd, f, g, *factr, *pgtol);
    if (!ok) {
        char buf[61];
        snprintf(buf, sizeof buf, "ERROR: CUDA FAILURE (see lbfgsb_b200_last_error)");
        put60(task, buf);
        return;
    }
    if (entry == 4) { print_after_call<T>(e, 4, x, l, u, g, *f, task); return; }   // the caller's STOP text stays in task
    if (entry == 5) { put60(task, "FG_START"); return; }
    export_state<T>(e, task, csave, lsave, isave, dsave);
    if (entry == 0 && pre60(task, "ERROR")) { isave[34] = e->s_host->info; isave[41] = (int32_t)e->s_host->errk; }
    print_after_call<T>(e, entry, x, l, u, g, *f, task);
}

// ---------------------------------------------------------------------------
// The task loop of the reference's sample programs (test/driver1.f90:263-292, driver2.f90:112-190) as a
// library call (the reference's own @todo, src/lbfgsb.f90:36-37).
// ---------------------------------------------------------------------------
// the caller's limits at NEW_X (driver2.f90:174-181): the STOP text to issue, or nullptr
static const char* limit_stop(const int32_t* isave, int32_t max_iter, int32_t max_fg) {
    const char* stop = nullptr;
    if (max_fg > 0 && isave[33] >= max_fg) stop = "STOP: TOTAL NO. of f AND g EVALUATIONS EXCEEDS LIMIT";   // driver2.f90:176
    if (max_iter > 0 && isave[29] >= max_iter) stop = "STOP: TOTAL NO. of ITERATIONS REACHED LIMIT";
    return stop;
}
// return code of a finished loop: 0 converged, 1 abnormal line search, 2 error or STOP of a failed callback
static int task_return_code(const char* task) {
    if (pre60(task, "CONV")) return 0;
    if (pre60(task, "ABNO")) return 1;
    return 2;
}
template <typename T, typename FG>
static int minimize_impl(lbfgsb_dev_t* h, T* x, const T* l, const T* u, const int32_t* nbd, FG fg, void* user, T factr, T pgtol,
                         int32_t max_iter, int32_t max_fg, int32_t iprint, T* f, T* g, char* task, char* csave, int32_t* lsave,
                         int32_t* isave, T* dsave) {
    Engine<T>* e = (Engine<T>*)h;
    if (!e || e->real_kind != (int)sizeof(T) || !fg) { put60(task, "ERROR: INVALID LBFGSB_B200 HANDLE"); return 2; }
    put60(task, "START");
    for (;;) {
        setulb_dev_impl<T>(h, x, l, u, nbd, f, g, &factr, &pgtol, task, &iprint, csave, lsave, isave, dsave);
        if (pre60(task, "FG")) {
            if (fg(user, e->n, x, g, f, (void*)e->stream) != 0) {
                put60(task, "STOP: THE OBJECTIVE CALLBACK FAILED");
                setulb_dev_impl<T>(h, x, l, u, nbd, f, g, &factr, &pgtol, task, &iprint, csave, lsave, isave, dsave);
                return 2;
            }
        } else if (pre60(task, "NEW_X")) {
            if (const char* stop = limit_stop(isave, max_iter, max_fg)) {
                put60(task, stop);
                setulb_dev_impl<T>(h, x, l, u, nbd, f, g, &factr, &pgtol, task, &iprint, csave, lsave, isave, dsave);
                return 0;
            }
        } else return task_return_code(task);
    }
}

// The same loop kept on the device: the objective callback only ENQUEUES work on the given stream and leaves f in device
// memory, so that one iteration step -- objective, FG_LNSRCH entry, NEW_X entry -- is captured once as a CUDA graph and
// replayed with one launch and one read-back of the state header per step (Engine::build_iter_graph / graph_step).
// START and FG_START, the STOP of a limit, and whatever leaves the fast pipeline's common path go through setulb as usual.
template <typename T, typename FGE>
static int minimize_graph_impl(lbfgsb_dev_t* h, T* x, const T* l, const T* u, const int32_t* nbd, FGE fg, void* user, T factr, T pgtol,
                               int32_t max_iter, int32_t max_fg, T* f, T* g, char* task, char* csave, int32_t* lsave,
                               int32_t* isave, T* dsave) {
    Engine<T>* e = (Engine<T>*)h;
    if (!e || e->real_kind != (int)sizeof(T) || !fg) { put60(task, "ERROR: INVALID LBFGSB_B200 HANDLE"); return 2; }
    const int32_t iprint = -1;
    auto eval_host = [&]() -> bool {   // one evaluation outside the graph: f comes back to the host
        if (fg(user, e->n, x, g, e->f_dev, (void*)e->stream) != 0) return false;
        if (cudaMemcpyAsync(f, e->f_dev, sizeof(T), cudaMemcpyDeviceToHost, e->stream) != cudaSuccess) return false;
        return cudaStreamSynchronize(e->stream) == cudaSuccess;
    };
    put60(task, "START");
    bool graph_ok = false, graph_tried = false;
    for (;;) {
        setulb_dev_impl<T>(h, x, l, u, nbd, f, g, &factr, &pgtol, task, &iprint, csave, lsave, isave, dsave);
        // the device-resident loop takes over whenever the state asks for a line-search evaluation
        if (pre60(task, "FG_LN") && e->fast && e->R == 1 && e->s_host->cnstnd) {
            if (!graph_tried) {
                graph_tried = true;
                e->w.x = x; e->w.l = l; e->w.u = u; e->w.nbd = nbd; e->w.g = g;
                graph_ok = e->build_iter_graph(fg, user, max_iter, max_fg);
            }
            if (graph_ok) {
                e->w.x = x; e->w.l = l; e->w.u = u; e->w.nbd = nbd; e->w.g = g; e->w.bp_hint = 0;
                bool ok = true;
                while (ok && e->s_host->task == TK_FG_LNSRCH) ok = e->graph_step();
                if (!ok) { put60(task, "ERROR: CUDA FAILURE (see lbfgsb_b200_last_error)"); return 2; }
                *f = e->s_host->f;
                export_state<T>(e, task, csave, lsave, isave, dsave);
            }
        }
        if (pre60(task, "FG")) {
            if (!eval_host()) {
                put60(task, "STOP: THE OBJECTIVE CALLBACK FAILED");
                setulb_dev_impl<T>(h, x, l, u, nbd, f, g, &factr, &pgtol, task, &iprint, csave, lsave, isave, dsave);
                return 2;
            }
        } else if (pre60(task, "NEW_X")) {
            if (const char* stop = limit_stop(isave, max_iter, max_fg)) {
                put60(task, stop);
                setulb_dev_impl<T>(h, x, l, u, nbd, f, g, &factr, &pgtol, task, &iprint, csave, lsave, isave, dsave);
                return 0;
            }
        } else return task_return_code(task);
    }
}

// ---------------------------------------------------------------------------
// host twin: device copies of the caller's vectors, handle in isave(17:19)
// ---------------------------------------------------------------------------
struct HostProblem {
    EngineBase* eng;
    void *x, *l, *u, *g; int32_t* nbd;
    i64 n; int kind;
};
static std::mutex g_reg_mu;
static std::unordered_set<HostProblem*> g_registry;
#define LB_MAGIC 0x4C424232   /* 'LBB2' */

static HostProblem* hp_from_isave(const int32_t* isave) {
    if (isave[18] != LB_MAGIC) return nullptr;
    uint64_t v = (uint64_t)(uint32_t)isave[16] | ((uint64_t)(uint32_t)isave[17] << 32);
    HostProblem* p = (HostProblem*)(uintptr_t)v;
    std::lock_guard<std::mutex> lk(g_reg_mu);
    return g_registry.count(p) ? p : nullptr;
}
static void hp_free(HostProblem* p) {
    {
        std::lock_guard<std::mutex> lk(g_reg_mu);
        if (!g_registry.erase(p)) return;
    }
    delete p->eng;
    cudaFree(p->x); cudaFree(p->l); cudaFree(p->u); cudaFree(p->g); cudaFree(p->nbd);
    delete p;
}

template <typename T>
static void setulb_host_impl(const int32_t* n, const int32_t* m, T* x, const T* l, const T* u, const int32_t* nbd, T* f,
                             T* g, const T* factr, const T* pgtol, char* task, const int32_t* iprint, char* csave,
                             int32_t* lsave, int32_t* isave, T* dsave, const char* itfile, int32_t itfile_len) {
    HostProblem* p = nullptr;
    if (eq60(task, "START")) {
        HostProblem* old = hp_from_isave(isave);
        if (old) hp_free(old);
        isave[18] = 0;
        // errclb's scalar checks (:1618-1620) that cannot reach the device
        if (*n <= 0) { put60(task, "ERROR: N <= 0"); if (*m <= 0) put60(task, "ERROR: M <= 0"); if (*factr < (T)0) put60(task, "ERROR: FACTR < 0"); return; }
        if (*m <= 0) { put60(task, "ERROR: M <= 0"); if (*factr < (T)0) put60(task, "ERROR: FACTR < 0"); return; }
        if (*m > LB_MMAX) { put60(task, "ERROR: M > 20 IS NOT SUPPORTED BY LBFGSB_B200"); return; }
        int ndev = 0;
        if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
            put60(task, "ERROR: NO CUDA DEVICE (LBFGSB_B200 HAS NO CPU PATH)");
            set_error("no CUDA device");
            return;
        }
        Engine<T>* e = new Engine<T>();
        if (!e->init(*n, 0, *n, *m, nullptr, nullptr, 0, 1)) { delete e; put60(task, "ERROR: CUDA FAILURE (see lbfgsb_b200_last_error)"); return; }
        if (itfile && itfile_len > 0) e->pr.itname = std::string(itfile, (size_t)itfile_len);   // iteration_file (:243)
        p = new HostProblem();
        p->eng = e; p->n = *n; p->kind = (int)sizeof(T);
        const size_t vb = (size_t)(*n) * sizeof(T);
        if (cudaMalloc(&p->x, vb) || cudaMalloc(&p->l, vb) || cudaMalloc(&p->u, vb) || cudaMalloc(&p->g, vb) ||
            cudaMalloc((void**)&p->nbd, (size_t)(*n) * 4)) {
            set_error("cudaMalloc failed for the host twin's staging vectors");
            put60(task, "ERROR: CUDA FAILURE (see lbfgsb_b200_last_error)");
            delete e; delete p; return;
        }
        cudaMemcpyAsync(p->x, x, vb, cudaMemcpyHostToDevice, e->stream);
        cudaMemcpyAsync(p->l, l, vb, cudaMemcpyHostToDevice, e->stream);
        cudaMemcpyAsync(p->u, u, vb, cudaMemcpyHostToDevice, e->stream);
        cudaMemcpyAsync(p->nbd, nbd, (size_t)(*n) * 4, cudaMemcpyHostToDevice, e->stream);
        {
            std::lock_guard<std::mutex> lk(g_reg_mu);
            g_registry.insert(p);
        }
        uint64_t v = (uint64_t)(uintptr_t)p;
        isave[16] = (int32_t)(uint32_t)(v & 0xffffffffu); isave[17] = (int32_t)(uint32_t)(v >> 32); isave[18] = LB_MAGIC;
    } else {
        p = hp_from_isave(isave);
        if (!p || p->kind != (int)sizeof(T)) { put60(task, "ERROR: SETULB CALLED WITHOUT A VALID START (ISAVE ALTERED?)"); return; }
    }
    Engine<T>* e = (Engine<T>*)p->eng;
    const size_t vb = (size_t)p->n * sizeof(T);
    if (pre60(task, "FG")) cudaMemcpyAsync(p->g, g, vb, cudaMemcpyHostToDevice, e->stream);
    setulb_dev_impl<T>((lbfgsb_dev_t*)e, (T*)p->x, (const T*)p->l, (const T*)p->u, p->nbd, f, (T*)p->g, factr, pgtol,
                       task, iprint, csave, lsave, isave, dsave);
    if (e->x_changed) cudaMemcpyAsync(x, p->x, vb, cudaMemcpyDeviceToHost, e->stream);
    if (e->g_changed) cudaMemcpyAsync(g, p->g, vb, cudaMemcpyDeviceToHost, e->stream);
    if (e->x_changed || e->g_changed) cudaStreamSynchronize(e->stream);
    if (pre60(task, "CONV") || pre60(task, "ABNO") || pre60(task, "ERROR") || pre60(task, "STOP")) {
        hp_free(p);
        isave[18] = 0;
    }
}

// ---------------------------------------------------------------------------
// sample problem (test/driver1.f90:274-289) on the device
// ---------------------------------------------------------------------------
// Line-search epilogue of an objective kernel (SURVEY section 8(f) f4; lnsrlb :2244, projgr :2610-2620): while the
// gradient of a trial point is still in registers the kernel also forms gd = g.d and max |proj g| in the engine's
// fixed reduction shape -- the same products in the same order as k_ls_trial, which the next setulb call then skips.
template <typename T>
struct TrialSums {
    const T* d; const T* l; const T* u; const int* nbd;   // search direction (engine), bounds (caller)
    T* gd_part; T* pg_part;                                // block partials: the engine's slots of k_ls_trial
};
template <typename T>
__device__ __forceinline__ void trial_sums_store(const TrialSums<T>& ts, T agd, T pg, T* sm) {
    T a[1]; a[0] = agd;
    __syncthreads();
    block_sum_store<T, 1>(a, 1, sm, ts.gd_part);
    __syncthreads();
    T r = block_max<T>(pg, sm);
    if (threadIdx.x == 0) ts.pg_part[blockIdx.x] = r;
}

template <typename T>
__global__ void __launch_bounds__(LBFGSB_BLOCK) k_rosenbrock(i64 n, const T* __restrict__ x, T* __restrict__ g,
                                                            T* part, int first, int last, T xl, T xr, const T* halo,
                                                            TrialSums<T> ts) {
    constexpr int VEC = Real<T>::VEC;
    __shared__ T sm[LBFGSB_BLOCK / 32];
    if (halo) { xl = halo[0]; xr = halo[1]; }   // the neighbours' boundary values, still on the device
    T agd = (T)0, pgm = (T)0;
    T acc[1]; acc[0] = (T)0;
    LB_FOR_TILES(T, n, base) {
        T xv[VEC], gv[VEC];
        ldv<T>(x, base, n, xv);
        T xm = (base > 0) ? x[base - 1] : xl;
        T xp = (base + VEC < n) ? x[base + VEC] : xr;
#pragma unroll
        for (int v = 0; v < VEC; ++v) {
            const i64 i = base + v;
            if (i < n) {
                const T xi = xv[v];
                const T xprev = (v == 0) ? xm : xv[v - 1];
                const T xnext = (v == VEC - 1 || i + 1 >= n) ? ((i + 1 < n) ? ((v == VEC - 1) ? xp : xv[v + 1]) : xr) : xv[v + 1];
                const bool is_first = first && i == 0, is_last = last && i == n - 1;
                T t2 = xi - xprev * xprev;       // x(i) - x(i-1)^2
                T t1 = xnext - xi * xi;          // x(i+1) - x(i)^2
                if (is_first) {
                    gv[v] = (T)2 * (xi - (T)1) - (T)16 * xi * t1;
                    acc[0] = acc[0] + (T)0.25 * (xi - (T)1) * (xi - (T)1);
                } else {
                    acc[0] = acc[0] + t2 * t2;
                    gv[v] = is_last ? (T)8 * t2 : ((T)8 * t2 - (T)16 * xi * t1);
                }
            } else gv[v] = (T)0;
        }
        stv<T>(g, base, n, gv);
        if (ts.d) {
            T d[VEC], l[VEC], u[VEC]; int nb[VEC];
            ldv<T>(ts.d, base, n, d); ldv<T>(ts.l, base, n, l); ldv<T>(ts.u, base, n, u); ldvi<T>(ts.nbd, base, n, nb);
#pragma unroll
            for (int v = 0; v < VEC; ++v)
                if (base + v < n) {
                    agd = agd + gv[v] * d[v];
                    pgm = dense::tmax(pgm, projg_one<T>(xv[v], gv[v], l[v], u[v], nb[v]));
                }
        }
    }
    block_sum_store<T, 1>(acc, 1, sm, part);
    if (ts.d) trial_sums_store<T>(ts, agd, pgm, sm);
}
template <typename T>
__global__ void k_rosenbrock_final(const T* part, T* out) {
    T s = final_sum_warp<T>(part);
    if (threadIdx.x == 0) out[0] = (T)4 * s;
}
template <typename T>
static int rosenbrock_impl(i64 n, const T* x, T* g, T* f_out, void* st, int first, int last, T xl, T xr, void* scratch) {
    cudaStream_t s = (cudaStream_t)st;
    T* part = (T*)scratch;
    T* out = part + LBFGSB_GRID;
    k_rosenbrock<T><<<LBFGSB_GRID, LBFGSB_BLOCK, 0, s>>>(n, x, g, part, first, last, xl, xr, nullptr, TrialSums<T>{});
    k_rosenbrock_final<T><<<1, 32, 0, s>>>(part, out);
    if (cudaMemcpyAsync(f_out, out, sizeof(T), cudaMemcpyDeviceToHost, s) != cudaSuccess) return 1;
    if (cudaStreamSynchronize(s) != cudaSuccess) { set_error("rosenbrock kernel failed: %s", cudaGetErrorString(cudaGetLastError())); return 1; }
    return 0;
}

// ---------------------------------------------------------------------------
// bound-constrained convex quadratic (include/lbfgsb_b200.h): f = 1/2 x'Ax - b'x, g = Ax - b,
// A = tridiag(-1, 2 + delta_i, -1); delta, b from a counter-based hash of the global index.
// ---------------------------------------------------------------------------
__host__ __device__ inline unsigned long long lb_mix64(unsigned long long v) {
    v += 0x9E3779B97F4A7C15ULL;
    v = (v ^ (v >> 30)) * 0xBF58476D1CE4E5B9ULL;
    v = (v ^ (v >> 27)) * 0x94D049BB133111EBULL;
    return v ^ (v >> 31);
}
template <typename T>
__device__ __forceinline__ void quad_coeff(unsigned long long gi, unsigned long long seedp, T& diag, T& b) {
    const double u1 = (double)(lb_mix64(2ULL * gi + 2ULL * seedp) >> 32) * (1.0 / 4294967296.0);
    const double u2 = (double)(lb_mix64(2ULL * gi + 1ULL + 2ULL * seedp) >> 32) * (1.0 / 4294967296.0);
    diag = (T)(2.0 + (0.1 + u1));
    b = (T)(2.0 * u2 - 1.0);
}
template <typename T>
__global__ void __launch_bounds__(LBFGSB_BLOCK) k_quadratic(i64 n, const T* __restrict__ x, T* __restrict__ g, T* part,
                                                           i64 off, unsigned long long seedp, T xl, T xr, const T* halo,
                                                           TrialSums<T> ts) {
    constexpr int VEC = Real<T>::VEC;
    __shared__ T sm[LBFGSB_BLOCK / 32];
    if (halo) { xl = halo[0]; xr = halo[1]; }
    T agd = (T)0, pgm = (T)0;
    T acc[1]; acc[0] = (T)0;
    LB_FOR_TILES(T, n, base) {
        T xv[VEC], gv[VEC];
        ldv<T>(x, base, n, xv);
        const T xm = (base > 0) ? x[base - 1] : xl;
        const T xp = (base + VEC < n) ? x[base + VEC] : xr;
#pragma unroll
        for (int v = 0; v < VEC; ++v) {
            const i64 i = base + v;
            gv[v] = (T)0;
            if (i < n) {
                const T xi = xv[v];
                const T xprev = (v == 0) ? xm : xv[v - 1];
                const T xnext = (i + 1 >= n) ? xr : ((v == VEC - 1) ? xp : xv[v + 1]);
                T diag, b;
                quad_coeff<T>((unsigned long long)(i + off), seedp, diag, b);
                const T ax = diag * xi - xprev - xnext;
                gv[v] = ax - b;
                acc[0] = acc[0] + ((T)0.5 * ax - b) * xi;
            }
        }
        stv<T>(g, base, n, gv);
        if (ts.d) {
            T d[VEC], l[VEC], u[VEC]; int nb[VEC];
            ldv<T>(ts.d, base, n, d); ldv<T>(ts.l, base, n, l); ldv<T>(ts.u, base, n, u); ldvi<T>(ts.nbd, base, n, nb);
#pragma unroll
            for (int v = 0; v < VEC; ++v)
                if (base + v < n) {
                    agd = agd + gv[v] * d[v];
                    pgm = dense::tmax(pgm, projg_one<T>(xv[v], gv[v], l[v], u[v], nb[v]));
                }
        }
    }
    block_sum_store<T, 1>(acc, 1, sm, part);
    if (ts.d) trial_sums_store<T>(ts, agd, pgm, sm);
}
template <typename T>
__global__ void k_sum_final(const T* part, T* out) {
    T s = final_sum_warp<T>(part);
    if (threadIdx.x == 0) out[0] = s;
}
template <typename T>
static int quadratic_impl(i64 n, const T* x, T* g, T* f_out, void* st, i64 off, unsigned long long seed, T xl, T xr, void* scratch) {
    cudaStream_t s = (cudaStream_t)st;
    T* part = (T*)scratch;
    T* out = part + LBFGSB_GRID;
    const unsigned long long seedp = seed * 0x9E3779B97F4A7C15ULL;
    k_quadratic<T><<<LBFGSB_GRID, LBFGSB_BLOCK, 0, s>>>(n, x, g, part, off, seedp, xl, xr, nullptr, TrialSums<T>{});
    k_sum_final<T><<<1, 32, 0, s>>>(part, out);
    if (cudaMemcpyAsync(f_out, out, sizeof(T), cudaMemcpyDeviceToHost, s) != cudaSuccess) return 1;
    if (cudaStreamSynchronize(s) != cudaSuccess) { set_error("quadratic kernel failed: %s", cudaGetErrorString(cudaGetLastError())); return 1; }
    return 0;
}

// ---------------------------------------------------------------------------
// The chain-coupled sample objectives on a sharded workspace, exchanged over peer memory: every rank stores its two
// boundary values of x into its neighbours' P2PBuf, the objective kernel's blocks poll the local flags before they
// read the halo, the per-rank parts of f are stored into every peer and summed in rank order.  One host read of f per
// evaluation; no collective launch, no host round trip for the halo.
// ---------------------------------------------------------------------------
template <typename T>
__global__ void k_fg_halo_push(const T* x, i64 n, Peers peers, int R, int rank, int slot, unsigned long long seq) {
    if (threadIdx.x != 0) return;
    P2PBuf<T>* left = rank > 0 ? (P2PBuf<T>*)peers.p[rank - 1] : nullptr;
    P2PBuf<T>* right = rank < R - 1 ? (P2PBuf<T>*)peers.p[rank + 1] : nullptr;
    if (left) left->halo[slot][1] = x[0];
    if (right) right->halo[slot][0] = x[n - 1];
    __threadfence_system();
    if (left) *(volatile unsigned long long*)&left->hflag[slot][1] = seq;
    if (right) *(volatile unsigned long long*)&right->hflag[slot][0] = seq;
}
// blocks of the objective kernel: wait for the neighbours' values of this evaluation, leave them in halo_out[0..1]
template <typename T>
__global__ void k_fg_halo_wait(Wk<T> w, P2PBuf<T>* mine, int R, int rank, int slot, unsigned long long seq, T* halo_out) {
    if (threadIdx.x != 0) return;
    const long long t0 = clock64();
    for (int side = 0; side < 2; ++side) {
        const bool need = side == 0 ? rank > 0 : rank < R - 1;
        T v = (T)0;
        if (need) {
            volatile unsigned long long* f = &mine->hflag[slot][side];
            while (*f != seq) { if (clock64() - t0 > LB_P2P_SPIN_LIMIT) { w.s->p2p_timeout = 1; break; } }
            __threadfence_system();
            v = *(volatile T*)&mine->halo[slot][side];
        }
        halo_out[side] = v;
    }
}
template <typename T>
__global__ void k_fg_fsum_push(const T* fpart_local, Peers peers, int R, int rank, int slot, unsigned long long seq) {
    if ((int)threadIdx.x >= R) return;
    P2PBuf<T>* dst = (P2PBuf<T>*)peers.p[threadIdx.x];
    dst->fpart[slot][rank] = fpart_local[0];
    __threadfence_system();
    *(volatile unsigned long long*)&dst->fflag[slot][rank] = seq;
}
template <typename T>
__global__ void k_fg_fsum_wait(Wk<T> w, P2PBuf<T>* mine, int R, int slot, unsigned long long seq, T* f_out) {
    p2p_wait<T>(w, mine->fflag[slot], R, seq);
    if (threadIdx.x != 0) return;
    T acc = *(volatile T*)&mine->fpart[slot][0];
    for (int q = 1; q < R; ++q) acc = acc + *(volatile T*)&mine->fpart[slot][q];
    f_out[0] = acc;
}

// Shard variants without a host round trip: the neighbours' boundary values are read from halo_dev[0..1] and the
// shard's part of f is left in f_part_dev[0]; nothing is synchronised (the caller all-reduces f_part_dev on the
// same stream and reads it once).
template <typename T>
static int rosenbrock_halo_impl(i64 n, const T* x, T* g, T* f_part_dev, void* st, int first, int last, const T* halo_dev, void* scratch) {
    cudaStream_t s = (cudaStream_t)st;
    T* part = (T*)scratch;
    k_rosenbrock<T><<<LBFGSB_GRID, LBFGSB_BLOCK, 0, s>>>(n, x, g, part, first, last, (T)0, (T)0, halo_dev, TrialSums<T>{});
    k_rosenbrock_final<T><<<1, 32, 0, s>>>(part, f_part_dev);
    return cudaGetLastError() != cudaSuccess;
}
template <typename T>
static int quadratic_halo_impl(i64 n, const T* x, T* g, T* f_part_dev, void* st, i64 off, unsigned long long seed, const T* halo_dev, void* scratch) {
    cudaStream_t s = (cudaStream_t)st;
    T* part = (T*)scratch;
    const unsigned long long seedp = seed * 0x9E3779B97F4A7C15ULL;
    k_quadratic<T><<<LBFGSB_GRID, LBFGSB_BLOCK, 0, s>>>(n, x, g, part, off, seedp, (T)0, (T)0, halo_dev, TrialSums<T>{});
    k_sum_final<T><<<1, 32, 0, s>>>(part, f_part_dev);
    return cudaGetLastError() != cudaSuccess;
}

// ---------------------------------------------------------------------------
// test-only single kernels
// ---------------------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(LBFGSB_BLOCK) k_test_sum(i64 n, const T* a, const T* b, T* part) {
    constexpr int VEC = Real<T>::VEC;
    __shared__ T sm[LBFGSB_BLOCK / 32];
    T acc[1]; acc[0] = (T)0;
    LB_FOR_TILES(T, n, base) {
        T av[VEC], bv[VEC];
        ldv<T>(a, base, n, av); ldv<T>(b, base, n, bv);
#pragma unroll
        for (int v = 0; v < VEC; ++v) if (base + v < n) acc[0] = acc[0] + av[v] * bv[v];
    }
    block_sum_store<T, 1>(acc, 1, sm, part);
}
template <typename T>
__global__ void k_test_sum_final(const T* part, T* out) {
    T s = final_sum_warp<T>(part);
    if (threadIdx.x == 0) out[0] = s;
}
template <typename T>
static int test_sum_impl(i64 n, const T* a, const T* b, T* out) {
    T* part = nullptr;
    if (cudaMalloc(&part, sizeof(T) * (LBFGSB_GRID + 1)) != cudaSuccess) return 1;
    k_test_sum<T><<<LBFGSB_GRID, LBFGSB_BLOCK>>>(n, a, b, part);
    k_test_sum_final<T><<<1, 32>>>(part, part + LBFGSB_GRID);
    cudaError_t e = cudaMemcpy(out, part + LBFGSB_GRID, sizeof(T), cudaMemcpyDeviceToHost);
    cudaFree(part);
    return e != cudaSuccess;
}

// ops 0-4: the single-thread routines (dense::); 10-14: the same by one warp (wdense::), as the scalar kernels run
// them; 15: the dense tail of formk (w_formk_dense with no new pair and no entering/leaving variable)
__global__ void k_test_dense(int op, int m, int col, double theta, double* a, double* b, double* c, int* info, DevState<double>* st) {
    if (blockIdx.x != 0 || threadIdx.x >= 32) return;
    int r = 0;
    if (op >= 10 && op <= 14) {
        if (op == 10) r = wdense::dpofa<double>(a, m, col);
        else if (op == 11) r = wdense::dtrsl<double>(a, m, col, b, 1);
        else if (op == 12) r = wdense::dtrsl<double>(a, m, col, b, 11);
        else if (op == 13) r = wdense::bmv<double>(m, a, b, col, c, c + 2 * m);
        else r = wdense::formt<double>(m, c, a, b, col, theta);
        if (threadIdx.x == 0) *info = r;
        return;
    }
    if (op == 15) {   // a = wn1 (2m x 2m, in), b = sy (m x m), c = wn (2m x 2m, out)
        if (threadIdx.x == 0) {
            st->m = m; st->col = col; st->theta = theta; st->do_formk = 1; st->updatd = 0; st->do_delta = 0; st->iupdat = m + 1;
            st->restart = 0; st->in_body = 1; st->ev_n = 0;
            for (int q = 0; q < m * m; ++q) st->sy[q] = b[q];
        }
        __syncwarp();
        Red<double>* red = nullptr;
        w_formk_dense<double>(st, *red, m <= 5 ? 5 : (m <= 10 ? 10 : 20), (const double*)nullptr, c, a);
        if (threadIdx.x == 0) *info = st->restart ? 1 : 0;
        return;
    }
    if (threadIdx.x != 0) return;
    if (op == 0) *info = dense::dpofa<double>(a, m, col);
    else if (op == 1) *info = dense::dtrsl<double>(a, m, col, b, 1);
    else if (op == 2) *info = dense::dtrsl<double>(a, m, col, b, 11);
    else if (op == 3) *info = dense::bmv<double>(m, a, b, col, c, c + 2 * m);      // a=sy, b=wt, c=[v | p]
    else if (op == 4) *info = dense::formt<double>(m, c, a, b, col, theta);         // a=sy, b=ss, c=wt
}
__global__ void k_test_dcsrch(double f, double g, double* stp, double stpmax, int* task, int* isave2, double* dsave13) {
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    dense::dcsrch<double>(f, g, *stp, 1.0e-3, 0.9, 0.1, 0.0, stpmax, *task, isave2[0], isave2[1], dsave13);
}
template <typename K>
__global__ void k_test_iota(int* v, i64 n) {
    for (i64 i = (i64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (i64)gridDim.x * blockDim.x) v[i] = (int)i;
}
__global__ void k_test_heap_order(unsigned long long* k, int* v, i64 n, int* order_out) {
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    heap_build<unsigned long long>(k - 1, v - 1, n);
    for (i64 nleft = n; nleft > 0; --nleft) {
        unsigned long long out; int var;
        heap_pop<unsigned long long>(k - 1, v - 1, nleft, out, var);
        order_out[n - nleft] = var;
    }
}
__global__ void k_test_setctl(SortCtl* c, i64 n) { if (threadIdx.x == 0) { c->count = n; c->cur = 0; c->skip = 0; } }

// Single-GPU objective with the line-search epilogue (and the shared implementation of the epilogue's bookkeeping).
// (the built-in objectives go through the same two public calls a caller's own kernel would use)
extern "C" int lbfgsb_dev_trial_sums(lbfgsb_dev_t* h, lbfgsb_trial_sums_t* out);
extern "C" void lbfgsb_dev_trial_sums_commit(lbfgsb_dev_t* h);
template <typename T>
static TrialSums<T> trial_sums_of(Engine<T>* e, const T* l, const T* u, const int32_t* nbd) {
    TrialSums<T> ts; memset(&ts, 0, sizeof ts);
    lbfgsb_trial_sums_t pub;
    if (l && u && nbd && lbfgsb_dev_trial_sums((lbfgsb_dev_t*)e, &pub) == 0) {
        ts.d = (const T*)pub.d_dev; ts.l = l; ts.u = u; ts.nbd = nbd;
        ts.gd_part = (T*)pub.gd_part_dev; ts.pg_part = (T*)pub.pg_part_dev;
        lbfgsb_dev_trial_sums_commit((lbfgsb_dev_t*)e);
    }
    return ts;
}

// ---------------------------------------------------------------------------
// Batched small problems (batch.cuh; include/lbfgsb_b200.h section 6)
// ---------------------------------------------------------------------------
struct BatchBase {
    virtual ~BatchBase() {}
    int real_kind;
};
template <typename T>
struct BatchEngine : BatchBase {
    BatchWk<T> bw;
    cudaStream_t stream = 0;
    bool own_stream = false;
    std::vector<void*> allocs;
    int* entry_dev = nullptr; int* entry_host = nullptr;
    char* hdr_host = nullptr;          // [nprob][header_bytes], pinned
    size_t header_bytes = 0;
    std::vector<char> started;
    int n_fg = 0, n_newx = 0, n_done = 0;
    i64 launches = 0;
    template <typename P> bool dalloc(P** p, size_t bytes) {
        void* q = nullptr;
        if (bytes == 0) bytes = 16;
        cudaError_t e = cudaMalloc(&q, bytes);
        if (e != cudaSuccess) { set_error("cudaMalloc(%zu) failed: %s", bytes, cudaGetErrorString(e)); return false; }
        allocs.push_back(q);
        *p = (P*)q;
        return true;
    }
    template <int MT> bool set_attr() {
        CK(cudaFuncSetAttribute(k_batch_setulb<T, MT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(BatchSm<T>)));
        return true;
    }
    bool init(int nprob, i64 n, int m, cudaStream_t st) {
        real_kind = (int)sizeof(T);
        memset(&bw, 0, sizeof bw);
        bw.nprob = nprob; bw.n = n; bw.m = m; bw.mt = (m <= 5) ? 5 : (m <= 10 ? 10 : 20);
        bw.ldw = (n + 31) / 32 * 32;
        if (st) stream = st;
        else { CK(cudaStreamCreateWithFlags(&stream, cudaStreamNonBlocking)); own_stream = true; }
        const size_t P = (size_t)nprob, vb = (size_t)bw.ldw * sizeof(T);
        if (!dalloc(&bw.ws, P * vb * m) || !dalloc(&bw.wy, P * vb * m)) return false;
        if (!dalloc(&bw.z, P * vb) || !dalloc(&bw.r, P * vb) || !dalloc(&bw.d, P * vb) || !dalloc(&bw.t, P * vb) || !dalloc(&bw.xp, P * vb) ||
            !dalloc(&bw.gold, P * vb) || !dalloc(&bw.bpt, P * vb)) return false;
        if (!dalloc(&bw.iwhere, P * bw.ldw * 4) || !dalloc(&bw.bpo, P * bw.ldw * 4) || !dalloc(&bw.state, P * bw.ldw)) return false;
        if (!dalloc(&bw.delta, P * sizeof(T) * 6 * LB_MMAX * LB_MMAX) || !dalloc(&bw.s, P * sizeof(DevState<T>))) return false;
        if (!dalloc(&entry_dev, P * sizeof(int)) || !dalloc(&bw.fgmask, P * sizeof(int))) return false;
        CK(cudaMemsetAsync(bw.fgmask, 0, P * sizeof(int), stream));
        CK(cudaMemsetAsync(bw.s, 0, P * sizeof(DevState<T>), stream));
        CK(cudaMemsetAsync(bw.ws, 0, P * vb * m, stream));
        CK(cudaMemsetAsync(bw.wy, 0, P * vb * m, stream));
        CK(cudaMemsetAsync(bw.delta, 0, P * sizeof(T) * 6 * LB_MMAX * LB_MMAX, stream));
        header_bytes = offsetof(DevState<T>, sy);
        CK(cudaMallocHost((void**)&hdr_host, P * header_bytes));
        CK(cudaMallocHost((void**)&entry_host, P * sizeof(int)));
        started.assign(P, 0);
        if (!(bw.mt == 5 ? set_attr<5>() : (bw.mt == 10 ? set_attr<10>() : set_attr<20>()))) return false;
        CK(cudaStreamSynchronize(stream));
        return true;
    }
    ~BatchEngine() {
        for (void* p : allocs) cudaFree(p);
        if (hdr_host) cudaFreeHost(hdr_host);
        if (entry_host) cudaFreeHost(entry_host);
        if (own_stream && stream) cudaStreamDestroy(stream);
    }
    bool call(T* x, const T* l, const T* u, const int32_t* nbd, T* f, T* g, T factr, T pgtol, char* task, char* csave, int32_t* lsave,
              int32_t* isave, T* dsave) {
        const int P = bw.nprob;
        bool any = false;
        for (int p = 0; p < P; ++p) {
            const char* t = task + 60 * (size_t)p;
            int e;
            if (eq60(t, "START")) { e = BE_START; started[p] = 1; }
            else if (started[p] == 2) e = BE_IDLE;   // ended by a STOP of its caller
            else if (!started[p]) { put60(task + 60 * (size_t)p, "ERROR: SETULB CALLED WITHOUT A VALID START"); e = BE_IDLE; }
            else if (pre60(t, "FG_LN")) e = BE_FG_LNSRCH;
            else if (pre60(t, "NEW_X")) e = BE_NEW_X;
            else if (pre60(t, "FG_ST")) e = BE_FG_START;
            else if (pre60(t, "STOP")) { e = (memcmp(t + 6, "CPU", 3) == 0) ? BE_STOP_CPU : BE_IDLE; started[p] = 2; }   // a plain STOP only ends the problem
            else if (pre60(t, "CONV") || pre60(t, "ABNO") || pre60(t, "ERROR")) e = BE_IDLE;
            else e = BE_OTHER;
            entry_host[p] = e;
            any = any || e != BE_IDLE;
        }
        n_fg = n_newx = n_done = 0;
        if (any) {
            bw.x = x; bw.l = l; bw.u = u; bw.nbd = nbd; bw.g = g; bw.f = f; bw.factr = factr; bw.pgtol = pgtol;
            bw.entry = entry_dev;
            CK(cudaMemcpyAsync(entry_dev, entry_host, sizeof(int) * P, cudaMemcpyHostToDevice, stream));
            const size_t smem = sizeof(BatchSm<T>);
            if (bw.mt == 5) k_batch_setulb<T, 5><<<P, LBFGSB_BLOCK, smem, stream>>>(bw);
            else if (bw.mt == 10) k_batch_setulb<T, 10><<<P, LBFGSB_BLOCK, smem, stream>>>(bw);
            else k_batch_setulb<T, 20><<<P, LBFGSB_BLOCK, smem, stream>>>(bw);
            launches++;
            CK(cudaMemcpy2DAsync(hdr_host, header_bytes, bw.s, sizeof(DevState<T>), header_bytes, P, cudaMemcpyDeviceToHost, stream));
            CK(cudaStreamSynchronize(stream));
            cudaError_t le = cudaGetLastError();
            if (le != cudaSuccess) { set_error("batch kernel failed: %s", cudaGetErrorString(le)); return false; }
        }
        const double ph[3] = {0, 0, 0};
        for (int p = 0; p < P; ++p) {
            char* t = task + 60 * (size_t)p;
            const int e = entry_host[p];
            if (e != BE_IDLE) {
                const DevState<T>* s = (const DevState<T>*)(hdr_host + (size_t)p * header_bytes);
                if (e == BE_STOP_CPU) { /* the caller's STOP text stays in task; x, g, f were restored */ }
                else {
                    export_state_of<T>(s, bw.n, ph, t, csave + 60 * (size_t)p, lsave + 4 * (size_t)p, isave + 44 * (size_t)p, dsave + 29 * (size_t)p);
                    if (e == BE_START && pre60(t, "ERROR")) { isave[44 * (size_t)p + 34] = s->info; isave[44 * (size_t)p + 41] = (int32_t)s->errk; }
                }
            }
            if (pre60(t, "FG")) n_fg++;
            else if (pre60(t, "NEW_X")) n_newx++;
            else n_done++;
        }
        return true;
    }
    // one problem's slice of a work vector (lbfgsb_batch_vector_copy), copied on the batch's stream
    int vector_copy(int p, int which, void* dst, i64 bytes) {
        if (p < 0 || p >= bw.nprob) { set_error("lbfgsb_batch_vector_copy: problem %d out of range [0, %d)", p, bw.nprob); return 1; }
        const i64 o = (i64)p * bw.ldw, vb = bw.ldw * (i64)sizeof(T);
        const void* src = nullptr;
        i64 cap = vb;
        switch (which) {
            case 0: src = bw.z + o; break;
            case 1: src = bw.r + o; break;
            case 2: src = bw.d + o; break;
            case 3: src = bw.t + o; break;
            case 4: src = bw.xp + o; break;
            case 5: src = bw.ws + o * bw.m; cap = bw.m * vb; break;
            case 6: src = bw.wy + o * bw.m; cap = bw.m * vb; break;
            case 7: src = bw.iwhere + o; cap = bw.ldw * 4; break;
            case 8: src = bw.gold + o; break;
            default: set_error("lbfgsb_batch_vector_copy: no vector %d", which); return 1;
        }
        if (bytes > cap) { set_error("lbfgsb_batch_vector_copy: %lld bytes requested, vector %d of a problem holds %lld", (long long)bytes, which, (long long)cap); return 1; }
        if (cudaMemcpyAsync(dst, src, (size_t)bytes, cudaMemcpyDeviceToDevice, stream) != cudaSuccess) return 1;
        return cudaStreamSynchronize(stream) != cudaSuccess;
    }
};

// sample objective for a batch (test/driver1.f90:274-289, one CTA per problem): the arithmetic and the summation shape
// of k_rosenbrock, f_dev[p] = 4 * sum
template <typename T>
__global__ void __launch_bounds__(LBFGSB_BLOCK) k_rosenbrock_batch(int nprob, i64 n, const T* __restrict__ xall, T* __restrict__ gall,
                                                                  T* __restrict__ f, const int* __restrict__ entry) {
    extern __shared__ __align__(16) unsigned char bsm_raw[];
    BatchSm<T>& sm = *reinterpret_cast<BatchSm<T>*>(bsm_raw);
    const int p = blockIdx.x;
    if (p >= nprob) return;
    if (entry && entry[p] == 0) return;   // this problem did not ask for f and g
    const T* x = xall + (i64)p * n;
    T* g = gall + (i64)p * n;
    B_TILES(T, n, tl) {
        T acc[1]; acc[0] = (T)0;
        B_ELEMS(T, n, tl, i) {
            const T xi = x[i];
            const T xprev = (i > 0) ? x[i - 1] : (T)0;
            const T xnext = (i + 1 < n) ? x[i + 1] : (T)0;
            const T t2 = xi - xprev * xprev;
            const T t1 = xnext - xi * xi;
            if (i == 0) {
                g[i] = (T)2 * (xi - (T)1) - (T)16 * xi * t1;
                acc[0] = acc[0] + (T)0.25 * (xi - (T)1) * (xi - (T)1);
            } else {
                acc[0] = acc[0] + t2 * t2;
                g[i] = (i == n - 1) ? (T)8 * t2 : ((T)8 * t2 - (T)16 * xi * t1);
            }
        }
        batch::tile_sum<T, 1>(acc, 1, tl, sm);
    }
    batch::final_sums<T>(1, n, sm, sm.red.rv);
    if (threadIdx.x == 0) f[p] = (T)4 * sm.red.rv[0];
}

// ---------------------------------------------------------------------------
// C ABI
// ---------------------------------------------------------------------------
// formk's entering/leaving corrections (:1801-1851) on their own: the compaction of the listed rows and k_formk_delta.
// ws_dev, wy_dev: m columns of ldw reals; state_dev: one byte per variable (bit 0 free now, bit 1 free before);
// out_host: six [LB_MMAX x LB_MMAX] column-major sums -- entering Wy'Wy, Ws'Ws, Ws'Wy, then the same for leaving rows.
template <typename T>
static int test_formk_delta_impl(int64_t n, int32_t m, int32_t col, int32_t head, int64_t ldw, const T* ws, const T* wy,
                                 const unsigned char* state, T* out_host) {
    if (n <= 0 || m <= 0 || m > LB_MMAX || col <= 0 || col > m || head < 1 || head > m || ldw < n) return 1;
    std::vector<char> hs(sizeof(DevState<T>), 0);
    DevState<T>* h = (DevState<T>*)hs.data();
    h->go = 1; h->in_body = 1; h->do_delta = 1; h->col = col; h->m = m; h->head = head;
    DevState<T>* st = nullptr; int* counts = nullptr; i64* offs = nullptr; int* list = nullptr; SortCtl* ctl = nullptr;
    typename Real<T>::key_t* keys = nullptr; T* parts = nullptr; T* delta = nullptr;
    const i64 tile = (i64)LBFGSB_BLOCK * Real<T>::VEC * Real<T>::UNROLL, ntiles = (n + tile - 1) / tile;
    const size_t ne = (size_t)6 * LB_MMAX * LB_MMAX;
    if (cudaMalloc(&st, sizeof(DevState<T>)) || cudaMalloc(&counts, 4 * (ntiles + 1)) || cudaMalloc(&offs, 8 * (ntiles + 1)) ||
        cudaMalloc(&list, 4 * (size_t)n) || cudaMalloc(&keys, sizeof(typename Real<T>::key_t) * (size_t)n) || cudaMalloc(&ctl, sizeof(SortCtl)) ||
        cudaMalloc(&parts, sizeof(T) * ne * LB_FD_GRID) || cudaMalloc(&delta, sizeof(T) * ne)) return 1;
    cudaMemcpy(st, h, sizeof(DevState<T>), cudaMemcpyHostToDevice);
    cudaMemset(delta, 0, sizeof(T) * ne);
    Wk<T> w; memset(&w, 0, sizeof w);
    w.n = n; w.m = m; w.ldw = ldw; w.ws = (T*)ws; w.wy = (T*)wy; w.state = (unsigned char*)state; w.s = st;
    k_el_count<T><<<LBFGSB_GRID, LBFGSB_BLOCK>>>(w, counts);
    k_tile_scan<T><<<1, 1024>>>(w, 1, counts, offs, ntiles, ctl);
    k_flag_write<T, 1><<<LBFGSB_GRID, LBFGSB_BLOCK>>>(w, counts, offs, keys, list);
    k_formk_delta<T><<<fd_grid<T>(), 256>>>(w, list, ctl, parts);
    k_formk_delta_final<T><<<(6 * LB_MMAX * LB_MMAX + 255) / 256, 256>>>(w, parts, fd_grid<T>(), delta);
    cudaError_t e = cudaMemcpy(out_host, delta, sizeof(T) * ne, cudaMemcpyDeviceToHost);
    cudaFree(st); cudaFree(counts); cudaFree(offs); cudaFree(list); cudaFree(keys); cudaFree(ctl); cudaFree(parts); cudaFree(delta);
    return e != cudaSuccess || cudaGetLastError() != cudaSuccess;
}
extern "C" {

int lbfgsb_b200_version(void) { return 100; }
const char* lbfgsb_b200_last_error(void) { return g_last_error.c_str(); }

lbfgsb_dev_t* lbfgsb_dev_create_sharded(int64_t n_local, int64_t offset, int64_t n_global, int32_t m, int32_t real_kind,
                                        void* cuda_stream, void* nccl_comm, int32_t rank, int32_t world) {
    if (n_local <= 0 || m <= 0 || m > LB_MMAX) { set_error("lbfgsb_dev_create: need n > 0 and 0 < m <= %d", LB_MMAX); return nullptr; }
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) { set_error("no CUDA device (lbfgsb_b200 has no CPU path)"); return nullptr; }
    if (world > 1 && (!nccl_comm || !nccl_api()->ok)) { set_error("sharded engine needs an NCCL communicator"); return nullptr; }
    if (real_kind == 8) {
        Engine<double>* e = new Engine<double>();
        if (!e->init(n_local, offset, n_global, m, (cudaStream_t)cuda_stream, (ncclComm_t)nccl_comm, rank, world)) { delete e; return nullptr; }
        return (lbfgsb_dev_t*)e;
    } else if (real_kind == 4) {
        Engine<float>* e = new Engine<float>();
        if (!e->init(n_local, offset, n_global, m, (cudaStream_t)cuda_stream, (ncclComm_t)nccl_comm, rank, world)) { delete e; return nullptr; }
        return (lbfgsb_dev_t*)e;
    }
    set_error("real_kind must be 8 or 4");
    return nullptr;
}
lbfgsb_dev_t* lbfgsb_dev_create(int64_t n, int32_t m, int32_t real_kind, void* cuda_stream) {
    return lbfgsb_dev_create_sharded(n, 0, n, m, real_kind, cuda_stream, nullptr, 0, 1);
}
void lbfgsb_dev_destroy(lbfgsb_dev_t* h) { delete (EngineBase*)h; }
void lbfgsb_dev_set_iteration_file(lbfgsb_dev_t* h, const char* name) {
    EngineBase* b = (EngineBase*)h;
    if (b && name && name[0]) b->pr.itname = name;
}

void lbfgsb_setulb_dev_f64(lbfgsb_dev_t* h, double* x, const double* l, const double* u, const int32_t* nbd, double* f,
                           double* g, const double* factr, const double* pgtol, char* task, const int32_t* iprint,
                           char* csave, int32_t* lsave, int32_t* isave, double* dsave) {
    setulb_dev_impl<double>(h, x, l, u, nbd, f, g, factr, pgtol, task, iprint, csave, lsave, isave, dsave);
}
void lbfgsb_setulb_dev_f32(lbfgsb_dev_t* h, float* x, const float* l, const float* u, const int32_t* nbd, float* f,
                           float* g, const float* factr, const float* pgtol, char* task, const int32_t* iprint,
                           char* csave, int32_t* lsave, int32_t* isave, float* dsave) {
    setulb_dev_impl<float>(h, x, l, u, nbd, f, g, factr, pgtol, task, iprint, csave, lsave, isave, dsave);
}

void lbfgsb_setulb_f64(const int32_t* n, const int32_t* m, double* x, const double* l, const double* u, const int32_t* nbd,
                       double* f, double* g, const double* factr, const double* pgtol, double* wa, int32_t* iwa, char* task,
                       const int32_t* iprint, char* csave, int32_t* lsave, int32_t* isave, double* dsave,
                       const char* itfile, int32_t itfile_len) {
    (void)wa; (void)iwa;
    setulb_host_impl<double>(n, m, x, l, u, nbd, f, g, factr, pgtol, task, iprint, csave, lsave, isave, dsave, itfile, itfile_len);
}
void lbfgsb_setulb_f32(const int32_t* n, const int32_t* m, float* x, const float* l, const float* u, const int32_t* nbd,
                       float* f, float* g, const float* factr, const float* pgtol, float* wa, int32_t* iwa, char* task,
                       const int32_t* iprint, char* csave, int32_t* lsave, int32_t* isave, float* dsave,
                       const char* itfile, int32_t itfile_len) {
    (void)wa; (void)iwa;
    setulb_host_impl<float>(n, m, x, l, u, nbd, f, g, factr, pgtol, task, iprint, csave, lsave, isave, dsave, itfile, itfile_len);
}
void lbfgsb_host_release(int32_t* isave) {
    HostProblem* p = hp_from_isave(isave);
    if (p) { hp_free(p); isave[18] = 0; }
}
int lbfgsb_host_previous_x_f64(const int32_t* isave, double* t_out) {
    HostProblem* p = hp_from_isave(isave);
    if (!p || p->kind != 8) return 1;
    Engine<double>* e = (Engine<double>*)p->eng;
    return cudaMemcpy(t_out, e->w.t, sizeof(double) * p->n, cudaMemcpyDeviceToHost) != cudaSuccess;
}
int lbfgsb_host_previous_x_f32(const int32_t* isave, float* t_out) {
    HostProblem* p = hp_from_isave(isave);
    if (!p || p->kind != 4) return 1;
    Engine<float>* e = (Engine<float>*)p->eng;
    return cudaMemcpy(t_out, e->w.t, sizeof(float) * p->n, cudaMemcpyDeviceToHost) != cudaSuccess;
}
// the host twin's engine, for diagnostics (active-set hash) in tests
lbfgsb_dev_t* lbfgsb_host_engine(const int32_t* isave) {
    HostProblem* p = hp_from_isave(isave);
    return p ? (lbfgsb_dev_t*)p->eng : nullptr;
}

int lbfgsb_dev_checkpoint_write(lbfgsb_dev_t* h, const char* path) {
    EngineBase* b = (EngineBase*)h;
    if (!b || !path) return 1;
    g_last_error.clear();
    return ((b->real_kind == 8) ? ((Engine<double>*)b)->checkpoint_io(path, true) : ((Engine<float>*)b)->checkpoint_io(path, true)) ? 0 : 1;
}
int lbfgsb_dev_checkpoint_read(lbfgsb_dev_t* h, const char* path) {
    EngineBase* b = (EngineBase*)h;
    if (!b || !path) return 1;
    g_last_error.clear();
    return ((b->real_kind == 8) ? ((Engine<double>*)b)->checkpoint_io(path, false) : ((Engine<float>*)b)->checkpoint_io(path, false)) ? 0 : 1;
}

int lbfgsb_minimize_dev_f64(lbfgsb_dev_t* h, double* x, const double* l, const double* u, const int32_t* nbd, lbfgsb_fg_dev_f64 fg,
                            void* user, double factr, double pgtol, int32_t max_iter, int32_t max_fg, int32_t iprint, double* f,
                            double* g, char* task, char* csave, int32_t* lsave, int32_t* isave, double* dsave) {
    return minimize_impl<double>(h, x, l, u, nbd, fg, user, factr, pgtol, max_iter, max_fg, iprint, f, g, task, csave, lsave, isave, dsave);
}
int lbfgsb_minimize_dev_f32(lbfgsb_dev_t* h, float* x, const float* l, const float* u, const int32_t* nbd, lbfgsb_fg_dev_f32 fg,
                            void* user, float factr, float pgtol, int32_t max_iter, int32_t max_fg, int32_t iprint, float* f,
                            float* g, char* task, char* csave, int32_t* lsave, int32_t* isave, float* dsave) {
    return minimize_impl<float>(h, x, l, u, nbd, fg, user, factr, pgtol, max_iter, max_fg, iprint, f, g, task, csave, lsave, isave, dsave);
}

int lbfgsb_minimize_graph_dev_f64(lbfgsb_dev_t* h, double* x, const double* l, const double* u, const int32_t* nbd, lbfgsb_fg_enqueue_f64 fg,
                                  void* user, double factr, double pgtol, int32_t max_iter, int32_t max_fg, double* f, double* g,
                                  char* task, char* csave, int32_t* lsave, int32_t* isave, double* dsave) {
    return minimize_graph_impl<double>(h, x, l, u, nbd, fg, user, factr, pgtol, max_iter, max_fg, f, g, task, csave, lsave, isave, dsave);
}
int lbfgsb_minimize_graph_dev_f32(lbfgsb_dev_t* h, float* x, const float* l, const float* u, const int32_t* nbd, lbfgsb_fg_enqueue_f32 fg,
                                  void* user, float factr, float pgtol, int32_t max_iter, int32_t max_fg, float* f, float* g,
                                  char* task, char* csave, int32_t* lsave, int32_t* isave, float* dsave) {
    return minimize_graph_impl<float>(h, x, l, u, nbd, fg, user, factr, pgtol, max_iter, max_fg, f, g, task, csave, lsave, isave, dsave);
}
int lbfgsb_dev_graph_stats(lbfgsb_dev_t* h, int64_t* graph_steps, int64_t* launches_per_step) {
    EngineBase* b = (EngineBase*)h;
    if (!b) return 1;
    if (b->real_kind == 8) { Engine<double>* e = (Engine<double>*)b; *graph_steps = e->graph_steps; *launches_per_step = e->graph_launches_per_step; }
    else { Engine<float>* e = (Engine<float>*)b; *graph_steps = e->graph_steps; *launches_per_step = e->graph_launches_per_step; }
    return 0;
}

int lbfgsb_dev_nccl_unique_id(void* id128) {
    if (!nccl_api()->ok) { set_error("libnccl.so.2 not found"); return 1; }
    return nccl_api()->GetUniqueId((ncclUniqueId*)id128);
}
void* lbfgsb_dev_nccl_init(const void* id128, int32_t rank, int32_t world) {
    if (!nccl_api()->ok) { set_error("libnccl.so.2 not found"); return nullptr; }
    ncclComm_t c = nullptr;
    ncclUniqueId id;
    memcpy(&id, id128, sizeof id);
    int rc = nccl_api()->CommInitRank(&c, world, id, rank);
    if (rc != 0) { set_error("ncclCommInitRank failed: %d", rc); return nullptr; }
    return c;
}
void lbfgsb_dev_nccl_destroy(void* comm) { if (comm && nccl_api()->ok) nccl_api()->CommDestroy((ncclComm_t)comm); }

int lbfgsb_dev_active_set_hash(lbfgsb_dev_t* h, uint64_t* hash, int64_t* count) {
    EngineBase* b = (EngineBase*)h;
    if (!b) return 1;
    i64 c = 0;
    bool ok = (b->real_kind == 8) ? ((Engine<double>*)b)->active_hash(hash, &c) : ((Engine<float>*)b)->active_hash(hash, &c);
    *count = c;
    return ok ? 0 : 1;
}
void* lbfgsb_dev_vector(lbfgsb_dev_t* h, int32_t which) {
    EngineBase* b = (EngineBase*)h;
    if (!b) return nullptr;
#define VSEL(E)                                                                                          \
    switch (which) { case 0: return E->w.z; case 1: return E->w.r; case 2: return E->w.d; case 3: return E->w.t; \
                     case 4: return E->w.xp; case 5: return E->w.ws; case 6: return E->w.wy; case 7: return E->w.iwhere; case 8: return E->w.gold; default: return nullptr; }
    if (b->real_kind == 8) { Engine<double>* e = (Engine<double>*)b; VSEL(e) }
    else { Engine<float>* e = (Engine<float>*)b; VSEL(e) }
}
int lbfgsb_dev_vector_copy(lbfgsb_dev_t* h, int32_t which, void* dst_dev, int64_t bytes) {
    void* src = lbfgsb_dev_vector(h, which);
    if (!src || !dst_dev || bytes < 0) return 1;
    // never copy past the vector's allocation: m columns of ldw reals for ws / wy, ldw int32 for iwhere, ldw reals else
    EngineBase* b = (EngineBase*)h;
    const i64 ldw = (b->real_kind == 8) ? ((Engine<double>*)b)->w.ldw : ((Engine<float>*)b)->w.ldw;
    const i64 m = (b->real_kind == 8) ? ((Engine<double>*)b)->w.m : ((Engine<float>*)b)->w.m;
    const i64 cap = (which == 7) ? ldw * 4 : ((which == 5 || which == 6) ? m : 1) * ldw * (i64)b->real_kind;
    if (bytes > cap) { set_error("lbfgsb_dev_vector_copy: %lld bytes requested, vector %d holds %lld", (long long)bytes, (int)which, (long long)cap); return 1; }
    if (cudaDeviceSynchronize() != cudaSuccess) return 1;
    return cudaMemcpy(dst_dev, src, (size_t)bytes, cudaMemcpyDeviceToDevice) != cudaSuccess;
}
int lbfgsb_dev_exchange_mode(lbfgsb_dev_t* h) {
    EngineBase* b = (EngineBase*)h;
    if (!b) return -1;
    if (b->real_kind == 8) { Engine<double>* e = (Engine<double>*)b; return e->R <= 1 ? 0 : (e->p2p ? 2 : 1); }
    Engine<float>* e = (Engine<float>*)b; return e->R <= 1 ? 0 : (e->p2p ? 2 : 1);
}
int lbfgsb_dev_counters(lbfgsb_dev_t* h, int64_t* launches, int64_t* syncs) {
    EngineBase* b = (EngineBase*)h;
    if (!b) return 1;
    if (b->real_kind == 8) { *launches = ((Engine<double>*)b)->launches; *syncs = ((Engine<double>*)b)->syncs; }
    else { *launches = ((Engine<float>*)b)->launches; *syncs = ((Engine<float>*)b)->syncs; }
    return 0;
}
void lbfgsb_dev_profile(lbfgsb_dev_t* h, int32_t enable) {
    EngineBase* b = (EngineBase*)h;
    if (!b) return;
    if (b->real_kind == 8) ((Engine<double>*)b)->profile = enable != 0; else ((Engine<float>*)b)->profile = enable != 0;
}
void lbfgsb_dev_set_tie_limit(lbfgsb_dev_t* h, int64_t max_breakpoints) {
    EngineBase* b = (EngineBase*)h;
    if (!b) return;
    i64 lim = max_breakpoints < 0 ? 0 : max_breakpoints;
    if (b->real_kind == 8) { Engine<double>* e = (Engine<double>*)b; cudaStreamSynchronize(e->stream); cudaMemcpy(&e->s_dev->tie_limit, &lim, sizeof lim, cudaMemcpyHostToDevice); }
    else { Engine<float>* e = (Engine<float>*)b; cudaStreamSynchronize(e->stream); cudaMemcpy(&e->s_dev->tie_limit, &lim, sizeof lim, cudaMemcpyHostToDevice); }
}
int lbfgsb_dev_tie_stats(lbfgsb_dev_t* h, int64_t* replays, int64_t* not_replayed) {
    EngineBase* b = (EngineBase*)h;
    if (!b) return 1;
    i64 ev = 0;
    cudaError_t e;
    if (b->real_kind == 8) { Engine<double>* g = (Engine<double>*)b; cudaStreamSynchronize(g->stream); e = cudaMemcpy(&ev, &g->s_dev->tie_events, sizeof ev, cudaMemcpyDeviceToHost); *replays = g->tie_replays; }
    else { Engine<float>* g = (Engine<float>*)b; cudaStreamSynchronize(g->stream); e = cudaMemcpy(&ev, &g->s_dev->tie_events, sizeof ev, cudaMemcpyDeviceToHost); *replays = g->tie_replays; }
    *not_replayed = ev;
    return e != cudaSuccess;
}
void lbfgsb_dev_profile_reset(lbfgsb_dev_t* h) {
    EngineBase* b = (EngineBase*)h;
    if (!b) return;
    for (int q = 0; q < F_COUNT; ++q) {
        if (b->real_kind == 8) { ((Engine<double>*)b)->fam_ms[q] = 0; ((Engine<double>*)b)->fam_calls[q] = 0; }
        else { ((Engine<float>*)b)->fam_ms[q] = 0; ((Engine<float>*)b)->fam_calls[q] = 0; }
    }
}
int lbfgsb_dev_profile_read(lbfgsb_dev_t* h, int32_t cap, char* names, double* ms, double* bytes, int64_t* calls) {
    EngineBase* b = (EngineBase*)h;
    if (!b) return 0;
    int k = 0;
    for (int q = 0; q < F_COUNT && k < cap; ++q, ++k) {
        snprintf(names + 32 * k, 32, "%s", fam_name[q]);
        if (b->real_kind == 8) { ms[k] = ((Engine<double>*)b)->fam_ms[q]; calls[k] = ((Engine<double>*)b)->fam_calls[q]; }
        else { ms[k] = ((Engine<float>*)b)->fam_ms[q]; calls[k] = ((Engine<float>*)b)->fam_calls[q]; }
        bytes[k] = 0;
    }
    return k;
}

int64_t lbfgsb_problem_scratch_bytes(void) { return (int64_t)sizeof(double) * (LBFGSB_GRID + 8); }
int lbfgsb_problem_rosenbrock_f64(int64_t n, const double* x, double* g, double* f_out, void* st, int32_t first, int32_t last,
                                  double xl, double xr, void* scratch) {
    return rosenbrock_impl<double>(n, x, g, f_out, st, first, last, xl, xr, scratch);
}
int lbfgsb_problem_rosenbrock_f32(int64_t n, const float* x, float* g, float* f_out, void* st, int32_t first, int32_t last,
                                  float xl, float xr, void* scratch) {
    return rosenbrock_impl<float>(n, x, g, f_out, st, first, last, xl, xr, scratch);
}

int lbfgsb_problem_rosenbrock_halo_f64(int64_t n, const double* x, double* g, double* f_part_dev, void* st, int32_t first,
                                       int32_t last, const double* halo_dev, void* scratch) {
    return rosenbrock_halo_impl<double>(n, x, g, f_part_dev, st, first, last, halo_dev, scratch);
}
int lbfgsb_problem_quadratic_halo_f64(int64_t n, const double* x, double* g, double* f_part_dev, void* st, int64_t off,
                                      uint64_t seed, const double* halo_dev, void* scratch) {
    return quadratic_halo_impl<double>(n, x, g, f_part_dev, st, off, seed, halo_dev, scratch);
}
int lbfgsb_dev_trial_sums(lbfgsb_dev_t* h, lbfgsb_trial_sums_t* out) {
    EngineBase* b = (EngineBase*)h;
    if (!b || !out) return 1;
    memset(out, 0, sizeof *out);
    if (b->real_kind == 8) {
        Engine<double>* e = (Engine<double>*)b;
        out->d_dev = e->w.d; out->gd_part_dev = LB_SLOT(e->w.part, 0); out->pg_part_dev = LB_SLOT(e->w.part, 1); out->n = e->n;
    } else {
        Engine<float>* e = (Engine<float>*)b;
        out->d_dev = e->w.d; out->gd_part_dev = LB_SLOT(e->w.part, 0); out->pg_part_dev = LB_SLOT(e->w.part, 1); out->n = e->n;
    }
    out->grid = LBFGSB_GRID; out->block = LBFGSB_BLOCK; out->unroll = LBFGSB_UNROLL(b->real_kind); out->real_kind = b->real_kind;
    out->vec = LBFGSB_VEC(b->real_kind);
    return 0;
}
void lbfgsb_dev_trial_sums_commit(lbfgsb_dev_t* h) {
    EngineBase* b = (EngineBase*)h;
    if (!b) return;
    if (b->real_kind == 8) ((Engine<double>*)b)->trial_ready = true;   // consumed (or dropped) by the next setulb call
    else ((Engine<float>*)b)->trial_ready = true;
}
int lbfgsb_problem_fused_f64(lbfgsb_dev_t* hh, int32_t kind, const double* x, double* g, const double* l, const double* u,
                             const int32_t* nbd, double* f_out, uint64_t seed) {
    EngineBase* b = (EngineBase*)hh;
    if (!b || b->real_kind != 8) return 2;
    Engine<double>* e = (Engine<double>*)b;
    if (e->R > 1) return 2;
    typedef double T;
    if (!e->fg_scratch) {
        if (!e->dalloc(&e->fg_scratch, sizeof(T) * (LBFGSB_GRID + 8)) || !e->dalloc(&e->fg_out, sizeof(T) * 8)) return 1;
        if (cudaMallocHost((void**)&e->fg_host, sizeof(T) * 8) != cudaSuccess) return 1;
    }
    cudaStream_t st = e->stream;
    const TrialSums<T> ts = trial_sums_of<T>(e, l, u, nbd);
    if (kind == 0) {
        k_rosenbrock<T><<<LBFGSB_GRID, LBFGSB_BLOCK, 0, st>>>(e->n, x, g, e->fg_scratch, 1, 1, (T)0, (T)0, nullptr, ts);
        k_rosenbrock_final<T><<<1, 32, 0, st>>>(e->fg_scratch, e->fg_out);
    } else {
        const unsigned long long seedp = seed * 0x9E3779B97F4A7C15ULL;
        k_quadratic<T><<<LBFGSB_GRID, LBFGSB_BLOCK, 0, st>>>(e->n, x, g, e->fg_scratch, 0, seedp, (T)0, (T)0, nullptr, ts);
        k_sum_final<T><<<1, 32, 0, st>>>(e->fg_scratch, e->fg_out);
    }
    if (cudaMemcpyAsync(e->fg_host, e->fg_out, sizeof(T), cudaMemcpyDeviceToHost, st) != cudaSuccess) return 1;
    if (cudaStreamSynchronize(st) != cudaSuccess) { set_error("objective kernel failed: %s", cudaGetErrorString(cudaGetLastError())); return 1; }
    *f_out = e->fg_host[0];
    return 0;
}
int lbfgsb_problem_sharded_f64(lbfgsb_dev_t* hh, int32_t kind, const double* x, double* g, const double* l, const double* u,
                               const int32_t* nbd, double* f_out, uint64_t seed) {
    EngineBase* b = (EngineBase*)hh;
    if (!b || b->real_kind != 8) return 2;
    Engine<double>* e = (Engine<double>*)b;
    if (e->R <= 1 || !e->p2p) return 2;   // the caller falls back to its own halo exchange and all-reduce
    typedef double T;
    const TrialSums<T> ts = trial_sums_of<T>(e, l, u, nbd);
    if (!e->fg_scratch) {
        if (!e->dalloc(&e->fg_scratch, sizeof(T) * (LBFGSB_GRID + 8)) || !e->dalloc(&e->fg_out, sizeof(T) * 8)) return 1;
        if (cudaMallocHost((void**)&e->fg_host, sizeof(T) * 8) != cudaSuccess) return 1;
    }
    cudaStream_t st = e->stream;
    const unsigned long long seq = ++e->fg_seq;
    const int slot = (int)(seq & 1ULL);
    T* halo = e->fg_out + 2;       // [2]
    T* fpart = e->fg_out + 4;      // [1]
    k_fg_halo_push<T><<<1, 32, 0, st>>>(x, e->n, e->peers, e->R, e->rank, slot, seq);
    k_fg_halo_wait<T><<<1, 32, 0, st>>>(e->w, e->p2p_local, e->R, e->rank, slot, seq, halo);
    if (kind == 0) {
        k_rosenbrock<T><<<LBFGSB_GRID, LBFGSB_BLOCK, 0, st>>>(e->n, x, g, e->fg_scratch, e->rank == 0 ? 1 : 0, e->rank == e->R - 1 ? 1 : 0, (T)0, (T)0, halo, ts);
        k_rosenbrock_final<T><<<1, 32, 0, st>>>(e->fg_scratch, fpart);
    } else {
        const unsigned long long seedp = seed * 0x9E3779B97F4A7C15ULL;
        k_quadratic<T><<<LBFGSB_GRID, LBFGSB_BLOCK, 0, st>>>(e->n, x, g, e->fg_scratch, e->offset, seedp, (T)0, (T)0, halo, ts);
        k_sum_final<T><<<1, 32, 0, st>>>(e->fg_scratch, fpart);
    }
    k_fg_fsum_push<T><<<1, 32, 0, st>>>(fpart, e->peers, e->R, e->rank, slot, seq);
    k_fg_fsum_wait<T><<<1, 32, 0, st>>>(e->w, e->p2p_local, e->R, slot, seq, e->fg_out);
    if (cudaMemcpyAsync(e->fg_host, e->fg_out, sizeof(T), cudaMemcpyDeviceToHost, st) != cudaSuccess) return 1;
    if (cudaStreamSynchronize(st) != cudaSuccess) { set_error("sharded objective failed: %s", cudaGetErrorString(cudaGetLastError())); return 1; }
    *f_out = e->fg_host[0];
    return 0;
}
int lbfgsb_problem_quadratic_f64(int64_t n, const double* x, double* g, double* f_out, void* st, int64_t off, uint64_t seed,
                                 double xl, double xr, void* scratch) {
    return quadratic_impl<double>(n, x, g, f_out, st, off, seed, xl, xr, scratch);
}
int lbfgsb_problem_quadratic_f32(int64_t n, const float* x, float* g, float* f_out, void* st, int64_t off, uint64_t seed,
                                 float xl, float xr, void* scratch) {
    return quadratic_impl<float>(n, x, g, f_out, st, off, seed, xl, xr, scratch);
}

int lbfgsb_test_projgr_f64(int64_t n, const double* l, const double* u, const int32_t* nbd, const double* x, const double* g,
                           double* out) {
    Wk<double> w; memset(&w, 0, sizeof w);
    DevState<double>* s = nullptr; double* part = nullptr;
    if (cudaMalloc(&s, sizeof(DevState<double>)) || cudaMalloc(&part, sizeof(double) * (LBFGSB_GRID + 1))) return 1;
    int one = 1;
    cudaMemcpy(&s->go, &one, sizeof(int), cudaMemcpyHostToDevice);
    w.n = n; w.l = l; w.u = u; w.nbd = nbd; w.x = (double*)x; w.g = (double*)g; w.part = part; w.s = s;
    k_projgr<double><<<LBFGSB_GRID, LBFGSB_BLOCK>>>(w);
    std::vector<double> hp(LBFGSB_GRID);
    cudaError_t e = cudaMemcpy(hp.data(), part, sizeof(double) * LBFGSB_GRID, cudaMemcpyDeviceToHost);
    double r = 0; for (double v : hp) r = v > r ? v : r;
    *out = r;
    cudaFree(s); cudaFree(part);
    return e != cudaSuccess;
}
int lbfgsb_test_sum_f64(int64_t n, const double* a, const double* b, double* out) { return test_sum_impl<double>(n, a, b, out); }
int lbfgsb_test_sum_f32(int64_t n, const float* a, const float* b, float* out) { return test_sum_impl<float>(n, a, b, out); }

int lbfgsb_test_sort_f64(int64_t n, const double* t, int32_t* order_out, double* sorted_out) {
    typedef unsigned long long K;
    K *k0, *k1; int *v0, *v1, *cnt; SortCtl* ctl;
    if (cudaMalloc(&k0, 8 * n) || cudaMalloc(&k1, 8 * n) || cudaMalloc(&v0, 4 * n) || cudaMalloc(&v1, 4 * n) ||
        cudaMalloc(&cnt, 4 * 256 * LB_RS_GRID) || cudaMalloc(&ctl, sizeof(SortCtl))) return 1;
    cudaMemcpy(k0, t, 8 * n, cudaMemcpyDeviceToDevice);   // t > 0: bit pattern order == value order
    k_test_iota<K><<<256, 256>>>(v0, n);
    k_test_setctl<<<1, 32>>>(ctl, n);
    for (int pass = 0; pass < 8; ++pass) {
        k_rs_hist<K><<<LB_RS_GRID, 256>>>(k0, k1, ctl, pass * 8, cnt);
        k_rs_scan<<<1, 1024>>>(cnt, ctl, LB_RS_GRID);
        k_rs_scatter<K><<<LB_RS_GRID, 256>>>(k0, k1, v0, v1, ctl, pass * 8, cnt);
        k_rs_flip<<<1, 32>>>(ctl);
    }
    SortCtl hc;
    cudaMemcpy(&hc, ctl, sizeof hc, cudaMemcpyDeviceToHost);
    cudaMemcpy(order_out, hc.cur ? v1 : v0, 4 * n, cudaMemcpyDeviceToDevice);
    cudaError_t e = cudaMemcpy(sorted_out, hc.cur ? k1 : k0, 8 * n, cudaMemcpyDeviceToDevice);
    cudaFree(k0); cudaFree(k1); cudaFree(v0); cudaFree(v1); cudaFree(cnt); cudaFree(ctl);
    return e != cudaSuccess || cudaGetLastError() != cudaSuccess;
}
// The host thread's heap replay on its own (no GPU): t_host = the breakpoints of a cauchy call in variable order; out = the
// variables whose breakpoint equals tk, in the order in which the reference takes them (the first minimum before the heap
// exists, :1384-1397, the others as hpsolb pops them, :2079-2157).
int lbfgsb_test_host_heap_group_f64(int64_t nb, const double* t_host, double tk, int32_t* group_out, int64_t* group_count) {
    if (nb <= 0 || !t_host || !group_out || !group_count) return 1;
    typedef unsigned long long K;
    std::vector<K> hk((size_t)nb); std::vector<int> hv((size_t)nb);
    int vmin = 0;
    for (int64_t i = 0; i < nb; ++i) {
        memcpy(&hk[(size_t)i], &t_host[i], 8); hv[(size_t)i] = (int)i;
        if (t_host[i] < t_host[vmin]) vmin = (int)i;   // strict <: lowest index among ties (:1310)
    }
    K kk; memcpy(&kk, &tk, 8);
    std::vector<K> gk; std::vector<int> gv;
    Engine<double>::heap_group_order<K>(kk, hk, hv, vmin, gk, gv);
    for (size_t i = 0; i < gv.size(); ++i) group_out[i] = gv[i];
    *group_count = (int64_t)gv.size();
    return 0;
}
int lbfgsb_test_heap_order_f64(int64_t n, const double* t, int32_t* order_out) {
    unsigned long long* k; int* v;
    if (n <= 0) return 1;
    if (cudaMalloc(&k, 8 * n) || cudaMalloc(&v, 4 * n)) return 1;
    cudaMemcpy(k, t, 8 * n, cudaMemcpyDeviceToDevice);   // t >= 0: bit pattern order == value order
    k_test_iota<unsigned long long><<<256, 256>>>(v, n);
    k_test_heap_order<<<1, 32>>>(k, v, n, order_out);
    cudaError_t e = cudaDeviceSynchronize();
    cudaFree(k); cudaFree(v);
    return e != cudaSuccess || cudaGetLastError() != cudaSuccess;
}
int lbfgsb_test_formk_delta_f64(int64_t n, int32_t m, int32_t col, int32_t head, int64_t ldw, const double* ws, const double* wy,
                                const unsigned char* state, double* out_host) {
    return test_formk_delta_impl<double>(n, m, col, head, ldw, ws, wy, state, out_host);
}
int lbfgsb_test_formk_delta_f32(int64_t n, int32_t m, int32_t col, int32_t head, int64_t ldw, const float* ws, const float* wy,
                                const unsigned char* state, float* out_host) {
    return test_formk_delta_impl<float>(n, m, col, head, ldw, ws, wy, state, out_host);
}
int lbfgsb_test_dense_f64(int32_t op, int32_t m, int32_t col, double theta, double* a, double* b, double* c, int32_t* info) {
    int* dinfo; DevState<double>* st;
    if (cudaMalloc(&dinfo, 4) || cudaMalloc(&st, sizeof(DevState<double>))) return 1;
    cudaMemset(st, 0, sizeof(DevState<double>));
    k_test_dense<<<1, 32>>>(op, m, col, theta, a, b, c, dinfo, st);
    cudaError_t e = cudaMemcpy(info, dinfo, 4, cudaMemcpyDeviceToHost);
    cudaFree(dinfo); cudaFree(st);
    return e != cudaSuccess;
}
int lbfgsb_test_dcsrch_f64(double f, double g, double* stp, double stpmax, int32_t* task, int32_t* isave2, double* dsave13) {
    double *dstp, *dds; int *dtask, *dis;
    if (cudaMalloc(&dstp, 8) || cudaMalloc(&dds, 8 * 13) || cudaMalloc(&dtask, 4) || cudaMalloc(&dis, 8)) return 1;
    cudaMemcpy(dstp, stp, 8, cudaMemcpyHostToDevice); cudaMemcpy(dds, dsave13, 8 * 13, cudaMemcpyHostToDevice);
    cudaMemcpy(dtask, task, 4, cudaMemcpyHostToDevice); cudaMemcpy(dis, isave2, 8, cudaMemcpyHostToDevice);
    k_test_dcsrch<<<1, 32>>>(f, g, dstp, stpmax, dtask, dis, dds);
    cudaMemcpy(stp, dstp, 8, cudaMemcpyDeviceToHost); cudaMemcpy(dsave13, dds, 8 * 13, cudaMemcpyDeviceToHost);
    cudaMemcpy(task, dtask, 4, cudaMemcpyDeviceToHost);
    cudaError_t e = cudaMemcpy(isave2, dis, 8, cudaMemcpyDeviceToHost);
    cudaFree(dstp); cudaFree(dds); cudaFree(dtask); cudaFree(dis);
    return e != cudaSuccess;
}

// ---- batched small problems ----
lbfgsb_batch_t* lbfgsb_batch_create(int32_t nprob, int64_t n, int32_t m, int32_t real_kind, void* cuda_stream) {
    if (nprob <= 0 || n <= 0 || m <= 0 || m > LB_MMAX) { set_error("lbfgsb_batch_create: need nprob > 0, n > 0 and 0 < m <= %d", LB_MMAX); return nullptr; }
    const int64_t nmax = (int64_t)LB_BATCH_MAXTILES * LBFGSB_BLOCK * LBFGSB_UNROLL(real_kind) * LBFGSB_VEC(real_kind);
    if (real_kind != 8 && real_kind != 4) { set_error("real_kind must be 8 or 4"); return nullptr; }
    if (n > nmax) { set_error("lbfgsb_batch_create: n = %lld exceeds the one-CTA-per-problem limit of %lld variables", (long long)n, (long long)nmax); return nullptr; }
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) { set_error("no CUDA device (lbfgsb_b200 has no CPU path)"); return nullptr; }
    if (real_kind == 8) {
        BatchEngine<double>* e = new BatchEngine<double>();
        if (!e->init(nprob, n, m, (cudaStream_t)cuda_stream)) { delete e; return nullptr; }
        return (lbfgsb_batch_t*)e;
    }
    BatchEngine<float>* e = new BatchEngine<float>();
    if (!e->init(nprob, n, m, (cudaStream_t)cuda_stream)) { delete e; return nullptr; }
    return (lbfgsb_batch_t*)e;
}
void lbfgsb_batch_destroy(lbfgsb_batch_t* h) { delete (BatchBase*)h; }
void lbfgsb_batch_setulb_dev_f64(lbfgsb_batch_t* h, double* x, const double* l, const double* u, const int32_t* nbd, double* f_dev, double* g,
                                 const double* factr, const double* pgtol, char* task, char* csave, int32_t* lsave, int32_t* isave,
                                 double* dsave) {
    BatchBase* b = (BatchBase*)h;
    if (!b || b->real_kind != 8) { set_error("invalid batch handle"); if (task) put60(task, "ERROR: INVALID LBFGSB_B200 HANDLE"); return; }
    BatchEngine<double>* e = (BatchEngine<double>*)b;
    if (!e->call(x, l, u, nbd, f_dev, g, *factr, *pgtol, task, csave, lsave, isave, dsave))
        for (int p = 0; p < e->bw.nprob; ++p) put60(task + 60 * (size_t)p, "ERROR: CUDA FAILURE (see lbfgsb_b200_last_error)");
}
void lbfgsb_batch_setulb_dev_f32(lbfgsb_batch_t* h, float* x, const float* l, const float* u, const int32_t* nbd, float* f_dev, float* g,
                                 const float* factr, const float* pgtol, char* task, char* csave, int32_t* lsave, int32_t* isave,
                                 float* dsave) {
    BatchBase* b = (BatchBase*)h;
    if (!b || b->real_kind != 4) { set_error("invalid batch handle"); if (task) put60(task, "ERROR: INVALID LBFGSB_B200 HANDLE"); return; }
    BatchEngine<float>* e = (BatchEngine<float>*)b;
    if (!e->call(x, l, u, nbd, f_dev, g, *factr, *pgtol, task, csave, lsave, isave, dsave))
        for (int p = 0; p < e->bw.nprob; ++p) put60(task + 60 * (size_t)p, "ERROR: CUDA FAILURE (see lbfgsb_b200_last_error)");
}
int lbfgsb_batch_counts(lbfgsb_batch_t* h, int32_t* n_fg, int32_t* n_newx, int32_t* n_done) {
    BatchBase* b = (BatchBase*)h;
    if (!b) return 1;
    if (b->real_kind == 8) { BatchEngine<double>* e = (BatchEngine<double>*)b; *n_fg = e->n_fg; *n_newx = e->n_newx; *n_done = e->n_done; }
    else { BatchEngine<float>* e = (BatchEngine<float>*)b; *n_fg = e->n_fg; *n_newx = e->n_newx; *n_done = e->n_done; }
    return 0;
}
void* lbfgsb_batch_fg_mask(lbfgsb_batch_t* h) {
    BatchBase* b = (BatchBase*)h;
    if (!b) return nullptr;
    return b->real_kind == 8 ? (void*)((BatchEngine<double>*)b)->bw.fgmask : (void*)((BatchEngine<float>*)b)->bw.fgmask;
}
int lbfgsb_batch_get_iwhere(lbfgsb_batch_t* h, int32_t* iwhere_host) {
    BatchBase* b = (BatchBase*)h;
    if (!b || !iwhere_host) return 1;
    const int* src; i64 ldw, n; int nprob; cudaStream_t st;
    if (b->real_kind == 8) { BatchEngine<double>* e = (BatchEngine<double>*)b; src = e->bw.iwhere; ldw = e->bw.ldw; n = e->bw.n; nprob = e->bw.nprob; st = e->stream; }
    else { BatchEngine<float>* e = (BatchEngine<float>*)b; src = e->bw.iwhere; ldw = e->bw.ldw; n = e->bw.n; nprob = e->bw.nprob; st = e->stream; }
    if (cudaMemcpy2DAsync(iwhere_host, (size_t)n * 4, src, (size_t)ldw * 4, (size_t)n * 4, (size_t)nprob, cudaMemcpyDeviceToHost, st) != cudaSuccess) return 1;
    return cudaStreamSynchronize(st) != cudaSuccess;
}
int lbfgsb_batch_vector_copy(lbfgsb_batch_t* h, int32_t problem, int32_t which, void* dst_dev, int64_t bytes) {
    BatchBase* b = (BatchBase*)h;
    if (!b || !dst_dev || bytes < 0) return 1;
    if (b->real_kind == 8) return ((BatchEngine<double>*)b)->vector_copy(problem, which, dst_dev, bytes);
    return ((BatchEngine<float>*)b)->vector_copy(problem, which, dst_dev, bytes);
}
void* lbfgsb_batch_stream(lbfgsb_batch_t* h) {
    BatchBase* b = (BatchBase*)h;
    if (!b) return nullptr;
    return b->real_kind == 8 ? (void*)((BatchEngine<double>*)b)->stream : (void*)((BatchEngine<float>*)b)->stream;
}
int lbfgsb_problem_rosenbrock_batch_f64(int32_t nprob, int64_t n, const double* x_dev, double* g_dev, double* f_dev, const int32_t* mask_dev,
                                        void* st) {
    static bool attr = false;
    if (!attr) { cudaFuncSetAttribute(k_rosenbrock_batch<double>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(BatchSm<double>)); attr = true; }
    k_rosenbrock_batch<double><<<nprob, LBFGSB_BLOCK, sizeof(BatchSm<double>), (cudaStream_t)st>>>(nprob, n, x_dev, g_dev, f_dev, mask_dev);
    return cudaGetLastError() != cudaSuccess;
}
int lbfgsb_problem_rosenbrock_batch_f32(int32_t nprob, int64_t n, const float* x_dev, float* g_dev, float* f_dev, const int32_t* mask_dev,
                                        void* st) {
    static bool attr = false;
    if (!attr) { cudaFuncSetAttribute(k_rosenbrock_batch<float>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(BatchSm<float>)); attr = true; }
    k_rosenbrock_batch<float><<<nprob, LBFGSB_BLOCK, sizeof(BatchSm<float>), (cudaStream_t)st>>>(nprob, n, x_dev, g_dev, f_dev, mask_dev);
    return cudaGetLastError() != cudaSuccess;
}

}  // extern "C"

