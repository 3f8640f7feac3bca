// The generalized-Cauchy-point search on a problem sharded over R GPUs
// (src/lbfgsb.f90:1378-1497 needs the breakpoints of ALL variables in increasing t).
//
//   1. every rank compacts and radix-sorts its own breakpoints (cauchy_walk.cuh);
//   2. sample sort: S regular samples (t, global index) per rank are all-gathered, every rank
//      derives the same R-1 splitters, and cuts its sorted list at them (k_dw_partition);
//   3. one record per breakpoint -- t, d_i, z_i and the row of [Y theta*S] -- is packed in sorted
//      order (k_dw_pack) and exchanged so that rank r receives the r-th key range of every
//      rank (grouped ncclSend/ncclRecv = all-to-all-v over NVLink);
//   4. the received runs are concatenated in source-rank order (= global index order, the
//      shards being contiguous blocks) and stably sorted by t, which reproduces the single-GPU
//      order (t, index) exactly;
//   5. the scans of cauchy_walk.cuh run over each rank's range in rank order, the carries
//      (two 2col-vector prefix sums, f1, f2, the last two keys, the exit) travel from rank to
//      rank in an all-gathered record (k_dw_turn_end / k_dw_adopt);
//   6. every rank fixes those of its own variables that precede the exit (k_dw_fixcount
//      tells it how many of its records do).
#pragma once
#include "cauchy_walk.cuh"

#define LB_MAXR 16          // ranks on one node
#define LB_DW_SAMPLES 64    // samples per rank

struct DwCtl {
    i64 pos[LB_MAXR + 1];   // cut positions of the local sorted list (destination q gets [pos[q], pos[q+1]))
    i64 roff[LB_MAXR + 1];  // offsets of the received runs by source rank; roff[R] = nrecv
    i64 goff;               // breakpoints held by lower ranks (global position of this rank's first)
    i64 nb_glob;            // all breakpoints
    i64 fixcnt[LB_MAXR];    // per source rank: records of that rank that precede the exit in this rank's range
    i64 jloc;               // how many entries of the local sorted list are fixed
};

template <typename T>
struct WalkCarry {
    T A[2 * LB_MMAX], B[2 * LB_MMAX];
    T f1, f2, tlast, tprev2;
    i64 found;              // 1: the exit lies in the sender's range (or before); 2: it lies inside a group of equal
                            // breakpoints that is to be replayed in the reference's heap order (tie_key); nothing is closed
    unsigned long long tie_key;
    i64 tie_unreplayed;     // found = 1 inside such a group, but the heap is too long to replay: counted
    i64 fixcnt[LB_MAXR];
    // valid when found:
    T fin_f1, fin_f2, dtm, tsum;
    i64 nseg;
    T p[2 * LB_MMAX], c[2 * LB_MMAX];
};

// (key, global index) lexicographic compare
__device__ __forceinline__ bool dw_less(unsigned long long ka, i64 ga, unsigned long long kb, i64 gb) {
    return ka < kb || (ka == kb && ga < gb);
}

// S regular samples of the local sorted list; sentinel (max, max) when the list is empty.
// out: [S] keys as 64-bit, then [S] global indices, then 1 entry: the local count.
template <typename T>
__global__ void k_dw_sample(Wk<T> w, WalkBuf<T> b, unsigned long long* out) {
    const int i = threadIdx.x;
    const i64 cnt = b.ctl->count;
    if (i < LB_DW_SAMPLES) {
        unsigned long long k = 0xffffffffffffffffULL;
        i64 g = LB_I64MAX;
        if (cnt > 0) {
            const i64 idx = ((2 * (i64)i + 1) * cnt) / (2 * LB_DW_SAMPLES);
            k = (unsigned long long)cur_keys<T>(b)[idx];
            g = w.off + (i64)cur_vals<T>(b)[idx];
        }
        out[i] = k;
        out[LB_DW_SAMPLES + i] = (unsigned long long)g;
    }
    if (i == 0) out[2 * LB_DW_SAMPLES] = (unsigned long long)cnt;
}

// cut positions: pos[q] = first local entry with (key, gidx) >= splitter q  (q = 1..R-1)
template <typename T>
__global__ void k_dw_partition(Wk<T> w, WalkBuf<T> b, int R, const unsigned long long* spl /* [R-1] keys, [R-1] gidx */, DwCtl* dc) {
    const int q = threadIdx.x;
    if (q > R) return;
    const i64 cnt = b.ctl->count;
    if (q == 0) { dc->pos[0] = 0; return; }
    if (q == R) { dc->pos[R] = cnt; return; }
    const unsigned long long sk = spl[q - 1];
    const i64 sg = (i64)spl[(R - 1) + (q - 1)];
    const typename Real<T>::key_t* keys = cur_keys<T>(b);
    const int* vals = cur_vals<T>(b);
    i64 lo = 0, hi = cnt;
    while (lo < hi) {
        const i64 mid = (lo + hi) >> 1;
        if (dw_less((unsigned long long)keys[mid], w.off + (i64)vals[mid], sk, sg)) lo = mid + 1; else hi = mid;
    }
    dc->pos[q] = lo;
}

// records of the local breakpoints in sorted order: [t, d, z, Wy row (col), theta*Ws row (col)]
template <typename T>
__global__ void __launch_bounds__(256) k_dw_pack(Wk<T> w, WalkBuf<T> b, T* rec, int rs) {
    const DevState<T>* s = w.s;
    const int col = s->col, m = s->m, head0 = s->head - 1;
    const T theta = s->theta;
    const i64 cnt = b.ctl->count;
    const typename Real<T>::key_t* keys = cur_keys<T>(b);
    const int* vals = cur_vals<T>(b);
    for (i64 j = (i64)blockIdx.x * blockDim.x + threadIdx.x; j < cnt; j += (i64)gridDim.x * blockDim.x) {
        const int var = vals[j];
        const T dl = cauchy_dir<T>(w.iwhere[var], w.g[var]);
        T* r = rec + j * rs;
        // what the receiver sorts by: t -- or, in a replayed tie group, the member's position in the heap order
        r[0] = (s->tie_round == 2) ? (T)(i64)keys[j] : KeyBits<T>::from(keys[j]);
        r[1] = dl;
        r[2] = (dl > (T)0) ? (w.u[var] - w.x[var]) : (w.l[var] - w.x[var]);
        int pj = head0;
        for (int c = 0; c < col; ++c) {
            r[3 + c] = w.wy[(i64)pj * w.ldw + var];
            r[3 + col + c] = theta * w.ws[(i64)pj * w.ldw + var];
            pj = (pj + 1 == m) ? 0 : pj + 1;
        }
    }
}

// sort keys of the received records: key = bits of t, value = record number
template <typename T>
__global__ void __launch_bounds__(256) k_dw_keys(const T* rec, int rs, i64 nrecv, typename Real<T>::key_t* keys, int* vals, SortCtl* ctl) {
    for (i64 j = (i64)blockIdx.x * blockDim.x + threadIdx.x; j < nrecv; j += (i64)gridDim.x * blockDim.x) {
        keys[j] = KeyBits<T>::to(rec[j * rs]);
        vals[j] = (int)j;
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) { ctl->count = nrecv; ctl->cur = 0; ctl->skip = 0; }
}

// gather of one chunk from the received records (the sharded twin of k_walk_gather)
template <typename T>
__global__ void __launch_bounds__(LB_WB) k_dw_gather(Wk<T> w, WalkBuf<T> b, const T* rec, int rs, i64 start, i64 len) {
    const DevState<T>* s = w.s;
    if (!s->go || !s->in_body || !s->need_walk || s->walk_J >= 0) return;
    const int col = s->col, col2 = 2 * col, m = s->m;
    __shared__ T ssy[LB_MMAX * LB_MMAX], swt[LB_MMAX * LB_MMAX];
    __shared__ T red[LB_WB / 32];
    for (int q = threadIdx.x; q < m * m; q += LB_WB) { ssy[q] = s->sy[q]; swt[q] = s->wt[q]; }
    __syncthreads();
    const i64 j = (i64)blockIdx.x * LB_WB + threadIdx.x;
    const bool ok = j < len;
    T dl = (T)0, ze = (T)0;
    T wl[2 * LB_MMAX], vl[2 * LB_MMAX];
    if (ok) {
        const T* r = rec + (i64)cur_vals<T>(b)[start + j] * rs;
        dl = r[1]; ze = r[2];
        b.delta[j] = dl; b.zeta[j] = ze;
        if (col > 0) {
            for (int c = 0; c < col2; ++c) wl[c] = r[3 + c];
            dense::bmv<T>(m, ssy, swt, col, wl, vl);
            T om = (T)0;
            for (int c = 0; c < col2; ++c) { om = om + wl[c] * vl[c]; b.wj[(i64)c * b.cap + j] = wl[c]; b.vj[(i64)c * b.cap + j] = vl[c]; }
            b.omega[j] = om;
        } else b.omega[j] = (T)0;
    }
    for (int c = 0; c < col2; ++c) {
        for (int which = 0; which < 2; ++which) {
            T v = ok ? ((which == 0 ? dl : ze) * wl[c]) : (T)0;
            v = warp_sum<T>(v);
            if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
            __syncthreads();
            if (threadIdx.x == 0) {
                T t = red[0];
                for (int q = 1; q < LB_WB / 32; ++q) t = t + red[q];
                (which == 0 ? b.blkA : b.blkB)[(i64)blockIdx.x * (2 * LB_MMAX) + c] = t;
            }
            __syncthreads();
        }
    }
}

// how many records of each source rank precede the exit position in this rank's sorted range
template <typename T>
__global__ void __launch_bounds__(256) k_dw_fixcount(Wk<T> w, WalkBuf<T> b, int R, DwCtl* dc) {
    const DevState<T>* s = w.s;
    const i64 J = s->walk_J;
    if (!s->go || !s->in_body || !s->need_walk || J < 0 || J == LB_I64MAX) return;
    const int* vals = cur_vals<T>(b);
    i64 cnt[LB_MAXR];
#pragma unroll
    for (int q = 0; q < LB_MAXR; ++q) cnt[q] = 0;
    for (i64 j = (i64)blockIdx.x * blockDim.x + threadIdx.x; j < J; j += (i64)gridDim.x * blockDim.x) {
        const i64 p = vals[j];
#pragma unroll
        for (int q = 0; q < LB_MAXR; ++q)
            if (q < R && p >= dc->roff[q] && p < dc->roff[q + 1]) cnt[q]++;
    }
#pragma unroll
    for (int q = 0; q < LB_MAXR; ++q) {
        if (q < R) {
            const i64 v = warp_sum<i64>(cnt[q]);
            if ((threadIdx.x & 31) == 0 && v) atomicAdd((unsigned long long*)&dc->fixcnt[q], (unsigned long long)v);
        }
    }
}

// End of a rank's turn: the carry it hands on.  One block of LB_WB threads.
// `mine`: this rank just ran its chunks (otherwise the record is a placeholder).
template <typename T>
__global__ void __launch_bounds__(LB_WB) k_dw_turn_end(Wk<T> w, WalkBuf<T> b, const DwCtl* dc, i64 chunk_cap, int mine, int R,
                                                      WalkCarry<T>* out) {
    DevState<T>* s = w.s;
    __shared__ T AJ[2 * LB_MMAX], BJ[2 * LB_MMAX];
    __shared__ T sm[33];
    if (!s->go || !s->in_body || !s->need_walk) return;
    const int col = s->col, col2 = 2 * col;
    const i64 nrecv = dc->roff[R];
    const i64 J = s->walk_J;
    if (!mine) { if (threadIdx.x == 0) out->found = 0; return; }
    if (J >= 0 && J != LB_I64MAX) {
        // the exit is in this rank's range: state at the exit (as k_walk_final)
        const typename Real<T>::key_t* keys = cur_keys<T>(b);
        const i64 start = (J / chunk_cap) * chunk_cap;
        const i64 jl = J - start;
        const i64 blk = jl / LB_WB;
        const i64 j = blk * LB_WB + threadIdx.x;
        const bool in = j < jl;
        for (int c = 0; c < col2; ++c) {
            const T wv_ = in ? b.wj[(i64)c * b.cap + j] : (T)0;
            T tot;
            block_excl_scan<T>(in ? b.delta[j] * wv_ : (T)0, sm, tot);
            if (threadIdx.x == 0) AJ[c] = b.blkA[blk * (2 * LB_MMAX) + c] + tot;
            block_excl_scan<T>(in ? b.zeta[j] * wv_ : (T)0, sm, tot);
            if (threadIdx.x == 0) BJ[c] = b.blkB[blk * (2 * LB_MMAX) + c] + tot;
        }
        __syncthreads();
        if (threadIdx.x != 0) return;
        out->tie_unreplayed = 0;
        if (!s->tie_round) {
            // the exit inside a group of equal breakpoints (cauchy_walk.cuh "heap replay"): the entry before the exit is
            // the one before J in this range, or the last entry of the lower ranks' ranges (its t is the carried tlast)
            const bool tie = (J > 0) ? (keys[J - 1] == keys[J]) : (dc->goff > 0 && KeyBits<T>::to(s->walk_tlast) == keys[0]);
            if (tie) {
                if (s->tie_limit > 0 && s->nbreak <= s->tie_limit) {
                    out->found = 2; out->tie_key = (unsigned long long)keys[J];
                    for (int q = 0; q < R; ++q) out->fixcnt[q] = 0;
                    return;
                }
                out->tie_unreplayed = 1;
            }
        }
        const T f1 = b.f1a[jl], f2 = b.f2a[jl];
        const T tprev = (J > 0) ? walk_t_of<T>(s, keys[J - 1]) : s->walk_tlast;
        T dtm = -f1 / f2;
        if (dtm <= (T)0) dtm = (T)0;
        out->found = 1;
        out->fin_f1 = f1; out->fin_f2 = f2; out->dtm = dtm; out->tsum = tprev + dtm;
        out->nseg = 1 + s->walk_base + dc->goff + J;
        for (int c = 0; c < col2; ++c) {
            const T pJ = s->p0[c] - AJ[c];
            out->p[c] = pJ;
            out->c[c] = (tprev * pJ + BJ[c]) + dtm * pJ;
        }
        for (int q = 0; q < R; ++q) out->fixcnt[q] = dc->fixcnt[q];
        return;
    }
    if (threadIdx.x != 0) return;
    // every breakpoint of this range was passed: hand on the running state
    const typename Real<T>::key_t* keys = cur_keys<T>(b);
    out->found = 0;
    for (int c = 0; c < col2; ++c) { out->A[c] = s->walkA[c]; out->B[c] = s->walkB[c]; }
    out->f1 = s->walk_f1; out->f2 = s->walk_f2;
    if (nrecv >= 2) { out->tlast = walk_t_of<T>(s, keys[nrecv - 1]); out->tprev2 = walk_t_of<T>(s, keys[nrecv - 2]); }
    else if (nrecv == 1) { out->tlast = walk_t_of<T>(s, keys[0]); out->tprev2 = s->walk_tlast; }
    else { out->tlast = s->walk_tlast; out->tprev2 = s->walk_tprev2; }
}

// Every rank adopts the carry of rank `turn`; after the last turn of the last round the search is
// closed (all-passed exits :1436-1442, :1484-1495, walk_close_all_passed).
template <typename T>
__global__ void k_dw_adopt(Wk<T> w, const WalkCarry<T>* all, int turn, int R, int rank, DwCtl* dc, i64 n_global) {
    if (threadIdx.x != 0) return;
    DevState<T>* s = w.s;
    if (!s->go || !s->in_body || !s->need_walk) return;
    if (s->walk_J == LB_I64MAX) return;   // already closed by an earlier turn
    const WalkCarry<T>* cr = all + turn;
    const int col2 = 2 * s->col;
    if (cr->found == 2) {   // redo the round up to the tie group, then the group in heap order (Engine::tie_replay)
        s->tie_redo = 1; s->tie_key = cr->tie_key;
        s->walk_J = LB_I64MAX;   // the later turns of this round do nothing
        dc->jloc = 0;
        return;
    }
    if (cr->found) {
        if (cr->tie_unreplayed) s->tie_events += 1;
        s->f1 = cr->fin_f1; s->f2 = cr->fin_f2; s->dtm = cr->dtm; s->tsum = cr->tsum; s->nseg = cr->nseg;
        for (int c = 0; c < col2; ++c) { s->p[c] = cr->p[c]; s->c[c] = cr->c[c]; }
        // my entries before the exit: everything I sent to lower ranks + my records before J on rank `turn`
        dc->jloc = dc->pos[turn] + cr->fixcnt[rank];
        s->walk_J = LB_I64MAX;
        s->walk_closed = 1;
        return;
    }
    for (int c = 0; c < col2; ++c) { s->walkA[c] = cr->A[c]; s->walkB[c] = cr->B[c]; }
    s->walk_f1 = cr->f1; s->walk_f2 = cr->f2; s->walk_tlast = cr->tlast; s->walk_tprev2 = cr->tprev2;
    s->walk_J = -1;
    if (turn != R - 1) return;
    // every breakpoint of this round was passed
    s->walk_base += dc->nb_glob;
    dc->jloc = dc->pos[R];
    if (dc->nb_glob == s->walk_rem) { walk_close_all_passed<T>(s, n_global); s->walk_J = LB_I64MAX; }
}

// fix the first dc->jloc entries of the LOCAL sorted list (:1424-1434)
template <typename T>
__global__ void __launch_bounds__(256) k_dw_fix(Wk<T> w, WalkBuf<T> b, const DwCtl* dc) {
    const DevState<T>* s = w.s;
    if (!s->go || !s->in_body || !s->need_walk) return;
    const i64 J = dc->jloc;
    const int* vals = cur_vals<T>(b);
    for (i64 j = (i64)blockIdx.x * blockDim.x + threadIdx.x; j < J; j += (i64)gridDim.x * blockDim.x) {
        const int var = vals[j];
        const T dl = cauchy_dir<T>(w.iwhere[var], w.g[var]);
        if (dl > (T)0) { w.z[var] = w.u[var]; w.iwhere[var] = 2; }
        else { w.z[var] = w.l[var]; w.iwhere[var] = 1; }
        w.r[var] = (T)-1;   // no breakpoint any more (cauchy_walk.cuh: the stored breakpoints)
    }
}

// ---------------------------------------------------------------------------
// Small rounds (at most LB_RW_MAX breakpoints over all ranks -- the usual case: the search passes a few hundred).
// The sample sort above costs a hundred small launches, R all-gathers and two host read-backs whatever the size.
// Instead every rank all-gathers ALL records of the round (cap per rank, padded) and runs the single-GPU scans over the
// whole list redundantly: concatenated in rank order and stably sorted by key the list is the global (t, index) order,
// the scans are those of cauchy_walk.cuh on the same operands in the same order on every rank, and each rank fixes
// those of its own variables that were passed.
// ---------------------------------------------------------------------------
#define LB_RW_MAX 4096
// this rank's count of the round into its RoundRec (all-gathered next)
template <typename T>
__global__ void k_rw_count(Wk<T> w, WalkBuf<T> b, RoundRec* out) {
    if (threadIdx.x != 0) return;
    out->count = b.ctl->count; out->rem = 0; out->kmin = 0; out->pad = 0;
}
// sort keys of the gathered records: rank q's first count_q records of its block of `cap`, in rank order
template <typename T>
__global__ void __launch_bounds__(256) k_rw_keys(const T* rec, int rs, i64 cap, const RoundRec* all, int R,
                                                 typename Real<T>::key_t* keys, int* vals, SortCtl* ctl) {
    i64 off = 0;
    for (int q = 0; q < R; ++q) {
        const i64 c = all[q].count;
        for (i64 i = (i64)blockIdx.x * blockDim.x + threadIdx.x; i < c; i += (i64)gridDim.x * blockDim.x) {
            const i64 r = (i64)q * cap + i;
            keys[off + i] = KeyBits<T>::to(rec[r * rs]);
            vals[off + i] = (int)r;
        }
        off += c;
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) { ctl->count = off; ctl->cur = 0; ctl->skip = 0; }
}
// fix this rank's variables among the first walk_fixn entries of the global sorted list (:1424-1434):
// record number q * cap + i is entry i of rank q's local sorted list
template <typename T>
__global__ void __launch_bounds__(256) k_rw_fix(Wk<T> w, WalkBuf<T> local, WalkBuf<T> global, i64 cap, int rank) {
    const DevState<T>* s = w.s;
    if (!s->go || !s->in_body || !s->need_walk) return;
    const i64 J = s->walk_fixn;
    const int* gv = cur_vals<T>(global);
    const int* lv = cur_vals<T>(local);
    for (i64 j = (i64)blockIdx.x * blockDim.x + threadIdx.x; j < J; j += (i64)gridDim.x * blockDim.x) {
        const i64 r = gv[j];
        if (r / cap != rank) continue;
        const int var = lv[r % cap];
        const T dl = cauchy_dir<T>(w.iwhere[var], w.g[var]);
        if (dl > (T)0) { w.z[var] = w.u[var]; w.iwhere[var] = 2; }
        else { w.z[var] = w.l[var]; w.iwhere[var] = 1; }
        w.r[var] = (T)-1;
    }
}

