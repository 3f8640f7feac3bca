// Batched small problems (SURVEY.md section 8 f4): many independent bound-constrained problems of the same
// size, ONE CTA PER PROBLEM, one kernel launch per reverse-communication call for the whole batch.
//
// The reference keeps no state between calls (src/lbfgsb.f90:52-56), so a caller with thousands of small boxes
// runs thousands of independent copies of the task loop of test/driver1.f90:263-292.  Here every problem has its
// own state block (DevState, the same one the large-n engine uses), its own task, isave, dsave, and the batch
// advances with one call: each CTA takes its problem from its current task to the next return point of mainlb
// (:552-872) -- 'FG_START', 'FG_LNSRCH', 'NEW_X' or a terminal task -- exactly as setulb would.
//
// Arithmetic.  Per-variable loops follow the formulas of the unfused streaming kernels (kernels_stream.cuh,
// kernels_tma.cuh) and every O(n) sum is formed in the engine's fixed reduction shape
// (include/lbfgsb_b200_shape.h): the CTA plays the blocks 0..ntiles-1 of the 592-block grid one after the other
// (n <= 32 tiles, i.e. 65 536 real64 / 131 072 real32 variables, so every grid block owns at most one tile) and a
// warp finishes the tile partials lane by lane like final_sum_warp.  The 2m x 2m algebra and the line search are
// the very functions the scalar kernels of the engine run (kernels_dense.cuh w_*, t0_*).  The generalized Cauchy
// point is found as the reference finds it: one thread pops the breakpoints from hpsolb's heap (:1378-1497,
// :2079-2157), so equal breakpoints are taken in the reference's order by construction.
#pragma once
#include "cauchy_walk.cuh"

#define LB_BATCH_MAXTILES 32

template <typename T>
struct BatchWk {
    int nprob, m, mt;
    i64 n, ldw;
    // caller's arrays, [nprob][n]; f [nprob]
    T* x; const T* l; const T* u; const int* nbd; T* g; T* f;
    // workspace, problem-major
    T *ws, *wy;                           // [nprob][m][ldw]
    T *z, *r, *d, *t, *xp, *gold, *bpt;   // [nprob][ldw]
    int *iwhere, *bpo;                    // [nprob][ldw]
    unsigned char* state;                 // [nprob][ldw]
    T* delta;                             // [nprob][6*MMAX*MMAX]
    DevState<T>* s;                       // [nprob]
    const int* entry;                     // [nprob] what the caller's task asks for (BE_*)
    int* fgmask;                          // [nprob] out: 1 where the problem's new task asks for f and g
    T factr, pgtol;
};
enum { BE_START = 0, BE_FG_START = 1, BE_FG_LNSRCH = 2, BE_NEW_X = 3, BE_STOP = 4, BE_STOP_CPU = 5, BE_OTHER = 6, BE_IDLE = 7 };

// shared scratch of one CTA (dynamic shared memory)
template <typename T>
struct BatchSm {
    Red<T> red;
    T warp[LB_KMAX * (LBFGSB_BLOCK / 32)];      // per-warp sums of one tile
    T tile[LB_KMAX * LB_BATCH_MAXTILES];        // tile partials (= the engine's block partials)
    T sy[LB_MMAX * LB_MMAX], ss[LB_MMAX * LB_MMAX], wt[LB_MMAX * LB_MMAX];
    T wn[4 * LB_MMAX * LB_MMAX], wn1[4 * LB_MMAX * LB_MMAX];
    T smv[LBFGSB_BLOCK / 32]; i64 smi[LBFGSB_BLOCK / 32]; i64 scan[33];
    T coef[4 * LB_MMAX];
    i64 bc[4];
};

namespace batch {

template <typename T> __device__ __forceinline__ i64 tile_size() { return (i64)LBFGSB_BLOCK * Real<T>::VEC * Real<T>::UNROLL; }
template <typename T> __device__ __forceinline__ i64 ntiles_of(i64 n) { return (n + tile_size<T>() - 1) / tile_size<T>(); }
// In tile `tl` a thread meets its elements in the order k = 0..UNROLL-1, v = 0..VEC-1 (include/lbfgsb_b200_shape.h).
#define B_TILES(T, n, tl) for (i64 tl = 0; tl < batch::ntiles_of<T>(n); ++tl)
#define B_ELEMS(T, n, tl, i)                                                                                         \
    for (int _kv = 0; _kv < Real<T>::UNROLL * Real<T>::VEC; ++_kv)                                                     \
        for (i64 i = (tl) * batch::tile_size<T>() + (i64)(_kv / Real<T>::VEC) * (LBFGSB_BLOCK * Real<T>::VEC) +      \
                     (i64)threadIdx.x * Real<T>::VEC + (_kv % Real<T>::VEC), _o = 1; _o && i < (n); _o = 0)

// block sum of the first kcount accumulators of one tile -> sm.tile[k*MAXTILES + tl]   (the engine's block_sum_store)
template <typename T, int K>
__device__ __forceinline__ void tile_sum(const T (&acc)[K], int kcount, i64 tl, BatchSm<T>& sm) {
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    constexpr int NW = LBFGSB_BLOCK / 32;
#pragma unroll
    for (int k = 0; k < K; ++k) {
        if (k < kcount) {
            T v = warp_sum<T>(acc[k]);
            if (lane == 0) sm.warp[k * NW + w] = v;
        }
    }
    __syncthreads();
    for (int k = threadIdx.x; k < kcount; k += LBFGSB_BLOCK) {
        T s = sm.warp[k * NW];
#pragma unroll
        for (int q = 1; q < NW; ++q) s = s + sm.warp[k * NW + q];
        sm.tile[k * LB_BATCH_MAXTILES + (int)tl] = s;
    }
    __syncthreads();
}
// final stage over the tile partials -> out[k]   (final_sum_warp: lane t adds partial t to zero, then the butterfly)
template <typename T>
__device__ __forceinline__ void final_sums(int kcount, i64 n, BatchSm<T>& sm, T* out) {
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const i64 nt = ntiles_of<T>(n);
    for (int k = w; k < kcount; k += LBFGSB_BLOCK / 32) {
        T acc = (T)0;
        if (lane < nt) acc = acc + sm.tile[k * LB_BATCH_MAXTILES + lane];
        acc = warp_sum<T>(acc);
        if (lane == 0) out[k] = acc;
    }
    __syncthreads();
}
template <typename T> __device__ __forceinline__ i64 bimax(i64 v, BatchSm<T>& sm) {
    v = warp_max<i64>(v);
    if ((threadIdx.x & 31) == 0) sm.smi[threadIdx.x >> 5] = v;
    __syncthreads();
    i64 r = sm.smi[0];
    for (int q = 1; q < LBFGSB_BLOCK / 32; ++q) r = sm.smi[q] > r ? sm.smi[q] : r;
    __syncthreads();
    return r;
}
// column at ring position j (0 = oldest pair) of a history array
template <typename T> __device__ __forceinline__ T* ringcol(T* base, i64 ldw, int m, int head0, int j) {
    int pj = head0 + j; if (pj >= m) pj -= m;
    return base + (i64)pj * ldw;
}

// ---- START: s_start + errclb (:1601-1643) + active (:965-1040) ---------------------------------------------
template <typename T>
__device__ void start(Wk<T>& w, BatchSm<T>& sm, T factr, T pgtol) {
    DevState<T>* s = w.s;
    const i64 n = w.n;
    if (threadIdx.x == 0) {
        const T zero = (T)0;
        s->go = 1; s->pause = 0; s->in_body = 0; s->restart = 0; s->need_walk = 0; s->cauchy_mode = 0;
        s->do_subspace = s->do_formk = s->do_delta = s->do_backtrack = s->do_update = s->do_step = s->do_restore = 0;
        s->z_in_x = 0; s->save_z = 0; s->fuse_uc = 0; s->classify_done = 0; s->lsinit_done = 0; s->ev_n = 0;
        s->spec_step = 0; s->step_done = 0; s->do_unstep = 0; s->lazy_gcp = 0; s->fuse_gf = 0; s->lazy_z = 0;
        s->task = TK_START; s->csave = CS_BLANK; s->info = 0;
        s->col = 0; s->head = 1; s->theta = (T)1; s->iupdat = 0; s->updatd = 0;
        s->iback = 0; s->itail = 0; s->iword = 0; s->nact = 0; s->nleave = 0; s->nenter = 0;
        s->fold = zero; s->dnorm = zero; s->gd = zero; s->stpmx = zero; s->sbgnrm = zero; s->stp = zero;
        s->gdold = zero; s->dtd = zero; s->xstep = zero;
        s->iter = 0; s->nfgv = 0; s->nseg = 0; s->nintol = 0; s->nskip = 0; s->nfree = n; s->ifun = 0;
        s->epsmch = Real<T>::eps();
        s->tol = factr * s->epsmch; s->pgtol = pgtol; s->factr = factr;
        s->brackt = 0; s->stage = 0; s->prjctd = s->cnstnd = s->boxed = 0; s->wrk = 0; s->bnded = 0;
        s->errk = 0; s->nbdd = 0; s->n = n; s->m = w.m;
        s->nbreak = 0; s->nfreec = 0; s->ibkmin = 0; s->ibd = -1; s->n_el = 0; s->tie_events = 0;
        for (int q = 0; q < 13; ++q) s->ls[q] = zero;
        s->f = zero; s->rr = zero; s->dr = zero; s->ddum = zero; s->tsum = zero; s->dtm = zero;
        if (factr < zero) s->task = TK_ERR_FACTR;
    }
    __syncthreads();
    i64 k6 = -1, k7 = -1;   // errclb: last offending index of each kind
    for (i64 i = threadIdx.x; i < n; i += LBFGSB_BLOCK) {
        const int nb = w.nbd[i];
        if (nb < 0 || nb > 3) k6 = i;
        if (nb == 2 && w.l[i] > w.u[i]) k7 = i;
    }
    k6 = bimax<T>(k6, sm); k7 = bimax<T>(k7, sm);
    if (threadIdx.x == 0) {
        if (k6 >= 0 || k7 >= 0) {
            if (k6 > k7) { s->task = TK_ERR_NBD; s->info = -6; s->errk = k6 + 1; }
            else { s->task = TK_ERR_INFEAS; s->info = -7; s->errk = k7 + 1; }
            s->go = 0;
        } else if (s->task >= TK_ERR_N) s->go = 0;
    }
    __syncthreads();
    if (!s->go) return;
    i64 nbdd = 0, prj = 0, cns = 0, nbx = 0;
    for (i64 i = threadIdx.x; i < n; i += LBFGSB_BLOCK) {
        const int nb = w.nbd[i];
        T x = w.x[i];
        const T l = w.l[i], u = w.u[i];
        if (nb > 0) {
            if (nb <= 2 && x <= l) { if (x < l) { prj = 1; x = l; } nbdd++; }
            else if (nb >= 2 && x >= u) { if (x > u) { prj = 1; x = u; } nbdd++; }
        }
        if (nb != 2) nbx = 1;
        int iw;
        if (nb == 0) iw = -1;
        else { cns = 1; iw = (nb == 2 && u - l <= (T)0) ? 3 : 0; }
        w.x[i] = x; w.iwhere[i] = iw; w.state[i] = 3;
    }
    const i64 r0 = block_isum(nbdd, sm.smi), r1 = block_isum(prj, sm.smi), r2 = block_isum(cns, sm.smi), r3 = block_isum(nbx, sm.smi);
    if (threadIdx.x == 0) {
        s->nbdd = r0; s->prjctd = r1 > 0; s->cnstnd = r2 > 0; s->boxed = !(r3 > 0);
        s->task = TK_FG_START; s->go = 0;
    }
    __syncthreads();
}

// ---- projgr (:2594-2622) ------------------------------------------------------------------------------------
template <typename T>
__device__ T projgr(const Wk<T>& w, BatchSm<T>& sm) {
    T acc = (T)0;
    for (i64 i = threadIdx.x; i < w.n; i += LBFGSB_BLOCK)
        acc = dense::tmax(acc, projg_one<T>(w.x[i], w.g[i], w.l[i], w.u[i], w.nbd[i]));
    return block_max<T>(acc, sm.smv);
}

// ---- y/s preparation (:813-824) + matupd's long sums (:2313-2338), as k_update -> red = site_update ------------
template <typename T, int MT>
__device__ void update(Wk<T>& w, BatchSm<T>& sm) {
    DevState<T>* s = w.s;
    const i64 n = w.n;
    const int col = s->col, m = s->m, head0 = s->head - 1, itail0 = s->itail - 1;
    const T stp = s->stp;
    T* wsn = w.ws + (i64)itail0 * w.ldw;
    T* wyn = w.wy + (i64)itail0 * w.ldw;
    B_TILES(T, n, tl) {
        T acc[2 * MT + 1];
#pragma unroll
        for (int k = 0; k < 2 * MT + 1; ++k) acc[k] = (T)0;
        B_ELEMS(T, n, tl, i) {
            const T y = w.g[i] - w.gold[i];
            T sv = w.d[i];
            if (stp != (T)1) sv = stp * sv;
            acc[0] = acc[0] + y * y;
#pragma unroll
            for (int j = 0; j < MT; ++j)
                if (j < col - 1) {
                    acc[1 + j] = acc[1 + j] + sv * ringcol<T>(w.wy, w.ldw, m, head0, j)[i];
                    acc[1 + MT + j] = acc[1 + MT + j] + ringcol<T>(w.ws, w.ldw, m, head0, j)[i] * sv;
                }
            wsn[i] = sv; wyn[i] = y;
        }
        tile_sum<T, 2 * MT + 1>(acc, 2 * MT + 1, tl, sm);
    }
    final_sums<T>(2 * MT + 1, n, sm, sm.red.rv);
}

// ---- cauchy, per-variable pass (:1270-1341), as k_cauchy_classify with d and xcp = x written out -> red = site_cauchy
template <typename T, int MT>
__device__ void classify(Wk<T>& w, BatchSm<T>& sm) {
    DevState<T>* s = w.s;
    const i64 n = w.n;
    const int col = s->col, head0 = s->head - 1, m = s->m;
    CauchyScan<T> cs; cs.init();
    B_TILES(T, n, tl) {
        T acc[2 * MT + 1];
#pragma unroll
        for (int k = 0; k < 2 * MT + 1; ++k) acc[k] = (T)0;
        B_ELEMS(T, n, tl, i) {
            int iw = w.iwhere[i];
            T d = (T)0; bool mv = false;
            const T x = w.x[i];
            T tbp;
            cauchy_classify_one<T>(x, w.l[i], w.u[i], w.g[i], w.nbd[i], iw, d, mv, acc[2 * MT], cs, i, tbp);
            w.iwhere[i] = iw; w.d[i] = d; w.z[i] = x;
            if (mv) {
#pragma unroll
                for (int j = 0; j < MT; ++j)
                    if (j < col) {
                        acc[j] = acc[j] + ringcol<T>(w.wy, w.ldw, m, head0, j)[i] * d;
                        acc[MT + j] = acc[MT + j] + ringcol<T>(w.ws, w.ldw, m, head0, j)[i] * d;
                    }
            }
        }
        tile_sum<T, 2 * MT + 1>(acc, 2 * MT + 1, tl, sm);
    }
    final_sums<T>(2 * MT + 1, n, sm, sm.red.rv);
    block_argmin<T>(cs.bk, cs.ibk, sm.smv, sm.smi);
    const i64 r1 = block_isum(cs.nbr, sm.smi), r2 = block_isum(cs.nfc, sm.smi), r3 = block_isum(cs.bnd ? 0 : 1, sm.smi);
    if (threadIdx.x == 0) {
        sm.red.rv[2 * MT + 1] = cs.bk;
        sm.red.iv[0] = cs.ibk; sm.red.iv[1] = r1; sm.red.iv[2] = r2; sm.red.iv[3] = (r3 > 0) ? 0 : 1;
    }
    __syncthreads();
}

// ---- the breakpoint loop of cauchy (:1378-1526), sequential like the reference ---------------------------------
// all threads: the breakpoints (t_i, i) in variable order, as cauchy's per-variable pass leaves them in t / iorder
// (:1305-1322); thread 0: the loop with hpsolb's heap.
template <typename T>
__device__ void walk(Wk<T>& w, T* bpt, int* bpo, BatchSm<T>& sm) {
    DevState<T>* s = w.s;
    const i64 n = w.n;
    if (threadIdx.x == 0) { sm.bc[0] = 0; sm.bc[1] = -1; }
    __syncthreads();
    for (i64 c0 = 0; c0 < n; c0 += LBFGSB_BLOCK) {
        const i64 i = c0 + threadIdx.x;
        T t = (T)0;
        const bool has = i < n && bp_of<T>(w.d[i], w.x[i], w.l[i], w.u[i], w.nbd[i], t);
        i64 tot;
        const i64 pos = sm.bc[0] + block_excl_scan<i64>(has ? 1 : 0, sm.scan, tot);
        if (has) { bpt[pos] = t; bpo[pos] = (int)i; if (i == s->ibkmin) sm.bc[1] = pos; }
        __syncthreads();
        if (threadIdx.x == 0) sm.bc[0] += tot;
        __syncthreads();
    }
    if (threadIdx.x != 0) return;
    const int col = s->col, col2 = 2 * col, m = s->m, head0 = s->head - 1;
    const T zero = (T)0, two = (T)2, theta = s->theta;
    const i64 nbreak = s->nbreak;
    T* t1 = bpt - 1; int* io1 = bpo - 1;   // 1-based views
    const i64 ibkmin = sm.bc[1] + 1;       // position of the smallest breakpoint in t (1-based)
    i64 nleft = nbreak, iter = 1, nseg = 1;
    T tj = zero, f1 = s->f1, f2 = s->f2, dtm = s->dtm, tsum = zero;
    const T f2_org = s->f2_org;
    T wbp[2 * LB_MMAX], v[2 * LB_MMAX];
    bool all_fixed = false;
    for (;;) {
        const T tj0 = tj;
        i64 ibp;
        if (iter == 1) { tj = s->bkmin; ibp = io1[ibkmin]; }
        else {
            if (iter == 2) {
                if (ibkmin != nbreak) { t1[ibkmin] = t1[nbreak]; io1[ibkmin] = io1[nbreak]; }
                heap_build<T>(t1, io1, nleft);
            }
            T out; int var;
            heap_pop<T>(t1, io1, nleft, out, var);
            tj = out; ibp = var;
        }
        const T dt = tj - tj0;
        if (dtm < dt) break;
        tsum = tsum + dt;
        nleft -= 1; iter += 1;
        const T dibp = w.d[ibp];
        w.d[ibp] = zero;
        T zibp;
        if (dibp > zero) { zibp = w.u[ibp] - w.x[ibp]; w.z[ibp] = w.u[ibp]; w.iwhere[ibp] = 2; }
        else { zibp = w.l[ibp] - w.x[ibp]; w.z[ibp] = w.l[ibp]; w.iwhere[ibp] = 1; }
        if (nleft == 0 && nbreak == n) { dtm = dt; all_fixed = true; break; }   // :1436-1442
        nseg += 1;
        const T dibp2 = dibp * dibp;
        f1 = f1 + dt * f2 + dibp2 - theta * dibp * zibp;
        f2 = f2 - theta * dibp2;
        if (col > 0) {
            dense::daxpy<T>(col2, dt, s->p, s->c);
            for (int j = 0; j < col; ++j) {
                wbp[j] = ringcol<T>(w.wy, w.ldw, m, head0, j)[ibp];
                wbp[col + j] = theta * ringcol<T>(w.ws, w.ldw, m, head0, j)[ibp];
            }
            const int info = dense::bmv<T>(m, s->sy, s->wt, col, wbp, v);
            if (info != 0) {   // :620-635
                ev_push<T>(s, EV_CAUCHY_SINGULAR);
                reset_memory<T>(s);
                s->restart = 1; s->in_body = 0;
                return;
            }
            const T wmc = dense::ddot<T>(col2, s->c, v);
            const T wmp = dense::ddot<T>(col2, s->p, v);
            const T wmw = dense::ddot<T>(col2, wbp, v);
            dense::daxpy<T>(col2, -dibp, wbp, s->p);
            f1 = f1 + dibp * wmc;
            f2 = f2 + two * dibp * wmp - dibp2 * wmw;
        }
        f2 = dense::tmax(s->epsmch * f2_org, f2);
        if (nleft > 0) dtm = -f1 / f2;
        else if (s->bnded) { f1 = zero; f2 = zero; dtm = zero; break; }
        else { dtm = -f1 / f2; break; }
    }
    if (!all_fixed) {
        if (dtm <= zero) dtm = zero;
        tsum = tsum + dtm;
    }
    if (col > 0) dense::daxpy<T>(col2, dtm, s->p, s->c);
    s->f1 = f1; s->f2 = f2; s->dtm = dtm; s->tsum = tsum; s->nseg = nseg;
}

// ---- cauchy's tail xcp += tsum d (:1515) + freev (:1980-2059), as k_gcp_freev -> red.iv = site_freev ------------
template <typename T>
__device__ void gcp_freev(Wk<T>& w, BatchSm<T>& sm) {
    DevState<T>* s = w.s;
    const i64 n = w.n;
    const T tsum = s->tsum;
    const bool axpy = (s->cauchy_mode == 0) && (tsum != (T)0);
    const bool cnt = (s->iter > 0 && s->cnstnd);
    i64 nfr = 0, nen = 0, nle = 0;
    for (i64 i = threadIdx.x; i < n; i += LBFGSB_BLOCK) {
        if (axpy) w.z[i] = w.z[i] + tsum * w.d[i];
        const int fr = w.iwhere[i] <= 0 ? 1 : 0;
        const int old = w.state[i] & 1;
        nfr += fr;
        if (cnt) { nen += (fr && !old); nle += (!fr && old); }
        w.state[i] = (unsigned char)(fr | ((cnt ? old : fr) << 1));
    }
    const i64 r0 = block_isum(nfr, sm.smi), r1 = block_isum(nen, sm.smi), r2 = block_isum(nle, sm.smi);
    if (threadIdx.x == 0) { sm.red.iv[0] = r0; sm.red.iv[1] = r1; sm.red.iv[2] = r2; }
    __syncthreads();
}

// ---- formk, new row / column of WN1 (:1756-1793), as k_formk_gram -> red = site_formk ---------------------------
template <typename T, int MT>
__device__ void formk_gram(Wk<T>& w, BatchSm<T>& sm) {
    DevState<T>* s = w.s;
    const i64 n = w.n;
    const int col = s->col, head0 = s->head - 1, m = s->m;
    const T* wyl = ringcol<T>(w.wy, w.ldw, m, head0, col - 1);
    const T* wsl = ringcol<T>(w.ws, w.ldw, m, head0, col - 1);
    B_TILES(T, n, tl) {
        T acc[4 * MT];
#pragma unroll
        for (int k = 0; k < 4 * MT; ++k) acc[k] = (T)0;
        B_ELEMS(T, n, tl, i) {
            const bool fr = (w.state[i] & 1) != 0;
            const T yl = wyl[i], sl = wsl[i];
#pragma unroll
            for (int j = 0; j < MT; ++j)
                if (j < col) {
                    const T wy = ringcol<T>(w.wy, w.ldw, m, head0, j)[i], wsv = ringcol<T>(w.ws, w.ldw, m, head0, j)[i];
                    if (fr) { acc[j] = acc[j] + yl * wy; acc[3 * MT + j] = acc[3 * MT + j] + wsv * yl; }
                    else { acc[MT + j] = acc[MT + j] + sl * wsv; acc[2 * MT + j] = acc[2 * MT + j] + sl * wy; }
                }
        }
        tile_sum<T, 4 * MT>(acc, 4 * MT, tl, sm);
    }
    final_sums<T>(4 * MT, n, sm, sm.red.rv);
}

// ---- formk, corrections for the variables that entered or left the free set (:1801-1851) -----------------------
// delta[b][i + j*MMAX], b = 0..2 entering (Wy.Wy, Ws.Ws, Ws.Wy), 3..5 leaving; each entry one fixed-shape masked sum.
template <typename T>
__device__ void formk_delta(Wk<T>& w, T* delta, BatchSm<T>& sm) {
    DevState<T>* s = w.s;
    const i64 n = w.n;
    const int col = s->col, head0 = s->head - 1, m = s->m;
    constexpr int KC = 8;   // pairs per sweep
    // pair list: blocks 0, 1 on and below the diagonal, block 2 in full
    const int ntri = col * (col + 1) / 2, npairs = 2 * ntri + col * col;
    for (int p0 = 0; p0 < npairs; p0 += KC) {
        int pb[KC], pi[KC], pj[KC];
#pragma unroll
        for (int q = 0; q < KC; ++q) {
            int p = p0 + q;
            pb[q] = -1; pi[q] = 0; pj[q] = 0;
            if (p < npairs) {
                if (p < 2 * ntri) {
                    pb[q] = p / ntri;
                    int k = p % ntri, i = 0;
                    while (k >= i + 1) { k -= i + 1; ++i; }
                    pi[q] = i; pj[q] = k;
                } else { pb[q] = 2; const int k = p - 2 * ntri; pi[q] = k / col; pj[q] = k % col; }
            }
        }
        B_TILES(T, n, tl) {
            T acc[2 * KC];
#pragma unroll
            for (int k = 0; k < 2 * KC; ++k) acc[k] = (T)0;
            B_ELEMS(T, n, tl, i) {
                const int st = w.state[i];
                if (!el_of(st)) continue;
                const bool ent = (st & 1) != 0;
#pragma unroll
                for (int q = 0; q < KC; ++q) {
                    if (pb[q] < 0) continue;
                    const T a = (pb[q] == 0 ? ringcol<T>(w.wy, w.ldw, m, head0, pi[q]) : ringcol<T>(w.ws, w.ldw, m, head0, pi[q]))[i];
                    const T b = (pb[q] == 1 ? ringcol<T>(w.ws, w.ldw, m, head0, pj[q]) : ringcol<T>(w.wy, w.ldw, m, head0, pj[q]))[i];
                    if (ent) acc[q] = acc[q] + a * b; else acc[KC + q] = acc[KC + q] + a * b;
                }
            }
            tile_sum<T, 2 * KC>(acc, 2 * KC, tl, sm);
        }
        final_sums<T>(2 * KC, n, sm, sm.warp);
        if (threadIdx.x < KC && pb[threadIdx.x] >= 0) {
            const int q = threadIdx.x;
            delta[pb[q] * LB_MMAX * LB_MMAX + pi[q] + pj[q] * LB_MMAX] = sm.warp[q];
            delta[(3 + pb[q]) * LB_MMAX * LB_MMAX + pi[q] + pj[q] * LB_MMAX] = sm.warp[KC + q];
        }
        __syncthreads();
    }
}

// ---- cmprlb (:1565-1583) + wv = W'Zr (:2742-2754), as k_cmprlb_wv -> red = site_wv ------------------------------
template <typename T, int MT>
__device__ void cmprlb_wv(Wk<T>& w, BatchSm<T>& sm) {
    DevState<T>* s = w.s;
    const i64 n = w.n;
    const int col = s->col, head0 = s->head - 1, m = s->m;
    const T theta = s->theta;
    const bool uc = (!s->cnstnd && col > 0);
    if (threadIdx.x < 2 * MT) {
        const int j = threadIdx.x % MT;
        sm.coef[threadIdx.x] = (j < col) ? ((threadIdx.x < MT) ? s->a[j] : theta * s->a[col + j]) : (T)0;
    }
    __syncthreads();
    B_TILES(T, n, tl) {
        T acc[2 * MT];
#pragma unroll
        for (int k = 0; k < 2 * MT; ++k) acc[k] = (T)0;
        B_ELEMS(T, n, tl, i) {
            if (!(w.state[i] & 1)) continue;
            const T g = w.g[i];
            T r = uc ? -g : (-theta * (w.z[i] - w.x[i]) - g);
            if (!uc) {
#pragma unroll
                for (int j = 0; j < MT; ++j)
                    if (j < col) r = r + ringcol<T>(w.wy, w.ldw, m, head0, j)[i] * sm.coef[j] + ringcol<T>(w.ws, w.ldw, m, head0, j)[i] * sm.coef[MT + j];
            }
#pragma unroll
            for (int j = 0; j < MT; ++j)
                if (j < col) {
                    acc[j] = acc[j] + ringcol<T>(w.wy, w.ldw, m, head0, j)[i] * r;
                    acc[MT + j] = acc[MT + j] + ringcol<T>(w.ws, w.ldw, m, head0, j)[i] * r;
                }
            w.r[i] = r;
        }
        tile_sum<T, 2 * MT>(acc, 2 * MT, tl, sm);
    }
    final_sums<T>(2 * MT, n, sm, sm.red.rv);
}

// ---- subsm, second half (:2770-2827), as k_subsm_step -> red = site_subsm ---------------------------------------
template <typename T, int MT>
__device__ void subsm_step(Wk<T>& w, BatchSm<T>& sm) {
    DevState<T>* s = w.s;
    const i64 n = w.n;
    const int col = s->col, head0 = s->head - 1, m = s->m;
    const T theta = s->theta, rtheta = (T)1 / theta;
    if (threadIdx.x < 2 * MT) {
        const int j = threadIdx.x % MT;
        sm.coef[threadIdx.x] = (j < col) ? ((threadIdx.x < MT) ? s->wv[j] : s->wv[col + j]) : (T)0;
    }
    __syncthreads();
    i64 iwd = 0;
    B_TILES(T, n, tl) {
        T acc[1]; acc[0] = (T)0;
        B_ELEMS(T, n, tl, i) {
            T z = w.z[i];
            const T x = w.x[i];
            w.xp[i] = z;   // :2787
            if (w.state[i] & 1) {
                T dk = w.r[i];
#pragma unroll
                for (int j = 0; j < MT; ++j)
                    if (j < col) dk = dk + ringcol<T>(w.wy, w.ldw, m, head0, j)[i] * sm.coef[j] / theta + ringcol<T>(w.ws, w.ldw, m, head0, j)[i] * sm.coef[MT + j];
                dk = rtheta * dk;
                const int nb = w.nbd[i];
                const T l = w.l[i], u = w.u[i];
                T xk = z;
                if (nb != 0) {
                    if (nb == 1) { z = dense::tmax(l, xk + dk); if (z == l) iwd = 1; }
                    else if (nb == 2) { xk = dense::tmax(l, xk + dk); z = dense::tmin(u, xk); if (z == l || z == u) iwd = 1; }
                    else if (nb == 3) { z = dense::tmin(u, xk + dk); if (z == u) iwd = 1; }
                } else z = xk + dk;
                w.r[i] = dk; w.z[i] = z;
            }
            acc[0] = acc[0] + (z - x) * w.g[i];
        }
        tile_sum<T, 1>(acc, 1, tl, sm);
    }
    final_sums<T>(1, n, sm, sm.red.rv);
    const i64 r0 = block_isum(iwd, sm.smi);
    if (threadIdx.x == 0) sm.red.iv[0] = r0;
    __syncthreads();
}

// ---- subsm backtrack (:2830-2879), as k_bt_alpha + s_bt + k_bt_apply ----------------------------------------------
template <typename T>
__device__ void backtrack(Wk<T>& w, BatchSm<T>& sm) {
    DevState<T>* s = w.s;
    const i64 n = w.n;
    T best = LB_INF(T); i64 ib = LB_I64MAX;
    for (i64 i = threadIdx.x; i < n; i += LBFGSB_BLOCK) {
        const int nb = w.nbd[i];
        if ((w.state[i] & 1) && nb != 0) {
            const T dk = w.r[i], xk = w.xp[i];
            T cand = LB_INF(T);
            if (dk < (T)0 && nb <= 2) { const T t2 = w.l[i] - xk; cand = (t2 >= (T)0) ? (T)0 : t2 / dk; }
            else if (dk > (T)0 && nb >= 2) { const T t2 = w.u[i] - xk; cand = (t2 <= (T)0) ? (T)0 : t2 / dk; }
            if (cand < best || (cand == best && i < ib)) { best = cand; ib = i; }
        }
    }
    block_argmin<T>(best, ib, sm.smv, sm.smi);
    if (threadIdx.x == 0) {
        T alpha = (T)1; i64 ibd = -1;
        if (best < alpha) { alpha = best; ibd = ib; }
        s->alpha = alpha; s->ibd = ibd; s->lazy_z = 0;
    }
    __syncthreads();
    const T alpha = s->alpha;
    const i64 ibd = s->ibd;
    for (i64 i = threadIdx.x; i < n; i += LBFGSB_BLOCK) {
        T xk = w.xp[i];
        if (w.state[i] & 1) {
            T dk = w.r[i];
            if (alpha < (T)1 && i == ibd) {
                if (dk > (T)0) { xk = w.u[i]; dk = (T)0; }
                else if (dk < (T)0) { xk = w.l[i]; dk = (T)0; }
            }
            xk = xk + alpha * dk;
        }
        w.z[i] = xk;
    }
    __syncthreads();
}

// ---- d = z - x (:720-722) + first entry of lnsrlb (:2196-2244), as k_ls_init -> red = site_lsinit ----------------
template <typename T>
__device__ void ls_init(Wk<T>& w, BatchSm<T>& sm) {
    DevState<T>* s = w.s;
    const i64 n = w.n;
    const bool bounds = (s->cnstnd && s->iter != 0);
    T smx = LB_INF(T);
    B_TILES(T, n, tl) {
        T acc[2]; acc[0] = (T)0; acc[1] = (T)0;
        B_ELEMS(T, n, tl, i) {
            const T x = w.x[i], g = w.g[i];
            const T d = w.z[i] - x;
            acc[0] = acc[0] + d * d; acc[1] = acc[1] + g * d;
            w.d[i] = d; w.t[i] = x; w.gold[i] = g;
            const int nb = w.nbd[i];
            if (bounds && nb != 0) {
                if (d < (T)0 && nb <= 2) { const T a2 = w.l[i] - x; smx = dense::tmin(smx, (a2 >= (T)0) ? (T)0 : a2 / d); }
                else if (d > (T)0 && nb >= 2) { const T a2 = w.u[i] - x; smx = dense::tmin(smx, (a2 <= (T)0) ? (T)0 : a2 / d); }
            }
        }
        tile_sum<T, 2>(acc, 2, tl, sm);
    }
    final_sums<T>(2, n, sm, sm.red.rv);
    const T rm = block_min<T>(smx, sm.smv);
    if (threadIdx.x == 0) sm.red.rv[2] = rm;
    __syncthreads();
}

// ---- lnsrlb trial point (:2264-2270), restore (:736-738), as k_ls_step / k_restore ------------------------------
template <typename T>
__device__ void ls_step(Wk<T>& w) {
    DevState<T>* s = w.s;
    const i64 n = w.n;
    if (s->do_unstep) { for (i64 i = threadIdx.x; i < n; i += LBFGSB_BLOCK) w.x[i] = w.t[i]; }
    else if (s->do_step && !s->step_done) {
        const T stp = s->stp;
        if (stp == (T)1) { for (i64 i = threadIdx.x; i < n; i += LBFGSB_BLOCK) w.x[i] = w.z[i]; }
        else { for (i64 i = threadIdx.x; i < n; i += LBFGSB_BLOCK) w.x[i] = stp * w.d[i] + w.t[i]; }
    }
    __syncthreads();
}
template <typename T>
__device__ void restore(Wk<T>& w) {
    for (i64 i = threadIdx.x; i < w.n; i += LBFGSB_BLOCK) { w.x[i] = w.t[i]; w.g[i] = w.gold[i]; }
    __syncthreads();
}

// ---- lnsrlb re-entry (:2244) + projgr at the trial point, as k_ls_trial -> red = site_lstrial ---------------------
template <typename T>
__device__ void ls_trial(Wk<T>& w, BatchSm<T>& sm) {
    const i64 n = w.n;
    T pg = (T)0;
    B_TILES(T, n, tl) {
        T acc[1]; acc[0] = (T)0;
        B_ELEMS(T, n, tl, i) {
            const T g = w.g[i];
            acc[0] = acc[0] + g * w.d[i];
            pg = dense::tmax(pg, projg_one<T>(w.x[i], g, w.l[i], w.u[i], w.nbd[i]));
        }
        tile_sum<T, 1>(acc, 1, tl, sm);
    }
    final_sums<T>(1, n, sm, sm.red.rv);
    const T r = block_max<T>(pg, sm.smv);
    if (threadIdx.x == 0) sm.red.rv[1] = r;
    __syncthreads();
}

// staged copies of the small matrices (the w_* functions shift from the originals into the copies)
template <typename T> __device__ void stage3_in(DevState<T>* s, BatchSm<T>& sm) {
    const int mm = s->m * s->m;
    stage_in<T>(sm.sy, s->sy, mm); stage_in<T>(sm.ss, s->ss, mm); stage_in<T>(sm.wt, s->wt, mm);
    __syncthreads();
}
template <typename T> __device__ void stage3_out(DevState<T>* s, BatchSm<T>& sm) {
    const int mm = s->m * s->m;
    __syncthreads();
    stage_out<T>(s->sy, sm.sy, mm); stage_out<T>(s->ss, sm.ss, mm); stage_out<T>(s->wt, sm.wt, mm);
    __syncthreads();
}

// The restart flag, as every thread of the CTA saw it after the step.  Thread 0 clears s->restart next (begin_body):
// each thread takes the flag into a register and the barrier keeps that store behind every thread's read, so no
// warp can see the cleared flag and leave while the others run the restarted iteration without it.
template <typename T> __device__ __forceinline__ bool restart_taken(const DevState<T>* s) {
    const int rs = s->restart;
    __syncthreads();
    return rs != 0;
}

// ---- prelims + first lnsrlb (:601-773): the general pipeline of Engine::enqueue_body inside one CTA --------------
template <typename T, int MT>
__device__ void body(Wk<T>& w, T* bpt, int* bpo, T* delta, BatchSm<T>& sm) {
    DevState<T>* s = w.s;
    const i64 n = w.n;
    for (;;) {
        __syncthreads();
        if (!(s->go && s->in_body)) return;
        // -- cauchy
        if (s->cauchy_mode != 0) {
            for (i64 i = threadIdx.x; i < n; i += LBFGSB_BLOCK) w.z[i] = w.x[i];   // xcp = x (:609, :1247)
            __syncthreads();
        } else {
            classify<T, MT>(w, sm);
            stage3_in<T>(s, sm);
            if (threadIdx.x < 32) w_cauchy<T>(s, sm.red, MT, sm.sy, sm.wt, 0);
            __syncthreads();
            if (s->go && s->in_body && s->need_walk) { walk<T>(w, bpt, bpo, sm); __syncthreads(); }
        }
        // -- cauchy's tail + freev
        if (s->go && s->in_body) {
            const int mode = s->cauchy_mode;
            if (mode != 1) gcp_freev<T>(w, sm);
            if (threadIdx.x < 32) w_freev<T>(s, sm.red, n, false, mode != 1);
            __syncthreads();
        }
        // -- formk
        if (s->go && s->in_body && s->do_subspace) {
            const bool newrow = s->do_formk && s->updatd;
            if (s->do_delta) formk_delta<T>(w, delta, sm);
            if (newrow) formk_gram<T, MT>(w, sm);
            const int m4 = 4 * s->m * s->m;
            stage_in<T>(sm.wn, s->wn, m4); stage_in<T>(sm.wn1, s->wn1, m4);
            __syncthreads();
            if (threadIdx.x < 32) w_formk_dense<T>(s, sm.red, MT, delta, sm.wn, sm.wn1);
            __syncthreads();
            stage_out<T>(s->wn, sm.wn, m4); stage_out<T>(s->wn1, sm.wn1, m4);
            __syncthreads();
        }
        // -- cmprlb + subsm
        if (s->go && s->in_body && s->do_subspace) {
            cmprlb_wv<T, MT>(w, sm);
            if (threadIdx.x < 32) w_subsm_dense<T>(s, sm.red, MT, sm.wn, 0);
            __syncthreads();
        }
        if (s->go && s->in_body && s->do_subspace) {
            subsm_step<T, MT>(w, sm);
            if (threadIdx.x == 0) t0_subsm_post<T>(s, sm.red, 0);
            __syncthreads();
            if (s->do_backtrack) backtrack<T>(w, sm);
        }
        // -- lnsrlb, first entry
        if (s->go && s->in_body) {
            ls_init<T>(w, sm);
            if (threadIdx.x == 0) t0_ls_init<T>(s, sm.red);
            __syncthreads();
        }
        ls_step<T>(w);
        if (!restart_taken(s)) return;
        if (threadIdx.x == 0) { s->go = 1; s->pause = 0; s->classify_done = 0; begin_body<T>(s); }   // s_restart_body
    }
}

}  // namespace batch

// One reverse-communication call for the whole batch.
template <typename T, int MT>
__global__ void __launch_bounds__(LBFGSB_BLOCK) k_batch_setulb(BatchWk<T> bw) {
    extern __shared__ __align__(16) unsigned char bsm_raw[];
    BatchSm<T>& sm = *reinterpret_cast<BatchSm<T>*>(bsm_raw);
    const int p = blockIdx.x;
    if (p >= bw.nprob) return;
    const int entry = bw.entry[p];
    if (entry == BE_IDLE) { if (threadIdx.x == 0) bw.fgmask[p] = 0; return; }
    Wk<T> w;
    w.n = bw.n; w.ldw = bw.ldw; w.off = 0; w.m = bw.m;
    w.ws = bw.ws + (i64)p * bw.m * bw.ldw; w.wy = bw.wy + (i64)p * bw.m * bw.ldw;
    const i64 o = (i64)p * bw.ldw;
    w.z = bw.z + o; w.r = bw.r + o; w.d = bw.d + o; w.t = bw.t + o; w.xp = bw.xp + o; w.gold = bw.gold + o;
    w.iwhere = bw.iwhere + o; w.state = bw.state + o;
    w.part = nullptr; w.ipart = nullptr; w.part2 = nullptr; w.ipart2 = nullptr;
    w.s = bw.s + p;
    const i64 on = (i64)p * bw.n;
    w.x = bw.x + on; w.l = bw.l + on; w.u = bw.u + on; w.nbd = bw.nbd + on; w.g = bw.g + on;
    T* bpt = bw.bpt + o; int* bpo = bw.bpo + o;
    T* delta = bw.delta + (i64)p * 6 * LB_MMAX * LB_MMAX;
    DevState<T>* s = w.s;
    const T f = bw.f[p];

    if (entry == BE_START) {
        batch::start<T>(w, sm, bw.factr, bw.pgtol);
        if (threadIdx.x == 0) bw.fgmask[p] = (s->task == TK_FG_START) ? 1 : 0;
        return;
    }
    if (entry == BE_STOP || entry == BE_STOP_CPU) {
        if (entry == BE_STOP_CPU) {   // :565-571
            batch::restore<T>(w);
            if (threadIdx.x == 0) { s->f = s->fold; bw.f[p] = s->fold; }
        }
        if (threadIdx.x == 0) { s->task = TK_STOP; bw.fgmask[p] = 0; }
        return;
    }
    if (entry == BE_OTHER) { if (threadIdx.x == 0) { s->task = TK_FG_START; bw.fgmask[p] = 1; } return; }

    if (entry == BE_FG_START) {
        if (threadIdx.x == 0) t0_call_begin<T>(s, f);
        const T sbg = batch::projgr<T>(w, sm);
        if (threadIdx.x == 0) {
            s->nfgv = 1; s->sbgnrm = sbg;
            if (s->sbgnrm <= s->pgtol) { s->task = TK_CONV_PG; s->go = 0; }
            else begin_body<T>(s);
        }
        batch::body<T, MT>(w, bpt, bpo, delta, sm);
    } else if (entry == BE_FG_LNSRCH) {
        batch::ls_trial<T>(w, sm);
        if (threadIdx.x == 0) { t0_call_begin<T>(s, f); t0_ls_trial<T>(s, sm.red); }
        __syncthreads();
        if (s->do_restore) batch::restore<T>(w);
        batch::ls_step<T>(w);
        if (batch::restart_taken(s)) {
            if (threadIdx.x == 0) { s->go = 1; s->pause = 0; s->classify_done = 0; begin_body<T>(s); }
            batch::body<T, MT>(w, bpt, bpo, delta, sm);
        }
    } else {   // BE_NEW_X
        if (threadIdx.x == 0) { t0_call_begin<T>(s, f); t0_newx_tests<T>(s, 0); }
        __syncthreads();
        if (s->go) {
            const bool upd = s->do_update != 0;
            if (upd) {
                batch::update<T, MT>(w, sm);
                batch::stage3_in<T>(s, sm);
                if (threadIdx.x < 32) w_update_dense<T>(s, sm.red, MT, sm.sy, sm.ss, sm.wt);
                batch::stage3_out<T>(s, sm);
            }
            if (threadIdx.x == 0) begin_body<T>(s);
            batch::body<T, MT>(w, bpt, bpo, delta, sm);
        }
    }
    __syncthreads();
    if (threadIdx.x == 0) { bw.f[p] = s->f; bw.fgmask[p] = (s->task == TK_FG_START || s->task == TK_FG_LNSRCH) ? 1 : 0; }
}
