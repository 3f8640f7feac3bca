// ORACLE -- TEST INFRASTRUCTURE ONLY.  Not part of the shipped product.
//
// A CPU restatement, in plain C++ (double / float template), of the reference
// L-BFGS-B 3.0 hot path: everything below `setulb` in
//   /root/reference/src/lbfgsb.f90               (setulb, mainlb and all L1 kernels)
//   /root/reference/src/lbfgsb_blas_module.F90   (daxpy, dcopy, ddot, dscal)
//   /root/reference/src/lbfgsb_linpack_module.f90 (dpofa, dtrsl)
// Each function cites the reference file:line it follows.  It keeps the
// reference's 1-based loop structure, column-major ws/wy, the strict
// left-to-right single-accumulator summation of `ddot`
// (lbfgsb_blas_module.F90:187-202), `hpsolb` verbatim, and all state in the
// caller's arrays (wa, iwa, task, csave, lsave, isave, dsave).  Offsets into
// `wa` are 64-bit (the reference's default-integer offsets overflow at
// n*(2m+5) >= 2^31; see SURVEY.md section 5).
//
// Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline /
// `--impl reference` arms may load this library.  The product (lbfgsb_b200/)
// never does.
//
// Parity pin: this file is checked against the reference's own golden outputs
// test/OUTPUTS/output_90_{1,2,3} and test/OUTPUTS/iterate.dat by
// tests/test_oracle_golden.py.  The reference itself cannot be compiled in this
// image (no Fortran compiler), so oracle/_ref does not exist.
//
// A second summation mode ("device order") replays every O(n) reduction in the
// fixed block/warp/tree shape the CUDA kernels use (include/lbfgsb_b200_shape.h)
// so that the GPU can be gated tightly against a CPU run that differs from it
// only by what differs from the reference: the order of the long sums.
//
// Build: see oracle/Makefile  (g++ -O2 -ffp-contract=off, no -ffast-math).

#include <algorithm>
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <ctime>
#include <limits>
#include <vector>

#include "../include/lbfgsb_b200_shape.h"

namespace {

typedef int64_t i64;

// ---------------------------------------------------------------------------
// Summation mode.  0 = reference order (default), 1 = device order.
// ---------------------------------------------------------------------------
static int g_sum_mode = 0;
// 0: hpsolb's heap decides the order of equal breakpoints (the reference); 1: equal breakpoints are taken in
// variable order (what a stable sort gives -- the CUDA engine's order when its heap replay is switched off)
static int g_tie_mode = 0;
// path counters for the tests (how often the rare branches ran): 0 subsm backtrack (:2830), 1 ascent direction (:2247),
// 2 memory resets ("refresh the lbfgs memory"), 3 skipped updates (:826)
static long long g_events[8] = {0, 0, 0, 0, 0, 0, 0, 0};

// Replays the CUDA reduction shape of include/lbfgsb_b200_shape.h on the CPU:
// LBFGSB_GRID blocks of LBFGSB_BLOCK threads walk tiles b, b+G, b+2G, ...; in a
// tile thread t owns VEC consecutive elements at t*VEC + k*(BLOCK*VEC) for
// k = 0..UNROLL-1 and adds them serially; lanes combine by xor-butterfly
// (16,8,4,2,1), warps serially in warp order, blocks by the same shape of
// LBFGSB_FINAL_BLOCK threads striding over the block partials.
template <typename T, typename F>
static T device_order_sum(i64 n, F term) {
    const int VEC = LBFGSB_VEC((int)sizeof(T)), UNROLL = LBFGSB_UNROLL((int)sizeof(T));
    const i64 tile = (i64)LBFGSB_BLOCK * VEC * UNROLL;
    const i64 ntiles = (n + tile - 1) / tile;
    std::vector<T> block_partial(LBFGSB_GRID, (T)0);
    // The accumulators of all GRID x BLOCK threads are kept side by side and the elements are visited in MEMORY order:
    // a given thread still meets its own elements in the order tile, k, v -- the order of the kernels -- so every
    // accumulator receives the same additions in the same order as in a thread-by-thread replay, at a fraction of the
    // cache misses (n = 1e8: seconds instead of minutes per sum).
    const i64 nblk = ntiles < (i64)LBFGSB_GRID ? ntiles : (i64)LBFGSB_GRID;
    std::vector<T> acc((size_t)nblk * LBFGSB_BLOCK, (T)0);
    for (i64 tl = 0; tl < ntiles; ++tl) {
        T* a = acc.data() + (size_t)(tl % LBFGSB_GRID) * LBFGSB_BLOCK;
        for (int k = 0; k < UNROLL; ++k) {
            const i64 base0 = tl * tile + (i64)k * (LBFGSB_BLOCK * VEC);
            if (base0 >= n) break;
            for (int t = 0; t < LBFGSB_BLOCK; ++t) {
                const i64 base = base0 + (i64)t * VEC;
                for (int v = 0; v < VEC; ++v) {
                    const i64 i = base + v;
                    if (i < n) a[t] = a[t] + term(i);
                }
            }
        }
    }
    for (int b = 0; b < LBFGSB_GRID; ++b) {
        if ((i64)b >= ntiles) { block_partial[b] = (T)0; continue; }
        const T* lane = acc.data() + (size_t)b * LBFGSB_BLOCK;
        // warp butterflies
        T warp_sum[LBFGSB_BLOCK / 32];
        for (int w = 0; w < LBFGSB_BLOCK / 32; ++w) {
            T v[32];
            for (int q = 0; q < 32; ++q) v[q] = lane[w * 32 + q];
            for (int off = 16; off >= 1; off >>= 1) {
                T nv[32];
                for (int q = 0; q < 32; ++q) nv[q] = v[q] + v[q ^ off];
                for (int q = 0; q < 32; ++q) v[q] = nv[q];
            }
            warp_sum[w] = v[0];
        }
        T s = warp_sum[0];
        for (int w = 1; w < LBFGSB_BLOCK / 32; ++w) s = s + warp_sum[w];
        block_partial[b] = s;
    }
    // final stage: LBFGSB_FINAL_BLOCK threads stride over the block partials
    T fl[LBFGSB_FINAL_BLOCK];
    for (int t = 0; t < LBFGSB_FINAL_BLOCK; ++t) {
        T acc = (T)0;
        for (int b = t; b < LBFGSB_GRID; b += LBFGSB_FINAL_BLOCK) acc = acc + block_partial[b];
        fl[t] = acc;
    }
    T ws[LBFGSB_FINAL_BLOCK / 32];
    for (int w = 0; w < LBFGSB_FINAL_BLOCK / 32; ++w) {
        T v[32];
        for (int q = 0; q < 32; ++q) v[q] = fl[w * 32 + q];
        for (int off = 16; off >= 1; off >>= 1) {
            T nv[32];
            for (int q = 0; q < 32; ++q) nv[q] = v[q] + v[q ^ off];
            for (int q = 0; q < 32; ++q) v[q] = nv[q];
        }
        ws[w] = v[0];
    }
    T s = ws[0];
    for (int w = 1; w < LBFGSB_FINAL_BLOCK / 32; ++w) s = s + ws[w];
    return s;
}

// ---------------------------------------------------------------------------
// Fortran character(len=60) helpers (blank padded, compared like Fortran '==').
// ---------------------------------------------------------------------------
static void set_str(char* s60, const char* lit) {
    size_t k = std::strlen(lit);
    if (k > 60) k = 60;
    std::memcpy(s60, lit, k);
    for (size_t i = k; i < 60; ++i) s60[i] = ' ';
}
static bool str_eq(const char* s60, const char* lit) {  // task == 'LIT'
    size_t k = std::strlen(lit);
    if (k > 60) return false;
    if (std::memcmp(s60, lit, k) != 0) return false;
    for (size_t i = k; i < 60; ++i)
        if (s60[i] != ' ') return false;
    return true;
}
static bool str_pre(const char* s60, const char* lit) {  // task(1:len) == 'LIT'
    return std::memcmp(s60, lit, std::strlen(lit)) == 0;
}

static double cpu_time_now() {
    struct timespec ts;
    clock_gettime(CLOCK_PROCESS_CPUTIME_ID, &ts);
    return (double)ts.tv_sec + 1e-9 * (double)ts.tv_nsec;
}

template <typename T>
struct LB {
    // =======================================================================
    // BLAS-1 shims -- lbfgsb_blas_module.F90
    // =======================================================================
    // daxpy :37-88 (early-outs :49-50; element-wise, so unrolling is immaterial)
    static void daxpy(i64 n, T da, const T* dx, T* dy) {
        if (n <= 0) return;
        if (da == (T)0) return;
        for (i64 i = 0; i < n; ++i) dy[i] = dy[i] + da * dx[i];
    }
    // dcopy :100-153
    static void dcopy(i64 n, const T* dx, T* dy) {
        if (n <= 0) return;
        for (i64 i = 0; i < n; ++i) dy[i] = dx[i];
    }
    // ddot :165-221.  One accumulator; the 5-way unrolled statement
    //   dtemp = dtemp + a1 + a2 + a3 + a4 + a5   (:198-201)
    // associates left to right, i.e. it is the plain serial sum.
    static T ddot(i64 n, const T* dx, const T* dy) {
        T dtemp = (T)0;
        if (n <= 0) return dtemp;
        if (g_sum_mode == 1 && n > 64) {
            return device_order_sum<T>(n, [&](i64 i) { return dx[i] * dy[i]; });
        }
        i64 mm = n % 5;
        for (i64 i = 0; i < mm; ++i) dtemp = dtemp + dx[i] * dy[i];
        if (n < 5) return dtemp;
        for (i64 i = mm; i < n; i += 5) {
            dtemp = dtemp + dx[i] * dy[i] + dx[i + 1] * dy[i + 1] + dx[i + 2] * dy[i + 2] +
                    dx[i + 3] * dy[i + 3] + dx[i + 4] * dy[i + 4];
        }
        return dtemp;
    }
    // dscal :233-277
    static void dscal(i64 n, T da, T* dx) {
        if (n <= 0) return;
        for (i64 i = 0; i < n; ++i) dx[i] = da * dx[i];
    }

    // =======================================================================
    // LINPACK shims -- lbfgsb_linpack_module.f90
    // =======================================================================
    // dpofa :30-67.  a is column-major with leading dimension lda, 1-based.
    static void dpofa(T* a0, int lda, int n, int& info) {
#define A_(i, j) a0[((i)-1) + (i64)((j)-1) * lda]
        for (int j = 1; j <= n; ++j) {
            info = j;
            T s = (T)0;
            int jm1 = j - 1;
            if (jm1 >= 1) {
                for (int k = 1; k <= jm1; ++k) {
                    T t = A_(k, j) - ddot(k - 1, &A_(1, k), &A_(1, j));
                    t = t / A_(k, k);
                    A_(k, j) = t;
                    s = s + t * t;
                }
            }
            s = A_(j, j) - s;
            if (s <= (T)0) return;
            A_(j, j) = std::sqrt(s);
        }
        info = 0;
#undef A_
    }
    // dtrsl :87-165.  job 00/01/10/11.
    static void dtrsl(const T* t0, int ldt, int n, T* b0, int job, int& info) {
#define T_(i, j) t0[((i)-1) + (i64)((j)-1) * ldt]
        T* b = b0 - 1;
        for (info = 1; info <= n; ++info)
            if (T_(info, info) == (T)0) return;
        info = 0;
        int kase = 1;
        if (job % 10 != 0) kase = 2;
        if ((job % 100) / 10 != 0) kase = kase + 2;
        switch (kase) {
            case 1:  // t*x=b, t lower
                b[1] = b[1] / T_(1, 1);
                for (int j = 2; j <= n; ++j) {
                    T temp = -b[j - 1];
                    daxpy(n - j + 1, temp, &T_(j, j - 1), &b[j]);
                    b[j] = b[j] / T_(j, j);
                }
                break;
            case 2:  // t*x=b, t upper
                b[n] = b[n] / T_(n, n);
                for (int jj = 2; jj <= n; ++jj) {
                    int j = n - jj + 1;
                    T temp = -b[j + 1];
                    daxpy(j, temp, &T_(1, j + 1), &b[1]);
                    b[j] = b[j] / T_(j, j);
                }
                break;
            case 3:  // trans(t)*x=b, t lower
                b[n] = b[n] / T_(n, n);
                for (int jj = 2; jj <= n; ++jj) {
                    int j = n - jj + 1;
                    b[j] = b[j] - ddot(jj - 1, &T_(j + 1, j), &b[j + 1]);
                    b[j] = b[j] / T_(j, j);
                }
                break;
            case 4:  // trans(t)*x=b, t upper
                b[1] = b[1] / T_(1, 1);
                for (int j = 2; j <= n; ++j) {
                    b[j] = b[j] - ddot(j - 1, &T_(1, j), &b[1]);
                    b[j] = b[j] / T_(j, j);
                }
                break;
        }
#undef T_
    }

    // =======================================================================
    // lbfgsb.f90 L1 kernels.  All arrays arrive 0-based; local 1-based views
    // are made with the macros below.
    // =======================================================================

    // active :965-1040
    static void active(i64 n, const T* l0, const T* u0, const int* nbd0, T* x0, int* iwhere0,
                       bool& prjctd, bool& cnstnd, bool& boxed, i64& nbdd) {
        const T *l = l0 - 1, *u = u0 - 1;
        const int* nbd = nbd0 - 1;
        T* x = x0 - 1;
        int* iwhere = iwhere0 - 1;
        nbdd = 0;
        prjctd = false;
        cnstnd = false;
        boxed = true;
        for (i64 i = 1; i <= n; ++i) {
            if (nbd[i] > 0) {
                if (nbd[i] <= 2 && x[i] <= l[i]) {
                    if (x[i] < l[i]) {
                        prjctd = true;
                        x[i] = l[i];
                    }
                    nbdd = nbdd + 1;
                } else if (nbd[i] >= 2 && x[i] >= u[i]) {
                    if (x[i] > u[i]) {
                        prjctd = true;
                        x[i] = u[i];
                    }
                    nbdd = nbdd + 1;
                }
            }
        }
        for (i64 i = 1; i <= n; ++i) {
            if (nbd[i] != 2) boxed = false;
            if (nbd[i] == 0) {
                iwhere[i] = -1;
            } else {
                cnstnd = true;
                if (nbd[i] == 2 && u[i] - l[i] <= (T)0) {
                    iwhere[i] = 3;
                } else {
                    iwhere[i] = 0;
                }
            }
        }
    }

    // bmv :1057-1123
    static void bmv(int m, const T* sy0, const T* wt0, int col, const T* v0, T* p0, int& info) {
#define SY(i, j) sy0[((i)-1) + (i64)((j)-1) * m]
        const T* v = v0 - 1;
        T* p = p0 - 1;
        info = 0;
        if (col == 0) return;
        p[col + 1] = v[col + 1];
        for (int i = 2; i <= col; ++i) {
            int i2 = col + i;
            T sum = (T)0;
            for (int k = 1; k <= i - 1; ++k) sum = sum + SY(i, k) * v[k] / SY(k, k);
            p[i2] = v[i2] + sum;
        }
        dtrsl(wt0, m, col, &p[col + 1], 11, info);
        if (info != 0) return;
        for (int i = 1; i <= col; ++i) p[i] = v[i] / std::sqrt(SY(i, i));
        dtrsl(wt0, m, col, &p[col + 1], 1, info);
        if (info != 0) return;
        for (int i = 1; i <= col; ++i) p[i] = -p[i] / std::sqrt(SY(i, i));
        for (int i = 1; i <= col; ++i) {
            T sum = (T)0;
            for (int k = i + 1; k <= col; ++k) sum = sum + SY(k, i) * p[col + k] / SY(i, i);
            p[i] = p[i] + sum;
        }
#undef SY
    }

    // hpsolb :2079-2157 (verbatim heap; tie order is part of the behaviour)
    static void hpsolb(i64 n, T* t0, int* iorder0, i64 iheap) {
        T* t = t0 - 1;
        int* iorder = iorder0 - 1;
        if (iheap == 0) {
            for (i64 k = 2; k <= n; ++k) {
                T ddum = t[k];
                int indxin = iorder[k];
                i64 i = k;
                for (;;) {
                    if (i > 1) {
                        i64 j = i / 2;
                        if (ddum < t[j]) {
                            t[i] = t[j];
                            iorder[i] = iorder[j];
                            i = j;
                            continue;
                        }
                    }
                    break;
                }
                t[i] = ddum;
                iorder[i] = indxin;
            }
        }
        if (n > 1) {
            i64 i = 1;
            T out = t[1];
            int indxou = iorder[1];
            T ddum = t[n];
            int indxin = iorder[n];
            for (;;) {
                i64 j = i + i;
                if (j <= n - 1) {
                    if (t[j + 1] < t[j]) j = j + 1;
                    if (t[j] < ddum) {
                        t[i] = t[j];
                        iorder[i] = iorder[j];
                        i = j;
                        continue;
                    }
                }
                break;
            }
            t[i] = ddum;
            iorder[i] = indxin;
            t[n] = out;
            iorder[n] = indxou;
        }
    }

    // cauchy :1157-1532
    static void cauchy(i64 n, const T* x0, const T* l0, const T* u0, const int* nbd0, const T* g0,
                       int* iorder0, int* iwhere0, T* t0, T* d0, T* xcp0, int m, const T* wy0,
                       const T* ws0, const T* sy0, const T* wt0, T theta, int col, int head, T* p0,
                       T* c0, T* wbp0, T* v0, i64& nseg, T sbgnrm, int& info, T epsmch) {
        const T *x = x0 - 1, *l = l0 - 1, *u = u0 - 1, *g = g0 - 1;
        const int* nbd = nbd0 - 1;
        int *iorder = iorder0 - 1, *iwhere = iwhere0 - 1;
        T *t = t0 - 1, *d = d0 - 1, *xcp = xcp0 - 1, *p = p0 - 1, *c = c0 - 1, *wbp = wbp0 - 1,
          *v = v0 - 1;
#define WY(i, j) wy0[((i)-1) + (i64)((j)-1) * n]
#define WS(i, j) ws0[((i)-1) + (i64)((j)-1) * n]
        const T zero = (T)0, one = (T)1, two = (T)2;
        bool xlower, xupper, bnded;
        i64 i, nfree, nbreak, ibp = 0, nleft, ibkmin, iter;
        int j, col2, pointr;
        T f1, f2, dt, dtm, tsum, dibp, zibp, dibp2, bkmin, tu = zero, tl = zero, wmc, wmp, wmw,
                                                               tj, tj0, neggi, f2_org;

        if (sbgnrm <= zero) {  // :1245-1249
            dcopy(n, x0, xcp0);
            return;
        }
        bnded = true;
        nfree = n + 1;
        nbreak = 0;
        ibkmin = 0;
        bkmin = zero;
        col2 = 2 * col;
        f1 = zero;
        for (j = 1; j <= col2; ++j) p[j] = zero;

        // :1270-1330.  In device-order mode the p and f1 sums are formed after the
        // loop in the device's reduction shape; the classification is unchanged.
        for (i = 1; i <= n; ++i) {
            neggi = -g[i];
            if (iwhere[i] != 3 && iwhere[i] != -1) {
                if (nbd[i] <= 2) tl = x[i] - l[i];
                if (nbd[i] >= 2) tu = u[i] - x[i];
                xlower = nbd[i] <= 2 && tl <= zero;
                xupper = nbd[i] >= 2 && tu <= zero;
                iwhere[i] = 0;
                if (xlower) {
                    if (neggi <= zero) iwhere[i] = 1;
                } else if (xupper) {
                    if (neggi >= zero) iwhere[i] = 2;
                } else {
                    if (std::fabs(neggi) <= zero) iwhere[i] = -3;
                }
            }
            pointr = head;
            if (iwhere[i] != 0 && iwhere[i] != -1) {
                d[i] = zero;
            } else {
                d[i] = neggi;
                if (g_sum_mode == 0) {
                    f1 = f1 - neggi * neggi;
                    for (j = 1; j <= col; ++j) {
                        p[j] = p[j] + WY(i, pointr) * neggi;
                        p[col + j] = p[col + j] + WS(i, pointr) * neggi;
                        pointr = pointr % m + 1;
                    }
                }
                if (nbd[i] <= 2 && nbd[i] != 0 && neggi < zero) {
                    nbreak = nbreak + 1;
                    iorder[nbreak] = (int)i;
                    t[nbreak] = tl / (-neggi);
                    if (nbreak == 1 || t[nbreak] < bkmin) {
                        bkmin = t[nbreak];
                        ibkmin = nbreak;
                    }
                } else if (nbd[i] >= 2 && neggi > zero) {
                    nbreak = nbreak + 1;
                    iorder[nbreak] = (int)i;
                    t[nbreak] = tu / neggi;
                    if (nbreak == 1 || t[nbreak] < bkmin) {
                        bkmin = t[nbreak];
                        ibkmin = nbreak;
                    }
                } else {
                    nfree = nfree - 1;
                    iorder[nfree] = (int)i;
                    if (std::fabs(neggi) > zero) bnded = false;
                }
            }
        }
        if (g_sum_mode == 1) {
            // d(i) is exactly neggi for moving variables and 0 otherwise.
            f1 = -device_order_sum<T>(n, [&](i64 q) { return d0[q] * d0[q]; });
            pointr = head;
            for (j = 1; j <= col; ++j) {
                const T* wyc = &WY(1, pointr);
                const T* wsc = &WS(1, pointr);
                p[j] = device_order_sum<T>(n, [&](i64 q) { return wyc[q] * d0[q]; });
                p[col + j] = device_order_sum<T>(n, [&](i64 q) { return wsc[q] * d0[q]; });
                pointr = pointr % m + 1;
            }
        }

        if (theta != one) dscal(col, theta, &p[col + 1]);  // :1337
        dcopy(n, x0, xcp0);                                // :1341
        if (nbreak == 0 && nfree == n + 1) return;          // :1343-1347
        for (j = 1; j <= col2; ++j) c[j] = zero;

        f2 = -theta * f1;
        f2_org = f2;
        if (col > 0) {
            bmv(m, sy0, wt0, col, p0, v0, info);
            if (info != 0) return;
            f2 = f2 - ddot(col2, v0, p0);
        }
        dtm = -f1 / f2;
        tsum = zero;
        nseg = 1;

        bool skip_tail = false;
        if (nbreak != 0) {
            nleft = nbreak;
            iter = 1;
            tj = zero;
            for (;;) {  // :1378-1497
                tj0 = tj;
                if (iter == 1) {
                    tj = bkmin;
                    ibp = iorder[ibkmin];
                } else {
                    if (iter == 2) {
                        if (ibkmin != nbreak) {
                            t[ibkmin] = t[nbreak];
                            iorder[ibkmin] = iorder[nbreak];
                        }
                    }
                    if (g_tie_mode == 1) {
                        if (iter == 2) {   // descending (t, variable): reading from the end pops ascending
                            std::vector<std::pair<T, int>> bp((size_t)nleft);
                            for (i64 q = 1; q <= nleft; ++q) bp[(size_t)q - 1] = {t[q], iorder[q]};
                            std::sort(bp.begin(), bp.end(), [](const std::pair<T, int>& a, const std::pair<T, int>& b) {
                                return a.first > b.first || (a.first == b.first && a.second > b.second);
                            });
                            for (i64 q = 1; q <= nleft; ++q) { t[q] = bp[(size_t)q - 1].first; iorder[q] = bp[(size_t)q - 1].second; }
                        }
                    } else {
                        hpsolb(nleft, t0, iorder0, iter - 2);
                    }
                    tj = t[nleft];
                    ibp = iorder[nleft];
                }
                dt = tj - tj0;
                if (dtm < dt) break;  // :1416

                tsum = tsum + dt;
                nleft = nleft - 1;
                iter = iter + 1;
                dibp = d[ibp];
                d[ibp] = zero;
                if (dibp > zero) {
                    zibp = u[ibp] - x[ibp];
                    xcp[ibp] = u[ibp];
                    iwhere[ibp] = 2;
                } else {
                    zibp = l[ibp] - x[ibp];
                    xcp[ibp] = l[ibp];
                    iwhere[ibp] = 1;
                }
                if (nleft == 0 && nbreak == n) {  // :1436-1442
                    dtm = dt;
                    if (col > 0) daxpy(col2, dtm, p0, c0);
                    skip_tail = true;
                    break;
                }
                nseg = nseg + 1;
                dibp2 = dibp * dibp;
                f1 = f1 + dt * f2 + dibp2 - theta * dibp * zibp;
                f2 = f2 - theta * dibp2;
                if (col > 0) {
                    daxpy(col2, dt, p0, c0);
                    pointr = head;
                    for (j = 1; j <= col; ++j) {
                        wbp[j] = WY(ibp, pointr);
                        wbp[col + j] = theta * WS(ibp, pointr);
                        pointr = pointr % m + 1;
                    }
                    bmv(m, sy0, wt0, col, wbp0, v0, info);
                    if (info != 0) return;
                    wmc = ddot(col2, c0, v0);
                    wmp = ddot(col2, p0, v0);
                    wmw = ddot(col2, wbp0, v0);
                    daxpy(col2, -dibp, wbp0, p0);
                    f1 = f1 + dibp * wmc;
                    f2 = f2 + two * dibp * wmp - dibp2 * wmw;
                }
                f2 = std::max(epsmch * f2_org, f2);
                if (nleft > 0) {
                    dtm = -f1 / f2;
                } else if (bnded) {
                    f1 = zero;
                    f2 = zero;
                    dtm = zero;
                    break;
                } else {
                    dtm = -f1 / f2;
                    break;
                }
            }
        }
        if (skip_tail) return;
        if (dtm <= zero) dtm = zero;  // :1509
        tsum = tsum + dtm;
        daxpy(n, tsum, d0, xcp0);                    // :1515
        if (col > 0) daxpy(col2, dtm, p0, c0);      // :1526
        (void)v;
#undef WY
#undef WS
    }

    // cmprlb :1548-1586
    static void cmprlb(i64 n, int m, const T* x0, const T* g0, const T* ws0, const T* wy0,
                       const T* sy0, const T* wt0, const T* z0, T* r0, T* wa0, const int* index0,
                       T theta, int col, int head, i64 nfree, bool cnstnd, int& info) {
        const T *x = x0 - 1, *g = g0 - 1, *z = z0 - 1;
        T *r = r0 - 1, *wa = wa0 - 1;
        const int* index = index0 - 1;
#define WY(i, j) wy0[((i)-1) + (i64)((j)-1) * n]
#define WS(i, j) ws0[((i)-1) + (i64)((j)-1) * n]
        if (!cnstnd && col > 0) {
            for (i64 i = 1; i <= n; ++i) r[i] = -g[i];
        } else {
            for (i64 i = 1; i <= nfree; ++i) {
                i64 k = index[i];
                r[i] = -theta * (z[k] - x[k]) - g[k];
            }
            bmv(m, sy0, wt0, col, &wa[2 * m + 1], &wa[1], info);
            if (info != 0) {
                info = -8;
                return;
            }
            int pointr = head;
            for (int j = 1; j <= col; ++j) {
                T a1 = wa[j];
                T a2 = theta * wa[col + j];
                for (i64 i = 1; i <= nfree; ++i) {
                    i64 k = index[i];
                    r[i] = r[i] + WY(k, pointr) * a1 + WS(k, pointr) * a2;
                }
                pointr = pointr % m + 1;
            }
        }
#undef WY
#undef WS
    }

    // errclb :1601-1643
    static void errclb(i64 n, int m, T factr, const T* l0, const T* u0, const int* nbd0,
                       char* task, int& info, i64& k) {
        const T *l = l0 - 1, *u = u0 - 1;
        const int* nbd = nbd0 - 1;
        if (n <= 0) set_str(task, "ERROR: N <= 0");
        if (m <= 0) set_str(task, "ERROR: M <= 0");
        if (factr < (T)0) set_str(task, "ERROR: FACTR < 0");
        k = 0;
        for (i64 i = 1; i <= n; ++i) {
            if (nbd[i] < 0 || nbd[i] > 3) {
                set_str(task, "ERROR: INVALID NBD");
                info = -6;
                k = i;
            }
            if (nbd[i] == 2) {
                if (l[i] > u[i]) {
                    set_str(task, "ERROR: NO FEASIBLE SOLUTION");
                    info = -7;
                    k = i;
                }
            }
        }
    }

    // Gathered product sum over an index list, in list order (reference) or in
    // device order over the whole variable range with a membership mask.
    // member[k-1] != 0 marks the variables of the list (device mode only).
    template <typename F>
    static T list_sum(i64 n, const int* list1, i64 kbeg, i64 kend, F prod,
                      const unsigned char* member) {
        if (g_sum_mode == 1) {
            return device_order_sum<T>(n, [&](i64 q) { return member[q] ? prod(q + 1) : (T)0; });
        }
        T s = (T)0;
        for (i64 k = kbeg; k <= kend; ++k) {
            i64 k1 = list1[k];
            s = s + prod(k1);
        }
        return s;
    }

    // formk :1681-1908
    static void formk(i64 n, i64 nsub, const int* ind0, i64 nenter, i64 ileave, const int* indx20,
                      int iupdat, bool updatd, T* wn0, T* wn10, int m, const T* ws0, const T* wy0,
                      const T* sy0, T theta, int col, int head, int& info) {
        const int *ind = ind0 - 1, *indx2 = indx20 - 1;
        const int m2 = 2 * m;
#define WN(i, j) wn0[((i)-1) + (i64)((j)-1) * m2]
#define WN1(i, j) wn10[((i)-1) + (i64)((j)-1) * m2]
#define SY(i, j) sy0[((i)-1) + (i64)((j)-1) * m]
#define WY(i, j) wy0[((i)-1) + (i64)((j)-1) * n]
#define WS(i, j) ws0[((i)-1) + (i64)((j)-1) * n]
        const T zero = (T)0;
        int ipntr, jpntr, iy, is, jy, js, is1, js1, col2, upcl;
        i64 pbegin, pend, dbegin, dend;
        T temp1, temp2, temp3, temp4;

        // membership masks for device-order sums
        std::vector<unsigned char> mfree, mact, ment, mlea;
        if (g_sum_mode == 1) {
            mfree.assign(n, 0);
            mact.assign(n, 0);
            ment.assign(n, 0);
            mlea.assign(n, 0);
            for (i64 k = 1; k <= nsub; ++k) mfree[ind[k] - 1] = 1;
            for (i64 k = nsub + 1; k <= n; ++k) mact[ind[k] - 1] = 1;
            for (i64 k = 1; k <= nenter; ++k) ment[indx2[k] - 1] = 1;
            for (i64 k = ileave; k <= n; ++k) mlea[indx2[k] - 1] = 1;
        }
        const unsigned char *pf = mfree.data(), *pa = mact.data(), *pe = ment.data(),
                            *pl = mlea.data();

        if (updatd) {
            if (iupdat > m) {  // :1736-1744 shift old part of WN1
                for (jy = 1; jy <= m - 1; ++jy) {
                    js = m + jy;
                    dcopy(m - jy, &WN1(jy + 1, jy + 1), &WN1(jy, jy));
                    dcopy(m - jy, &WN1(js + 1, js + 1), &WN1(js, js));
                    dcopy(m - 1, &WN1(m + 2, jy + 1), &WN1(m + 1, jy));
                }
            }
            pbegin = 1;
            pend = nsub;
            dbegin = nsub + 1;
            dend = n;
            iy = col;
            is = m + col;
            ipntr = head + col - 1;
            if (ipntr > m) ipntr = ipntr - m;
            jpntr = head;
            for (jy = 1; jy <= col; ++jy) {  // :1756-1776
                js = m + jy;
                temp1 = list_sum(n, ind, pbegin, pend,
                                 [&](i64 k1) { return WY(k1, ipntr) * WY(k1, jpntr); }, pf);
                temp2 = list_sum(n, ind, dbegin, dend,
                                 [&](i64 k1) { return WS(k1, ipntr) * WS(k1, jpntr); }, pa);
                temp3 = list_sum(n, ind, dbegin, dend,
                                 [&](i64 k1) { return WS(k1, ipntr) * WY(k1, jpntr); }, pa);
                WN1(iy, jy) = temp1;
                WN1(is, js) = temp2;
                WN1(is, jy) = temp3;
                jpntr = jpntr % m + 1;
            }
            jy = col;
            jpntr = head + col - 1;
            if (jpntr > m) jpntr = jpntr - m;
            ipntr = head;
            for (int i = 1; i <= col; ++i) {  // :1783-1793
                is = m + i;
                temp3 = list_sum(n, ind, pbegin, pend,
                                 [&](i64 k1) { return WS(k1, ipntr) * WY(k1, jpntr); }, pf);
                ipntr = ipntr % m + 1;
                WN1(is, jy) = temp3;
            }
            upcl = col - 1;
        } else {
            upcl = col;
        }

        ipntr = head;
        for (iy = 1; iy <= upcl; ++iy) {  // :1802-1826
            is = m + iy;
            jpntr = head;
            for (jy = 1; jy <= iy; ++jy) {
                js = m + jy;
                temp1 = list_sum(n, indx2, 1, nenter,
                                 [&](i64 k1) { return WY(k1, ipntr) * WY(k1, jpntr); }, pe);
                temp2 = list_sum(n, indx2, 1, nenter,
                                 [&](i64 k1) { return WS(k1, ipntr) * WS(k1, jpntr); }, pe);
                temp3 = list_sum(n, indx2, ileave, n,
                                 [&](i64 k1) { return WY(k1, ipntr) * WY(k1, jpntr); }, pl);
                temp4 = list_sum(n, indx2, ileave, n,
                                 [&](i64 k1) { return WS(k1, ipntr) * WS(k1, jpntr); }, pl);
                WN1(iy, jy) = WN1(iy, jy) + temp1 - temp3;
                WN1(is, js) = WN1(is, js) - temp2 + temp4;
                jpntr = jpntr % m + 1;
            }
            ipntr = ipntr % m + 1;
        }
        ipntr = head;
        for (is = m + 1; is <= m + upcl; ++is) {  // :1830-1851
            jpntr = head;
            for (jy = 1; jy <= upcl; ++jy) {
                temp1 = list_sum(n, indx2, 1, nenter,
                                 [&](i64 k1) { return WS(k1, ipntr) * WY(k1, jpntr); }, pe);
                temp3 = list_sum(n, indx2, ileave, n,
                                 [&](i64 k1) { return WS(k1, ipntr) * WY(k1, jpntr); }, pl);
                if (is <= jy + m) {
                    WN1(is, jy) = WN1(is, jy) + temp1 - temp3;
                } else {
                    WN1(is, jy) = WN1(is, jy) - temp1 + temp3;
                }
                jpntr = jpntr % m + 1;
            }
            ipntr = ipntr % m + 1;
        }

        for (iy = 1; iy <= col; ++iy) {  // :1857-1873
            is = col + iy;
            is1 = m + iy;
            for (jy = 1; jy <= iy; ++jy) {
                js = col + jy;
                js1 = m + jy;
                WN(jy, iy) = WN1(iy, jy) / theta;
                WN(js, is) = WN1(is1, js1) * theta;
            }
            for (jy = 1; jy <= iy - 1; ++jy) WN(jy, is) = -WN1(is1, jy);
            for (jy = iy; jy <= col; ++jy) WN(jy, is) = WN1(is1, jy);
            WN(iy, iy) = WN(iy, iy) + SY(iy, iy);
        }

        dpofa(wn0, m2, col, info);  // :1880
        if (info != 0) {
            info = -1;
            return;
        }
        col2 = 2 * col;
        for (js = col + 1; js <= col2; ++js) dtrsl(wn0, m2, col, &WN(1, js), 11, info);
        for (is = col + 1; is <= col2; ++is)
            for (js = is; js <= col2; ++js)
                WN(is, js) = WN(is, js) + ddot(col, &WN(1, is), &WN(1, js));
        dpofa(&WN(col + 1, col + 1), m2, col, info);  // :1902
        if (info != 0) {
            info = -2;
            return;
        }
        (void)zero;
#undef WN
#undef WN1
#undef SY
#undef WY
#undef WS
    }

    // formt :1926-1963
    static void formt(int m, T* wt0, const T* sy0, const T* ss0, int col, T theta, int& info) {
#define WT(i, j) wt0[((i)-1) + (i64)((j)-1) * m]
#define SY(i, j) sy0[((i)-1) + (i64)((j)-1) * m]
#define SS(i, j) ss0[((i)-1) + (i64)((j)-1) * m]
        for (int j = 1; j <= col; ++j) WT(1, j) = theta * SS(1, j);
        for (int i = 2; i <= col; ++i) {
            for (int j = i; j <= col; ++j) {
                int k1 = std::min(i, j) - 1;
                T ddum = (T)0;
                for (int k = 1; k <= k1; ++k) ddum = ddum + SY(i, k) * SY(j, k) / SY(k, k);
                WT(i, j) = ddum + theta * SS(i, j);
            }
        }
        dpofa(wt0, m, col, info);
        if (info != 0) info = -3;
#undef WT
#undef SY
#undef SS
    }

    // freev :1980-2059
    static void freev(i64 n, i64& nfree, int* index0, i64& nenter, i64& ileave, int* indx20,
                      const int* iwhere0, bool& wrk, bool updatd, bool cnstnd, i64 iter) {
        int *index = index0 - 1, *indx2 = indx20 - 1;
        const int* iwhere = iwhere0 - 1;
        nenter = 0;
        ileave = n + 1;
        if (iter > 0 && cnstnd) {
            for (i64 i = 1; i <= nfree; ++i) {
                int k = index[i];
                if (iwhere[k] > 0) {
                    ileave = ileave - 1;
                    indx2[ileave] = k;
                }
            }
            for (i64 i = 1 + nfree; i <= n; ++i) {
                int k = index[i];
                if (iwhere[k] <= 0) {
                    nenter = nenter + 1;
                    indx2[nenter] = k;
                }
            }
        }
        wrk = (ileave < n + 1) || (nenter > 0) || updatd;
        nfree = 0;
        i64 iact = n + 1;
        for (i64 i = 1; i <= n; ++i) {
            if (iwhere[i] <= 0) {
                nfree = nfree + 1;
                index[nfree] = (int)i;
            } else {
                iact = iact - 1;
                index[iact] = (int)i;
            }
        }
    }

    // dcstep :3227-3415
    static void dcstep(T& stx, T& fx, T& dx, T& sty, T& fy, T& dy, T& stp, T fp, T dp,
                       bool& brackt, T stpmin, T stpmax) {
        const T zero = (T)0, two = (T)2, three = (T)3, p66 = (T)0.66;
        T gamma, p, q, r, s, sgnd, stpc, stpf, stpq, theta;
        sgnd = dp * (dx / std::fabs(dx));
        if (fp > fx) {
            theta = three * (fx - fp) / (stp - stx) + dx + dp;
            s = std::max(std::max(std::fabs(theta), std::fabs(dx)), std::fabs(dp));
            gamma = s * std::sqrt((theta / s) * (theta / s) - (dx / s) * (dp / s));
            if (stp < stx) gamma = -gamma;
            p = (gamma - dx) + theta;
            q = ((gamma - dx) + gamma) + dp;
            r = p / q;
            stpc = stx + r * (stp - stx);
            stpq = stx + ((dx / ((fx - fp) / (stp - stx) + dx)) / two) * (stp - stx);
            if (std::fabs(stpc - stx) < std::fabs(stpq - stx)) {
                stpf = stpc;
            } else {
                stpf = stpc + (stpq - stpc) / two;
            }
            brackt = true;
        } else if (sgnd < zero) {
            theta = three * (fx - fp) / (stp - stx) + dx + dp;
            s = std::max(std::max(std::fabs(theta), std::fabs(dx)), std::fabs(dp));
            gamma = s * std::sqrt((theta / s) * (theta / s) - (dx / s) * (dp / s));
            if (stp > stx) gamma = -gamma;
            p = (gamma - dp) + theta;
            q = ((gamma - dp) + gamma) + dx;
            r = p / q;
            stpc = stp + r * (stx - stp);
            stpq = stp + (dp / (dp - dx)) * (stx - stp);
            if (std::fabs(stpc - stp) > std::fabs(stpq - stp)) {
                stpf = stpc;
            } else {
                stpf = stpq;
            }
            brackt = true;
        } else if (std::fabs(dp) < std::fabs(dx)) {
            theta = three * (fx - fp) / (stp - stx) + dx + dp;
            s = std::max(std::max(std::fabs(theta), std::fabs(dx)), std::fabs(dp));
            gamma = s * std::sqrt(std::max(zero, (theta / s) * (theta / s) - (dx / s) * (dp / s)));
            if (stp > stx) gamma = -gamma;
            p = (gamma - dp) + theta;
            q = (gamma + (dx - dp)) + gamma;
            r = p / q;
            if (r < zero && gamma != zero) {
                stpc = stp + r * (stx - stp);
            } else if (stp > stx) {
                stpc = stpmax;
            } else {
                stpc = stpmin;
            }
            stpq = stp + (dp / (dp - dx)) * (stx - stp);
            if (brackt) {
                if (std::fabs(stpc - stp) < std::fabs(stpq - stp)) {
                    stpf = stpc;
                } else {
                    stpf = stpq;
                }
                if (stp > stx) {
                    stpf = std::min(stp + p66 * (sty - stp), stpf);
                } else {
                    stpf = std::max(stp + p66 * (sty - stp), stpf);
                }
            } else {
                if (std::fabs(stpc - stp) > std::fabs(stpq - stp)) {
                    stpf = stpc;
                } else {
                    stpf = stpq;
                }
                stpf = std::min(stpmax, stpf);
                stpf = std::max(stpmin, stpf);
            }
        } else {
            if (brackt) {
                theta = three * (fp - fy) / (sty - stp) + dy + dp;
                s = std::max(std::max(std::fabs(theta), std::fabs(dy)), std::fabs(dp));
                gamma = s * std::sqrt((theta / s) * (theta / s) - (dy / s) * (dp / s));
                if (stp > sty) gamma = -gamma;
                p = (gamma - dp) + theta;
                q = ((gamma - dp) + gamma) + dy;
                r = p / q;
                stpc = stp + r * (sty - stp);
                stpf = stpc;
            } else if (stp > stx) {
                stpf = stpmax;
            } else {
                stpf = stpmin;
            }
        }
        if (fp > fx) {
            sty = stp;
            fy = fp;
            dy = dp;
        } else {
            if (sgnd < zero) {
                sty = stx;
                fy = fx;
                dy = dx;
            }
            stx = stp;
            fx = fp;
            dx = dp;
        }
        stp = stpf;
    }

    // dcsrch :2942-3198.  isave(2), dsave(13) are 0-based here.
    static void dcsrch(T& f, T& g, T& stp, T ftol, T gtol, T xtol, T stpmin, T stpmax, char* task,
                       int* isave, T* dsave) {
        const T zero = (T)0, p5 = (T)0.5, p66 = (T)0.66, xtrapl = (T)1.1, xtrapu = (T)4.0;
        bool brackt;
        int stage;
        T finit, ftest, fm, fx, fxm, fy, fym, ginit, gtest, gm, gx, gxm, gy, gym, stx, sty, stmin,
            stmax, width, width1;
        auto save_locals = [&]() {
            isave[0] = brackt ? 1 : 0;
            isave[1] = stage;
            dsave[0] = ginit;
            dsave[1] = gtest;
            dsave[2] = gx;
            dsave[3] = gy;
            dsave[4] = finit;
            dsave[5] = fx;
            dsave[6] = fy;
            dsave[7] = stx;
            dsave[8] = sty;
            dsave[9] = stmin;
            dsave[10] = stmax;
            dsave[11] = width;
            dsave[12] = width1;
        };
        if (str_pre(task, "START")) {
            if (stp < stpmin) set_str(task, "ERROR: STP < STPMIN");
            if (stp > stpmax) set_str(task, "ERROR: STP > STPMAX");
            if (g >= zero) set_str(task, "ERROR: INITIAL G >= ZERO");
            if (ftol < zero) set_str(task, "ERROR: FTOL < ZERO");
            if (gtol < zero) set_str(task, "ERROR: GTOL < ZERO");
            if (xtol < zero) set_str(task, "ERROR: XTOL < ZERO");
            if (stpmin < zero) set_str(task, "ERROR: STPMIN < ZERO");
            if (stpmax < stpmin) set_str(task, "ERROR: STPMAX < STPMIN");
            if (str_pre(task, "ERROR")) return;
            brackt = false;
            stage = 1;
            finit = f;
            ginit = g;
            gtest = ftol * ginit;
            width = stpmax - stpmin;
            width1 = width / p5;
            stx = zero;
            fx = finit;
            gx = ginit;
            sty = zero;
            fy = finit;
            gy = ginit;
            stmin = zero;
            stmax = stp + xtrapu * stp;
            set_str(task, "FG");
            save_locals();
            return;
        } else {
            brackt = (isave[0] == 1);
            stage = isave[1];
            ginit = dsave[0];
            gtest = dsave[1];
            gx = dsave[2];
            gy = dsave[3];
            finit = dsave[4];
            fx = dsave[5];
            fy = dsave[6];
            stx = dsave[7];
            sty = dsave[8];
            stmin = dsave[9];
            stmax = dsave[10];
            width = dsave[11];
            width1 = dsave[12];
        }
        ftest = finit + stp * gtest;
        if (stage == 1 && f <= ftest && g >= zero) stage = 2;
        if (brackt && (stp <= stmin || stp >= stmax))
            set_str(task, "WARNING: ROUNDING ERRORS PREVENT PROGRESS");
        if (brackt && stmax - stmin <= xtol * stmax) set_str(task, "WARNING: XTOL TEST SATISFIED");
        if (stp == stpmax && f <= ftest && g <= gtest) set_str(task, "WARNING: STP = STPMAX");
        if (stp == stpmin && (f > ftest || g >= gtest)) set_str(task, "WARNING: STP = STPMIN");
        if (f <= ftest && std::fabs(g) <= gtol * (-ginit)) set_str(task, "CONVERGENCE");
        if (str_pre(task, "WARN") || str_pre(task, "CONV")) {
            save_locals();
            return;
        }
        if (stage == 1 && f <= fx && f > ftest) {
            fm = f - stp * gtest;
            fxm = fx - stx * gtest;
            fym = fy - sty * gtest;
            gm = g - gtest;
            gxm = gx - gtest;
            gym = gy - gtest;
            dcstep(stx, fxm, gxm, sty, fym, gym, stp, fm, gm, brackt, stmin, stmax);
            fx = fxm + stx * gtest;
            fy = fym + sty * gtest;
            gx = gxm + gtest;
            gy = gym + gtest;
        } else {
            dcstep(stx, fx, gx, sty, fy, gy, stp, f, g, brackt, stmin, stmax);
        }
        if (brackt) {
            if (std::fabs(sty - stx) >= p66 * width1) stp = stx + p5 * (sty - stx);
            width1 = width;
            width = std::fabs(sty - stx);
        }
        if (brackt) {
            stmin = std::min(stx, sty);
            stmax = std::max(stx, sty);
        } else {
            stmin = stp + xtrapl * (stp - stx);
            stmax = stp + xtrapu * (stp - stx);
        }
        stp = std::max(stp, stpmin);
        stp = std::min(stp, stpmax);
        if ((brackt && (stp <= stmin || stp >= stmax)) || (brackt && stmax - stmin <= xtol * stmax))
            stp = stx;
        set_str(task, "FG");
        save_locals();
    }

    // lnsrlb :2174-2275
    static void lnsrlb(i64 n, const T* l0, const T* u0, const int* nbd0, T* x0, T f, T& fold, T& gd,
                       T& gdold, const T* g0, const T* d0, T* r0, T* t0, const T* z0, T& stp,
                       T& dnorm, T& dtd, T& xstep, T& stpmx, i64 iter, int& ifun, int& iback,
                       int& nfgv, int& info, char* task, bool boxed, bool cnstnd, char* csave,
                       int* isave, T* dsave) {
        const T *l = l0 - 1, *u = u0 - 1, *d = d0 - 1, *t = t0 - 1;
        const int* nbd = nbd0 - 1;
        T* x = x0 - 1;
        const T zero = (T)0, one = (T)1;
        const T big = (T)1.0e+10, ftol = (T)1.0e-3, gtol = (T)0.9, xtol = (T)0.1;
        T a1, a2;
        if (!str_pre(task, "FG_LN")) {
            dtd = ddot(n, d0, d0);
            dnorm = std::sqrt(dtd);
            stpmx = big;
            if (cnstnd) {
                if (iter == 0) {
                    stpmx = one;
                } else {
                    for (i64 i = 1; i <= n; ++i) {
                        a1 = d[i];
                        if (nbd[i] != 0) {
                            if (a1 < zero && nbd[i] <= 2) {
                                a2 = l[i] - x[i];
                                if (a2 >= zero) {
                                    stpmx = zero;
                                } else if (a1 * stpmx < a2) {
                                    stpmx = a2 / a1;
                                }
                            } else if (a1 > zero && nbd[i] >= 2) {
                                a2 = u[i] - x[i];
                                if (a2 <= zero) {
                                    stpmx = zero;
                                } else if (a1 * stpmx > a2) {
                                    stpmx = a2 / a1;
                                }
                            }
                        }
                    }
                }
            }
            if (iter == 0 && !boxed) {
                stp = std::min(one / dnorm, stpmx);
            } else {
                stp = one;
            }
            dcopy(n, x0, t0);
            dcopy(n, g0, r0);
            fold = f;
            ifun = 0;
            iback = 0;
            set_str(csave, "START");
        }
        gd = ddot(n, g0, d0);
        if (ifun == 0) {
            gdold = gd;
            if (gd >= zero) {
                // the reference prints ' ascent direction in projection gd = ' here
                // unconditionally (:2250); the oracle stays silent.
                g_events[1]++;
                info = -4;
                return;
            }
        }
        T fcopy = f;
        dcsrch(fcopy, gd, stp, ftol, gtol, xtol, zero, stpmx, csave, isave, dsave);
        xstep = stp * dnorm;
        if (!str_pre(csave, "CONV") && !str_pre(csave, "WARN")) {
            set_str(task, "FG_LNSRCH");
            ifun = ifun + 1;
            nfgv = nfgv + 1;
            iback = ifun - 1;
            if (stp == one) {
                dcopy(n, z0, x0);
            } else {
                for (i64 i = 1; i <= n; ++i) x[i] = stp * d[i] + t[i];
            }
        } else {
            set_str(task, "NEW_X");
        }
    }

    // matupd :2291-2346
    static void matupd(i64 n, int m, T* ws0, T* wy0, T* sy0, T* ss0, const T* d0, const T* r0,
                       int& itail, int iupdat, int& col, int& head, T& theta, T rr, T dr, T stp,
                       T dtd) {
#define SY(i, j) sy0[((i)-1) + (i64)((j)-1) * m]
#define SS(i, j) ss0[((i)-1) + (i64)((j)-1) * m]
#define WY(i, j) wy0[((i)-1) + (i64)((j)-1) * n]
#define WS(i, j) ws0[((i)-1) + (i64)((j)-1) * n]
        if (iupdat <= m) {
            col = iupdat;
            itail = (head + iupdat - 2) % m + 1;
        } else {
            itail = itail % m + 1;
            head = head % m + 1;
        }
        dcopy(n, d0, &WS(1, itail));
        dcopy(n, r0, &WY(1, itail));
        theta = rr / dr;
        if (iupdat > m) {
            for (int j = 1; j <= col - 1; ++j) {
                dcopy(j, &SS(2, j + 1), &SS(1, j));
                dcopy(col - j, &SY(j + 1, j + 1), &SY(j, j));
            }
        }
        int pointr = head;
        for (int j = 1; j <= col - 1; ++j) {
            SY(col, j) = ddot(n, d0, &WY(1, pointr));
            SS(j, col) = ddot(n, &WS(1, pointr), d0);
            pointr = pointr % m + 1;
        }
        if (stp == (T)1) {
            SS(col, col) = dtd;
        } else {
            SS(col, col) = stp * stp * dtd;
        }
        SY(col, col) = dr;
#undef SY
#undef SS
#undef WY
#undef WS
    }

    // projgr :2594-2622
    static void projgr(i64 n, const T* l0, const T* u0, const int* nbd0, const T* x0, const T* g0,
                       T& sbgnrm) {
        const T *l = l0 - 1, *u = u0 - 1, *x = x0 - 1, *g = g0 - 1;
        const int* nbd = nbd0 - 1;
        sbgnrm = (T)0;
        for (i64 i = 1; i <= n; ++i) {
            T gi = g[i];
            if (nbd[i] != 0) {
                if (gi < (T)0) {
                    if (nbd[i] >= 2) gi = std::max((x[i] - u[i]), gi);
                } else {
                    if (nbd[i] <= 2) gi = std::min((x[i] - l[i]), gi);
                }
            }
            sbgnrm = std::max(sbgnrm, std::fabs(gi));
        }
    }

    // subsm :2676-2885
    static void subsm(i64 n, int m, i64 nsub, const int* ind0, const T* l0, const T* u0,
                      const int* nbd0, T* x0, T* d0, T* xp0, const T* ws0, const T* wy0, T theta,
                      const T* xx0, const T* gg0, int col, int head, int& iword, T* wv0,
                      const T* wn0, int& info) {
        const int* ind = ind0 - 1;
        const T *l = l0 - 1, *u = u0 - 1, *xx = xx0 - 1, *gg = gg0 - 1;
        const int* nbd = nbd0 - 1;
        T *x = x0 - 1, *d = d0 - 1, *wv = wv0 - 1;
#define WY(i, j) wy0[((i)-1) + (i64)((j)-1) * n]
#define WS(i, j) ws0[((i)-1) + (i64)((j)-1) * n]
        const T zero = (T)0, one = (T)1;
        int pointr, m2, col2, jy, js;
        i64 ibd, i, j, k;
        T alpha, xk, dk, temp1, temp2, dd_p;
        if (nsub <= 0) return;

        // wv = W'Zd :2742-2754
        std::vector<T> dfull;  // by-variable copy of the compact d for device-order sums
        if (g_sum_mode == 1) {
            dfull.assign(n, zero);
            for (j = 1; j <= nsub; ++j) dfull[ind[j] - 1] = d[j];
        }
        pointr = head;
        for (int ii = 1; ii <= col; ++ii) {
            if (g_sum_mode == 1) {
                const T* wyc = &WY(1, pointr);
                const T* wsc = &WS(1, pointr);
                const T* df = dfull.data();
                temp1 = device_order_sum<T>(n, [&](i64 q) { return wyc[q] * df[q]; });
                temp2 = device_order_sum<T>(n, [&](i64 q) { return wsc[q] * df[q]; });
            } else {
                temp1 = zero;
                temp2 = zero;
                for (j = 1; j <= nsub; ++j) {
                    k = ind[j];
                    temp1 = temp1 + WY(k, pointr) * d[j];
                    temp2 = temp2 + WS(k, pointr) * d[j];
                }
            }
            wv[ii] = temp1;
            wv[col + ii] = theta * temp2;
            pointr = pointr % m + 1;
        }
        m2 = 2 * m;
        col2 = 2 * col;
        dtrsl(wn0, m2, col2, wv0, 11, info);
        if (info != 0) return;
        for (int ii = 1; ii <= col; ++ii) wv[ii] = -wv[ii];
        dtrsl(wn0, m2, col2, wv0, 1, info);
        if (info != 0) return;

        pointr = head;
        for (jy = 1; jy <= col; ++jy) {  // :2770-2778
            js = col + jy;
            for (i = 1; i <= nsub; ++i) {
                k = ind[i];
                d[i] = d[i] + WY(k, pointr) * wv[jy] / theta + WS(k, pointr) * wv[js];
            }
            pointr = pointr % m + 1;
        }
        dscal(nsub, one / theta, d0);

        iword = 0;
        dcopy(n, x0, xp0);
        for (i = 1; i <= nsub; ++i) {  // :2789-2816
            k = ind[i];
            dk = d[i];
            xk = x[k];
            if (nbd[k] != 0) {
                if (nbd[k] == 1) {
                    x[k] = std::max(l[k], xk + dk);
                    if (x[k] == l[k]) iword = 1;
                } else {
                    if (nbd[k] == 2) {
                        xk = std::max(l[k], xk + dk);
                        x[k] = std::min(u[k], xk);
                        if (x[k] == l[k] || x[k] == u[k]) iword = 1;
                    } else {
                        if (nbd[k] == 3) {
                            x[k] = std::min(u[k], xk + dk);
                            if (x[k] == u[k]) iword = 1;
                        }
                    }
                }
            } else {
                x[k] = xk + dk;
            }
        }
        if (iword == 0) return;

        if (g_sum_mode == 1) {
            dd_p = device_order_sum<T>(n, [&](i64 q) { return (x0[q] - xx0[q]) * gg0[q]; });
        } else {
            dd_p = zero;
            for (i = 1; i <= n; ++i) dd_p = dd_p + (x[i] - xx[i]) * gg[i];
        }
        if (dd_p <= zero) return;
        g_events[0]++;

        dcopy(n, xp0, x0);
        alpha = one;
        temp1 = alpha;
        ibd = 0;
        for (i = 1; i <= nsub; ++i) {  // :2839-2863
            k = ind[i];
            dk = d[i];
            if (nbd[k] != 0) {
                if (dk < zero && nbd[k] <= 2) {
                    temp2 = l[k] - x[k];
                    if (temp2 >= zero) {
                        temp1 = zero;
                    } else if (dk * alpha < temp2) {
                        temp1 = temp2 / dk;
                    }
                } else if (dk > zero && nbd[k] >= 2) {
                    temp2 = u[k] - x[k];
                    if (temp2 <= zero) {
                        temp1 = zero;
                    } else if (dk * alpha > temp2) {
                        temp1 = temp2 / dk;
                    }
                }
                if (temp1 < alpha) {
                    alpha = temp1;
                    ibd = i;
                }
            }
        }
        if (alpha < one) {
            dk = d[ibd];
            k = ind[ibd];
            if (dk > zero) {
                x[k] = u[k];
                d[ibd] = zero;
            } else if (dk < zero) {
                x[k] = l[k];
                d[ibd] = zero;
            }
        }
        for (i = 1; i <= nsub; ++i) {
            k = ind[i];
            x[k] = x[k] + alpha * d[i];
        }
        (void)xp0;
#undef WY
#undef WS
    }

    // mainlb :312-949.  isave is mainlb's Isave(1:23) (0-based here), i.e. the
    // public isave(22:44).
    static void mainlb(i64 n, int m, T* x, const T* l, const T* u, const int* nbd, T& f, T* g,
                       T factr, T pgtol, T* ws, T* wy, T* sy, T* ss, T* wt, T* wn, T* snd, T* z,
                       T* r, T* d, T* t, T* xp, T* wa, int* index, int* iwhere, int* indx2,
                       char* task, int iprint, char* csave, int* lsave, int* isave, T* dsave) {
        const T zero = (T)0, one = (T)1;
        bool prjctd, cnstnd, boxed, updatd, wrk = false;
        i64 k = 0, nseg_l, nfree, nact, ileave, nenter, nintol, iter;
        int itfile, iback, nskip, head, col, itail, iupdat, nfgv, info, ifun, iword;
        T theta, fold, dr, rr, tol, xstep = zero, sbgnrm, ddum, dnorm, dtd, epsmch, cpu1, cpu2,
                                   cachyt, sbtime, lnscht, time1, gd, gdold, stp, stpmx;

        auto save_locals = [&]() {  // :904-947
            lsave[0] = prjctd;
            lsave[1] = cnstnd;
            lsave[2] = boxed;
            lsave[3] = updatd;
            isave[0] = (int)nintol;
            isave[2] = itfile;
            isave[3] = iback;
            isave[4] = nskip;
            isave[5] = head;
            isave[6] = col;
            isave[7] = itail;
            isave[8] = (int)iter;
            isave[9] = iupdat;
            isave[11] = (int)nseg_l;
            isave[12] = nfgv;
            isave[13] = info;
            isave[14] = ifun;
            isave[15] = iword;
            isave[16] = (int)nfree;
            isave[17] = (int)nact;
            isave[18] = (int)ileave;
            isave[19] = (int)nenter;
            dsave[0] = theta;
            dsave[1] = fold;
            dsave[2] = tol;
            dsave[3] = dnorm;
            dsave[4] = epsmch;
            dsave[5] = cpu1;
            dsave[6] = cachyt;
            dsave[7] = sbtime;
            dsave[8] = lnscht;
            dsave[9] = time1;
            dsave[10] = gd;
            dsave[11] = stpmx;
            dsave[12] = sbgnrm;
            dsave[13] = stp;
            dsave[14] = gdold;
            dsave[15] = dtd;
        };

        if (str_eq(task, "START")) {  // :430-507
            epsmch = std::numeric_limits<T>::epsilon();
            time1 = (T)cpu_time_now();
            col = 0;
            head = 1;
            theta = one;
            iupdat = 0;
            updatd = false;
            iback = 0;
            itail = 0;
            iword = 0;
            nact = 0;
            ileave = 0;
            nenter = 0;
            fold = zero;
            dnorm = zero;
            cpu1 = zero;
            gd = zero;
            stpmx = zero;
            sbgnrm = zero;
            stp = zero;
            gdold = zero;
            dtd = zero;
            iter = 0;
            nfgv = 0;
            nseg_l = 0;
            nintol = 0;
            nskip = 0;
            nfree = n;
            ifun = 0;
            tol = factr * epsmch;
            cachyt = 0;
            sbtime = 0;
            lnscht = 0;
            info = 0;
            itfile = 0;
            prjctd = cnstnd = boxed = false;
            errclb(n, m, factr, l, u, nbd, task, info, k);
            if (str_pre(task, "ERROR")) {
                // the reference returns here WITHOUT save_locals (:492-497)
                isave[13] = info;  // exposed for tests only (reference leaves isave untouched)
                isave[20] = (int)k;
                return;
            }
            i64 nbdd;
            active(n, l, u, nbd, x, iwhere, prjctd, cnstnd, boxed, nbdd);
            isave[1] = (int)nbdd;  // mainlb Isave(2) is unused by the reference; tests read nbdd here
            set_str(task, "FG_START");
            save_locals();
            return;
        }

        // restore :511-550
        prjctd = lsave[0] != 0;
        cnstnd = lsave[1] != 0;
        boxed = lsave[2] != 0;
        updatd = lsave[3] != 0;
        nintol = isave[0];
        itfile = isave[2];
        iback = isave[3];
        nskip = isave[4];
        head = isave[5];
        col = isave[6];
        itail = isave[7];
        iter = isave[8];
        iupdat = isave[9];
        nseg_l = isave[11];
        nfgv = isave[12];
        info = isave[13];
        ifun = isave[14];
        iword = isave[15];
        nfree = isave[16];
        nact = isave[17];
        ileave = isave[18];
        nenter = isave[19];
        theta = dsave[0];
        fold = dsave[1];
        tol = dsave[2];
        dnorm = dsave[3];
        epsmch = dsave[4];
        cpu1 = dsave[5];
        cachyt = dsave[6];
        sbtime = dsave[7];
        lnscht = dsave[8];
        time1 = dsave[9];
        gd = dsave[10];
        stpmx = dsave[11];
        sbgnrm = dsave[12];
        stp = dsave[13];
        gdold = dsave[14];
        dtd = dsave[15];

        bool compute_pg = true, prelims = true, linesearch = true;
        if (str_pre(task, "FG_LN")) {
            compute_pg = false;
            prelims = false;
        } else if (str_pre(task, "NEW_X")) {
            compute_pg = false;
            prelims = false;
            linesearch = false;
        } else if (!str_pre(task, "FG_ST")) {
            if (str_pre(task, "STOP")) {
                if (std::memcmp(task + 6, "CPU", 3) == 0) {  // task(7:9)=='CPU'
                    dcopy(n, t, x);
                    dcopy(n, r, g);
                    f = fold;
                }
                save_locals();  // finish()
            } else {
                set_str(task, "FG_START");  // start()
                save_locals();
            }
            return;
        }

        if (compute_pg) {  // :579-596
            nfgv = 1;
            projgr(n, l, u, nbd, x, g, sbgnrm);
            if (sbgnrm <= pgtol) {
                set_str(task, "CONVERGENCE: NORM_OF_PROJECTED_GRADIENT_<=_PGTOL");
                save_locals();
                return;
            }
        }

        for (;;) {  // main_loop :599-872
            if (prelims) {
                iword = -1;
                if (!cnstnd && col > 0) {
                    dcopy(n, x, z);
                    wrk = updatd;
                    nseg_l = 0;
                } else {
                    cpu1 = (T)cpu_time_now();
                    cauchy(n, x, l, u, nbd, g, indx2, iwhere, t, d, z, m, wy, ws, sy, wt, theta,
                           col, head, wa, wa + 2 * m, wa + 4 * m, wa + 6 * m, nseg_l, sbgnrm, info,
                           epsmch);
                    if (info != 0) {
                        g_events[2]++;  // refresh the lbfgs memory and restart the iteration
                        info = 0;
                        col = 0;
                        head = 1;
                        theta = one;
                        iupdat = 0;
                        updatd = false;
                        cpu2 = (T)cpu_time_now();
                        cachyt = cachyt + cpu2 - cpu1;
                        prelims = true;
                        linesearch = true;
                        continue;
                    }
                    cpu2 = (T)cpu_time_now();
                    cachyt = cachyt + cpu2 - cpu1;
                    nintol = nintol + nseg_l;
                    freev(n, nfree, index, nenter, ileave, indx2, iwhere, wrk, updatd, cnstnd,
                          iter);
                    nact = n - nfree;
                }
                if (nfree == 0 || col == 0) {
                    // skip the subspace minimization
                } else {
                    cpu1 = (T)cpu_time_now();
                    if (wrk)
                        formk(n, nfree, index, nenter, ileave, indx2, iupdat, updatd, wn, snd, m, ws,
                              wy, sy, theta, col, head, info);
                    if (info != 0) {
                        g_events[2]++;  // refresh the lbfgs memory and restart the iteration
                        info = 0;
                        col = 0;
                        head = 1;
                        theta = one;
                        iupdat = 0;
                        updatd = false;
                        cpu2 = (T)cpu_time_now();
                        sbtime = sbtime + cpu2 - cpu1;
                        prelims = true;
                        linesearch = true;
                        continue;
                    }
                    cmprlb(n, m, x, g, ws, wy, sy, wt, z, r, wa, index, theta, col, head, nfree,
                           cnstnd, info);
                    if (info == 0) {
                        subsm(n, m, nfree, index, l, u, nbd, z, r, xp, ws, wy, theta, x, g, col,
                              head, iword, wa, wn, info);
                    }
                    if (info != 0) {
                        g_events[2]++;  // refresh the lbfgs memory and restart the iteration
                        info = 0;
                        col = 0;
                        head = 1;
                        theta = one;
                        iupdat = 0;
                        updatd = false;
                        cpu2 = (T)cpu_time_now();
                        sbtime = sbtime + cpu2 - cpu1;
                        prelims = true;
                        linesearch = true;
                        continue;
                    }
                    cpu2 = (T)cpu_time_now();
                    sbtime = sbtime + cpu2 - cpu1;
                }
                for (i64 i = 0; i < n; ++i) d[i] = z[i] - x[i];  // :720-722
                cpu1 = (T)cpu_time_now();
            }

            if (linesearch) {
                lnsrlb(n, l, u, nbd, x, f, fold, gd, gdold, g, d, r, t, z, stp, dnorm, dtd, xstep,
                       stpmx, iter, ifun, iback, nfgv, info, task, boxed, cnstnd, csave,
                       isave + 21, dsave + 16);
                if (info != 0 || iback >= 20) {
                    dcopy(n, t, x);
                    dcopy(n, r, g);
                    f = fold;
                    if (col == 0) {
                        if (info == 0) {
                            info = -9;
                            nfgv = nfgv - 1;
                            ifun = ifun - 1;
                            iback = iback - 1;
                        }
                        set_str(task, "ABNORMAL_TERMINATION_IN_LNSRCH");
                        iter = iter + 1;
                        save_locals();  // finish()
                        return;
                    } else {
                        if (info == 0) nfgv = nfgv - 1;
                        g_events[2]++;  // refresh the lbfgs memory and restart the iteration
                        info = 0;
                        col = 0;
                        head = 1;
                        theta = one;
                        iupdat = 0;
                        updatd = false;
                        set_str(task, "RESTART_FROM_LNSRCH");
                        cpu2 = (T)cpu_time_now();
                        lnscht = lnscht + cpu2 - cpu1;
                        prelims = true;
                        linesearch = true;
                        continue;
                    }
                } else if (str_pre(task, "FG_LN")) {
                    save_locals();
                    return;
                } else {
                    cpu2 = (T)cpu_time_now();
                    lnscht = lnscht + cpu2 - cpu1;
                    iter = iter + 1;
                    projgr(n, l, u, nbd, x, g, sbgnrm);
                    save_locals();
                    return;
                }
            }

            // tests :795-810
            if (sbgnrm <= pgtol) {
                set_str(task, "CONVERGENCE: NORM_OF_PROJECTED_GRADIENT_<=_PGTOL");
                save_locals();
                return;
            }
            ddum = std::max(std::max(std::fabs(fold), std::fabs(f)), one);
            if ((fold - f) <= tol * ddum) {
                set_str(task, "CONVERGENCE: REL_REDUCTION_OF_F_<=_FACTR*EPSMCH");
                if (iback >= 10) info = -5;
                save_locals();
                return;
            }
            for (i64 i = 0; i < n; ++i) r[i] = g[i] - r[i];  // :813-815
            rr = ddot(n, r, r);
            if (stp == one) {
                dr = gd - gdold;
                ddum = -gdold;
            } else {
                dr = (gd - gdold) * stp;
                dscal(n, stp, d);
                ddum = -gdold * stp;
            }
            if (dr <= epsmch * ddum) {  // :826-834
                g_events[3]++;
                nskip = nskip + 1;
                updatd = false;
                prelims = true;
                linesearch = true;
                continue;
            }
            updatd = true;
            iupdat = iupdat + 1;
            matupd(n, m, ws, wy, sy, ss, d, r, itail, iupdat, col, head, theta, rr, dr, stp, dtd);
            formt(m, wt, sy, ss, col, theta, info);
            if (info != 0) {
                g_events[2]++;  // refresh the lbfgs memory and restart the iteration
                info = 0;
                col = 0;
                head = 1;
                theta = one;
                iupdat = 0;
                updatd = false;
            }
            prelims = true;
            linesearch = true;
        }
    }

    // setulb :88-286.  n is passed by value as 64-bit; the int32 isave(1:16)
    // slots are filled as the reference does when they fit.
    static void setulb(i64 n, int m, T* x, const T* l, const T* u, const int* nbd, T* f, T* g,
                       T factr, T pgtol, T* wa, int* iwa, char* task, int iprint, char* csave,
                       int* lsave, int* isave, T* dsave) {
        i64 mn = (i64)m * n, m2 = (i64)m * m, m24 = 4 * m2;
        i64 lws = 1, lwy = lws + mn, lsy = lwy + mn, lss = lsy + m2, lwt = lss + m2,
            lwn = lwt + m2, lsnd = lwn + m24, lz = lsnd + m24, lr = lz + n, ld = lr + n,
            lt = ld + n, lxp = lt + n, lwa = lxp + n;
        if (str_eq(task, "START")) {
            i64 v[16] = {mn, m2, m24, lws, lwy, lsy, lss, lwt, lwn, lsnd, lz, lr, ld, lt, lxp, lwa};
            for (int q = 0; q < 16; ++q)
                isave[q] = (v[q] <= 2147483647LL) ? (int)v[q] : -1;
        }
        mainlb(n, m, x, l, u, nbd, *f, g, factr, pgtol, wa + (lws - 1), wa + (lwy - 1),
               wa + (lsy - 1), wa + (lss - 1), wa + (lwt - 1), wa + (lwn - 1), wa + (lsnd - 1),
               wa + (lz - 1), wa + (lr - 1), wa + (ld - 1), wa + (lt - 1), wa + (lxp - 1),
               wa + (lwa - 1), iwa, iwa + n, iwa + 2 * n, task, iprint, csave, lsave, isave + 21,
               dsave);
    }

    // The sample problem of test/driver1.f90:274-289 (same in driver2/driver3):
    // bounded extended Rosenbrock, summed left to right.
    static void rosenbrock_fg(i64 n, const T* x0, T* f, T* g0) {
        const T* x = x0 - 1;
        T* g = g0 - 1;
        T ff = (T)0.25 * (x[1] - (T)1) * (x[1] - (T)1);
        for (i64 i = 2; i <= n; ++i) {
            T q = x[i] - x[i - 1] * x[i - 1];
            ff = ff + q * q;
        }
        *f = (T)4 * ff;
        T t1 = x[2] - x[1] * x[1], t2;
        g[1] = (T)2 * (x[1] - (T)1) - (T)16 * x[1] * t1;
        for (i64 i = 2; i <= n - 1; ++i) {
            t2 = t1;
            t1 = x[i + 1] - x[i] * x[i];
            g[i] = (T)8 * t2 - (T)16 * x[i] * t1;
        }
        g[n] = (T)8 * t1;
    }
};

static uint64_t splitmix64(uint64_t v) {
    v += 0x9E3779B97F4A7C15ULL;
    v = (v ^ (v >> 30)) * 0xBF58476D1CE4E5B9ULL;
    v = (v ^ (v >> 27)) * 0x94D049BB133111EBULL;
    return v ^ (v >> 31);
}

}  // namespace

// ---------------------------------------------------------------------------
// C ABI (mirrors include/lbfgsb_b200.h's host twin, so a test can drive either)
// ---------------------------------------------------------------------------
extern "C" {

void oracle_set_sum_mode(int mode) { g_sum_mode = mode; }
void oracle_set_tie_mode(int mode) { g_tie_mode = mode; }
void oracle_event_counts(long long* out, int reset) {
    for (int i = 0; i < 8; ++i) { out[i] = g_events[i]; if (reset) g_events[i] = 0; }
}
int oracle_get_sum_mode() { return g_sum_mode; }

void oracle_setulb_f64(const int64_t* n, const int32_t* m, double* x, const double* l,
                       const double* u, const int32_t* nbd, double* f, double* g,
                       const double* factr, const double* pgtol, double* wa, int32_t* iwa,
                       char* task, const int32_t* iprint, char* csave, int32_t* lsave,
                       int32_t* isave, double* dsave) {
    LB<double>::setulb(*n, *m, x, l, u, nbd, f, g, *factr, *pgtol, wa, iwa, task, *iprint, csave,
                       lsave, isave, dsave);
}
void oracle_setulb_f32(const int64_t* n, const int32_t* m, float* x, const float* l, const float* u,
                       const int32_t* nbd, float* f, float* g, const float* factr,
                       const float* pgtol, float* wa, int32_t* iwa, char* task,
                       const int32_t* iprint, char* csave, int32_t* lsave, int32_t* isave,
                       float* dsave) {
    LB<float>::setulb(*n, *m, x, l, u, nbd, f, g, *factr, *pgtol, wa, iwa, task, *iprint, csave,
                      lsave, isave, dsave);
}

void oracle_rosenbrock_fg_f64(int64_t n, const double* x, double* f, double* g) {
    LB<double>::rosenbrock_fg(n, x, f, g);
}
void oracle_rosenbrock_fg_f32(int64_t n, const float* x, float* f, float* g) {
    LB<float>::rosenbrock_fg(n, x, f, g);
}

// 64-bit identity of the active set {i : iwhere(i) > 0} (freev :2047): the sum
// (mod 2^64) of splitmix64(i), i 0-based -- order independent, so the CUDA
// path can produce the same number with integer adds in any order.
void oracle_active_set_hash(int64_t n, const int32_t* iwhere, uint64_t* hash, int64_t* count) {
    uint64_t h = 0;
    int64_t c = 0;
    for (int64_t i = 0; i < n; ++i)
        if (iwhere[i] > 0) {
            h += splitmix64((uint64_t)i);
            ++c;
        }
    *hash = h;
    *count = c;
}

// Stand-alone kernels for per-routine parity tests (0-based arrays in, same
// semantics as the reference routine named).
void oracle_projgr_f64(int64_t n, const double* l, const double* u, const int32_t* nbd,
                       const double* x, const double* g, double* sbgnrm) {
    LB<double>::projgr(n, l, u, nbd, x, g, *sbgnrm);
}
void oracle_dpofa_f64(double* a, int32_t lda, int32_t n, int32_t* info) {
    int inf = 0;
    LB<double>::dpofa(a, lda, n, inf);
    *info = inf;
}
void oracle_dtrsl_f64(const double* t, int32_t ldt, int32_t n, double* b, int32_t job,
                      int32_t* info) {
    int inf = 0;
    LB<double>::dtrsl(t, ldt, n, b, job, inf);
    *info = inf;
}
// bmv :1057-1123, formt :1926-1963 and the dense tail of formk :1853-1906 on their own (per-routine parity tests)
void oracle_bmv_f64(int32_t m, const double* sy, const double* wt, int32_t col, const double* v, double* p, int32_t* info) {
    int inf = 0;
    LB<double>::bmv(m, sy, wt, col, v, p, inf);
    *info = inf;
}
void oracle_formt_f64(int32_t m, double* wt, const double* sy, const double* ss, int32_t col, double theta, int32_t* info) {
    int inf = 0;
    LB<double>::formt(m, wt, sy, ss, col, theta, inf);
    *info = inf;
}
// formk with no new pair and no entering/leaving variable: WN1 stands as given and the routine is its tail --
// assembly of WN from WN1, theta and the diagonal of SY, the two Cholesky factorisations and the column solves.
void oracle_formk_tail_f64(int32_t m, int32_t col, double theta, double* wn, double* wn1, const double* sy, int32_t* info) {
    int inf = 0;
    const int ind[1] = {1}, indx2[1] = {0};
    std::vector<double> w((size_t)m, 0.0);
    LB<double>::formk(1, 1, ind, 0, 2, indx2, m + 1, false, wn, wn1, m, w.data(), w.data(), sy, theta, col, 1, inf);
    *info = inf;
}
void oracle_hpsolb_f64(int64_t n, double* t, int32_t* iorder, int64_t iheap) {
    LB<double>::hpsolb(n, t, iorder, iheap);
}
void oracle_dcsrch_f64(double* f, double* g, double* stp, double ftol, double gtol, double xtol,
                       double stpmin, double stpmax, char* task, int32_t* isave, double* dsave) {
    LB<double>::dcsrch(*f, *g, *stp, ftol, gtol, xtol, stpmin, stpmax, task, isave, dsave);
}

// The fixed-shape ("device order") dot product on its own, for the reduction parity tests.
double oracle_device_order_dot_f64(int64_t n, const double* a, const double* b) {
    return device_order_sum<double>(n, [&](i64 i) { return a[i] * b[i]; });
}
float oracle_device_order_dot_f32(int64_t n, const float* a, const float* b) {
    return device_order_sum<float>(n, [&](i64 i) { return a[i] * b[i]; });
}
int oracle_shape(int which) {
    switch (which) { case 0: return LBFGSB_BLOCK; case 1: return LBFGSB_UNROLL_F64; case 2: return LBFGSB_GRID; default: return LBFGSB_FINAL_BLOCK; }
}

}  // extern "C"
