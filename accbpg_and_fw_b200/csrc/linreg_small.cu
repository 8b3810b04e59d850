// Small-shape Poisson / KL regression: the WHOLE BPG loop (algorithms.py:11-72) in one launch.
//
// At the notebook shapes (ipynb/ex_Poisson_L2: 200 x 100, ipynb/ex_KL_regr_L1: 1000 x 100) the arithmetic of an
// iteration is a few microseconds of one SM, while the operator-by-operator loop spends a handful of launches and one
// blocking host read per line-search trip.  When A (m x n doubles) fits in the shared memory of one SM - or of a cluster
// of 2, 4 or 8 CTAs, CTA r holding a contiguous slice of the columns - one persistent launch runs every iteration of
//     BPG(f, h, L, x0, maxitrs, epsilon, linesearch, ls_ratio)
// with f = PoissonRegression / KLdivRegression and h = BurgEntropy(L1, L2) / ShannonEntropy(L1, Simplex):
//
//   top       r(Ax), f(Ax) from the A x the accepted trial formed (carried, not recomputed)   (functions.py:102-120, :140-158)
//             g = A^T r over this CTA's columns                                              (functions.py:112, :150)
//   trial     x1 = h.div_prox_map(x, g, L); this CTA's partial A x1 and its partial n-sums (dot(g, x1 - x), the divergence
//             terms, sum x1, x1.x1); ONE exchange through distributed shared memory adds the partials in rank order, so
//             every CTA holds a bit-identical A x1 and identical scalars, and takes the identical decision
//   test      f(x1) > f(x) + dot + L D(x1, x)  ->  L *= ls_ratio                                   (algorithms.py:46-56)
//
// x, x1 and g live only as the local column slice; the m-vectors (b, A x, A x1, r) are replicated.  Sums are fixed-order
// trees (per thread, warp butterfly, warps in order, CTAs in rank order); the only atomic is the integer OR of status bits.
// Compiled with -fmad=false, as linreg.cu and vecops.cu are: the scalar formulas are theirs and round like NumPy's.
#include <cooperative_groups.h>

#include "common.cuh"

namespace accbpg {

constexpr int LS_THREADS = 512;
constexpr int LS_WARPS = LS_THREADS / 32;
constexpr size_t LS_SMEM_LIMIT = 227 * 1024;       // the shared memory an sm_100 CTA may have (the kernel has no static)
constexpr int LS_NSC = 8;                           // scalars in an exchange: dot, div, sum y, sum x1, x1.x1, status, -, -
enum { SC_DOT = 0, SC_DIV, SC_SY, SC_SX, SC_SQ, SC_ST };

struct LsPlan {
    int NL, ldn;                  // columns per CTA, row pitch of the shared copy of A (odd: conflict-free column walks)
    size_t xstride;               // one exchange buffer: LS_NSC scalars + an m-vector
    size_t off_A, off_b, off_Ax, off_Ax1, off_r, off_xch, off_x, off_x1, off_g, off_scr, off_red, off_st, bytes;
};

__host__ __device__ inline LsPlan ls_plan(int64_t m, int64_t n, int C) {
    LsPlan p;
    p.NL = (int)((n + C - 1) / C);
    p.ldn = p.NL | 1;
    p.xstride = (size_t)LS_NSC + (size_t)m;
    size_t o = 0;
    p.off_A = o;   o += (size_t)m * p.ldn * 8;
    p.off_b = o;   o += (size_t)m * 8;
    p.off_Ax = o;  o += (size_t)m * 8;
    p.off_Ax1 = o; o += (size_t)m * 8;
    p.off_r = o;   o += (size_t)m * 8;
    p.off_xch = o; o += 2 * p.xstride * 8;         // double-buffered: the exchange after next reuses a buffer
    p.off_x = o;   o += (size_t)p.NL * 8;
    p.off_x1 = o;  o += (size_t)p.NL * 8;
    p.off_g = o;   o += (size_t)p.NL * 8;
    p.off_scr = o; o += (size_t)LS_THREADS * 8;    // split partial sums of the two matrix passes
    p.off_red = o; o += (size_t)2 * LS_NSC * LS_WARPS * 8;
    p.off_st = o;  o += 16;                          // this CTA's status word
    p.bytes = o;
    return p;
}

// smallest cluster whose plan fits; 0 when none of <= 8 CTAs does
static int ls_pick_cluster(int64_t m, int64_t n, size_t* bytes) {
    if (m < 1 || n < 1 || m > (1 << 20) || n > (1 << 20)) return 0;
    for (int C = 1; C <= 8; C *= 2) {
        const LsPlan pl = ls_plan(m, n, C);
        if (pl.bytes <= LS_SMEM_LIMIT) { if (bytes) *bytes = pl.bytes; return C; }
    }
    return 0;
}

struct LsParams {
    const double* A; const double* b; int m, n; int64_t lda;
    int kind, hkind;
    double lamda, delta;
    double* x;                       // in: x0, out: the last iterate
    double L, ls_ratio, epsilon;
    int linesearch, maxitrs;
    double* F; double* Ls; double* T;
    double* info;                    // [0] entries written, [1] line-search trials, [2] last L, [3] cluster size
    uint32_t* status;
};

struct LsCtx {
    const double* A; const double* b;
    double *Ax, *Ax1, *r, *xch, *x, *x1, *g, *scr, *red;
    int m, ldn, nloc, col0, rank, tid, lane, warp;
    int qmv, cwmv, qrm, rwrm;        // split of the matrix passes: groups and their widths
    int par, flip;
    uint32_t* st;                    // this CTA's status word (shared)
};

// ---- CTA-wide sums of K values with one barrier (partials alternate between two buffers; every thread adds the warp
//      partials in warp order, so all threads - and all CTAs given the same inputs - get the same bits)
template <int K>
__device__ __forceinline__ void ls_cta_sum(LsCtx& c, double (&v)[K]) {
    double* s = c.red + c.flip * (LS_NSC * LS_WARPS);
    c.flip ^= 1;
#pragma unroll
    for (int q = 0; q < K; ++q) {
        v[q] = warp_sum(v[q]);
        if (c.lane == 0) s[q * LS_WARPS + c.warp] = v[q];
    }
    __syncthreads();
#pragma unroll
    for (int q = 0; q < K; ++q) {
        double a = s[q * LS_WARPS];
#pragma unroll
        for (int w = 1; w < LS_WARPS; ++w) a += s[q * LS_WARPS + w];
        v[q] = a;
    }
}

__device__ __forceinline__ void ls_flag(LsCtx& c, uint32_t st) {
    st = __reduce_or_sync(0xffffffffu, st);
    if (c.lane == 0 && st) atomicOr(c.st, st);
}

// ---- f(Ax) and, when r != nullptr, the residual r(Ax)   (value_resid_kernel in linreg.cu; functions.py:106,110,119 /
//      :144,148,157), over all m rows in every CTA
__device__ __forceinline__ double ls_value(LsCtx& c, int kind, const double* Ax, double* r) {
    double acc[1] = {0.0};
    for (int i = c.tid; i < c.m; i += LS_THREADS) {
        const double a = Ax[i], bi = c.b[i];
        if (kind == ACCBPG_LINREG_POISSON) {
            const double q = bi / a;
            acc[0] += (bi * log(q) + a) - bi;
            if (r) r[i] = 1.0 - q;
        } else {
            const double lg = log(a / bi);
            acc[0] += (a * lg - a) + bi;
            if (r) r[i] = lg;
        }
    }
    ls_cta_sum<1>(c, acc);
    return acc[0];
}

// ---- part[i] = sum over this CTA's columns of A[i][j] v[j]; rows split into qmv column groups when m < LS_THREADS
__device__ __forceinline__ void ls_matvec(const LsCtx& c, const double* v, double* part) {
    const int m = c.m;
    if (c.qmv == 1) {
        for (int i = c.tid; i < m; i += LS_THREADS) {
            const double* a = c.A + (size_t)i * c.ldn;
            double s = 0.0;
            for (int j = 0; j < c.nloc; ++j) s += a[j] * v[j];
            part[i] = s;
        }
        return;
    }
    if (c.tid < c.qmv * m) {
        const int q = c.tid / m, i = c.tid - q * m;
        const int j0 = q * c.cwmv, j1 = min(j0 + c.cwmv, c.nloc);
        const double* a = c.A + (size_t)i * c.ldn;
        double s = 0.0;
        for (int j = j0; j < j1; ++j) s += a[j] * v[j];
        c.scr[c.tid] = s;
    }
    __syncthreads();
    for (int i = c.tid; i < m; i += LS_THREADS) {
        double s = c.scr[i];
        for (int q = 1; q < c.qmv; ++q) s += c.scr[q * m + i];
        part[i] = s;
    }
}

// ---- g[j] = sum_i A[i][j] r[i] for this CTA's columns; the rows split into qrm chunks when nloc < LS_THREADS
__device__ __forceinline__ void ls_rmatvec(const LsCtx& c) {
    const int nl = c.nloc;
    if (c.qrm == 1) {
        for (int j = c.tid; j < nl; j += LS_THREADS) {
            double s = 0.0;
            for (int i = 0; i < c.m; ++i) s += c.A[(size_t)i * c.ldn + j] * c.r[i];
            c.g[j] = s;
        }
    } else {
        if (c.tid < c.qrm * nl) {
            const int q = c.tid / nl, j = c.tid - q * nl;
            const int i0 = q * c.rwrm, i1 = min(i0 + c.rwrm, c.m);
            double s = 0.0;
            for (int i = i0; i < i1; ++i) s += c.A[(size_t)i * c.ldn + j] * c.r[i];
            c.scr[c.tid] = s;
        }
        __syncthreads();
        for (int j = c.tid; j < nl; j += LS_THREADS) {
            double s = c.scr[j];
            for (int q = 1; q < c.qrm; ++q) s += c.scr[q * nl + j];
            c.g[j] = s;
        }
    }
    __syncthreads();
}

// ---- the current exchange buffer's m-vector (ls_matvec writes its partial there)
__device__ __forceinline__ double* ls_part(const LsCtx& c) { return c.xch + (size_t)c.par * (LS_NSC + c.m) + LS_NSC; }

// ---- publish this CTA's LS_NSC scalars (uniform over the CTA) and the partial m-vector (nvec = m or 0), wait for the
//      cluster, add every CTA's partials in rank order: vec_out and sc are then the same bits in every CTA.  The status
//      scalar is OR-ed instead.  A buffer is written again only two exchanges later, after the next exchange's barrier,
//      which every CTA reaches only when it has finished reading this one.
// 32-bit shared::cluster address of p in CTA r of the cluster, and a load through it
__device__ __forceinline__ uint32_t ls_mapa(const void* p, int r) {
    const uint32_t a = (uint32_t)__cvta_generic_to_shared(p);
    uint32_t d;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(d) : "r"(a), "r"(r));
    return d;
}
__device__ __forceinline__ double ls_ld_cluster(uint32_t a) {
    double v;
    asm volatile("ld.shared::cluster.f64 %0, [%1];" : "=d"(v) : "r"(a) : "memory");
    return v;
}

template <int C>
__device__ __forceinline__ void ls_exchange(LsCtx& c, double (&sc)[LS_NSC], int nvec, double* vec_out) {
    namespace cg = cooperative_groups;
    double* buf = c.xch + (size_t)c.par * (LS_NSC + c.m);
    c.par ^= 1;
    if (c.tid == 0) {
#pragma unroll
        for (int q = 0; q < LS_NSC; ++q) buf[q] = sc[q];
    }
    if (C == 1) {
        __syncthreads();
#pragma unroll
        for (int q = 0; q < LS_NSC; ++q) sc[q] = buf[q];
        for (int i = c.tid; i < nvec; i += LS_THREADS) vec_out[i] = buf[LS_NSC + i];
        __syncthreads();
        return;
    }
    cg::this_cluster().sync();
    uint32_t src[C];
#pragma unroll
    for (int r = 0; r < C; ++r) src[r] = ls_mapa(buf, r);
#pragma unroll
    for (int q = 0; q < LS_NSC; ++q) {
        if (q == SC_ST) {
            uint32_t st = 0;
#pragma unroll
            for (int r = 0; r < C; ++r) st |= (uint32_t)ls_ld_cluster(src[r] + 8 * q);
            sc[q] = (double)st;
        } else {
            double a = ls_ld_cluster(src[0] + 8 * q);
#pragma unroll
            for (int r = 1; r < C; ++r) a += ls_ld_cluster(src[r] + 8 * q);
            sc[q] = a;
        }
    }
    for (int i = c.tid; i < nvec; i += LS_THREADS) {
        const uint32_t o = 8 * (LS_NSC + i);
        double a = ls_ld_cluster(src[0] + o);
#pragma unroll
        for (int r = 1; r < C; ++r) a += ls_ld_cluster(src[r] + o);
        vec_out[i] = a;
    }
    __syncthreads();
}

// ---- x1 = h.div_prox_map(x, g, L) on this CTA's columns and the partial n-sums of the trial:
//      dot(g, x1 - x) (vec_dot_diff), the divergence D(x1, x) (burg_divergence: sum (r - log r) - 1; shannon_divergence:
//      sum x1 log((x1+d)/(x+d)), sum x, sum x1), sum x1 and x1.x1 (Psi of x1).  Same formulas, checks and status bits as
//      BurgProxF / shannon_point / BurgDivF / ShannonDivF in vecops.cu.
template <int C>
__device__ __forceinline__ void ls_prox(LsCtx& c, const LsParams& p, double L, bool with_div, double (&sc)[LS_NSC]) {
    const int hk = p.hkind;
    const double lamda = p.lamda, delta = p.delta;
    const bool burg = hk <= ACCBPG_SMALL_H_BURG_L2;
    uint32_t st = 0;
    if (hk == ACCBPG_SMALL_H_SHANNON_SIMPLEX) {
        // y exp(-g/L), normalised by its sum over all n (ShannonProxSumF + DivideBySlotF)
        double s[1] = {0.0};
        for (int j = c.tid; j < c.nloc; j += LS_THREADS) {
            const double yj = c.x[j];
            if (!(yj > 0.0)) st |= ACCBPG_ST_Y_NOT_POS;
            const double v = yj * exp(-c.g[j] / L);
            c.x1[j] = v;
            s[0] += v;
        }
        ls_cta_sum<1>(c, s);
        double t[LS_NSC] = {s[0], 0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
        ls_exchange<C>(c, t, 0, nullptr);
        for (int j = c.tid; j < c.nloc; j += LS_THREADS) c.x1[j] = c.x1[j] / t[0];
    } else {
        const double lamL = lamda / L, four_lamL = 4 * lamL, two_lamL = 2 * lamL;
        for (int j = c.tid; j < c.nloc; j += LS_THREADS) {
            const double yj = c.x[j];
            double gj = c.g[j], v;
            if (burg) {
                if (!(yj > 0.0)) st |= ACCBPG_ST_ARG_NOT_POS;
                const double sj = gj - L * (-1.0 / yj);
                if (hk == ACCBPG_SMALL_H_BURG) {
                    if (!(sj > 0.0)) st |= ACCBPG_ST_PROX_NOT_POS;
                    v = L / sj;
                } else if (hk == ACCBPG_SMALL_H_BURG_L1) {
                    if (!(sj > -lamda)) st |= ACCBPG_ST_PROX_NOT_POS;
                    v = L / (lamda + sj);
                } else {
                    const double gg = sj / L;
                    v = (sqrt(gg * gg + four_lamL) - gg) / two_lamL;
                }
            } else {
                if (lamda != 0.0) gj = lamda + gj;
                if (!(yj >= 0.0)) st |= ACCBPG_ST_ARG_NEGATIVE;
                v = yj * exp(-gj / L);
            }
            c.x1[j] = v;
        }
    }
    double a[5] = {0.0, 0.0, 0.0, 0.0, 0.0};
    for (int j = c.tid; j < c.nloc; j += LS_THREADS) {
        const double xj = c.x1[j], yj = c.x[j];
        if (with_div) {
            a[SC_DOT] += c.g[j] * (xj - yj);
            if (burg) {
                if (!(xj > 0.0) || !(yj > 0.0)) st |= ACCBPG_ST_ARG_NOT_POS;
                const double r = xj / yj;
                a[SC_DIV] += (r - log(r)) - 1.0;
            } else {
                if (!(xj >= 0.0) || !(yj >= 0.0)) st |= ACCBPG_ST_ARG_NEGATIVE;
                a[SC_DIV] += xj * log((xj + delta) / (yj + delta));
                a[SC_SY] += yj;
            }
        }
        a[SC_SX] += xj;
        a[SC_SQ] += xj * xj;
    }
    ls_flag(c, st);
    ls_cta_sum<5>(c, a);                                // (its barrier also publishes x1 and the status word)
#pragma unroll
    for (int q = 0; q < 5; ++q) sc[q] = a[q];
    sc[SC_ST] = (double)*c.st;
    sc[6] = sc[7] = 0.0;
}

// Psi(x) from the exchanged sums, in the operator path's rounding order (BurgEntropyL1 / ShannonEntropyL1: lamda * sum x;
// BurgEntropyL2: (lamda / 2) * x.x)
__device__ __forceinline__ double ls_psi(const LsParams& p, const double (&sc)[LS_NSC]) {
    if (p.hkind == ACCBPG_SMALL_H_BURG_L1 || p.hkind == ACCBPG_SMALL_H_SHANNON_L1) return p.lamda * sc[SC_SX];
    if (p.hkind == ACCBPG_SMALL_H_BURG_L2) return (p.lamda / 2) * sc[SC_SQ];
    return 0.0;
}

__device__ __forceinline__ unsigned long long ls_clock() {
    unsigned long long ns;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(ns));
    return ns;
}

template <int C>
__global__ void __launch_bounds__(LS_THREADS, 1) linreg_bpg_small_kernel(LsParams p) {
    extern __shared__ __align__(16) unsigned char ls_raw[];
    namespace cg = cooperative_groups;
    const unsigned long long ns0 = ls_clock();
    const LsPlan pl = ls_plan(p.m, p.n, C);
    LsCtx c;
    c.A = (const double*)(ls_raw + pl.off_A);
    c.b = (const double*)(ls_raw + pl.off_b);
    c.Ax = (double*)(ls_raw + pl.off_Ax);   c.Ax1 = (double*)(ls_raw + pl.off_Ax1);
    c.r = (double*)(ls_raw + pl.off_r);     c.xch = (double*)(ls_raw + pl.off_xch);
    c.x = (double*)(ls_raw + pl.off_x);     c.x1 = (double*)(ls_raw + pl.off_x1);
    c.g = (double*)(ls_raw + pl.off_g);     c.scr = (double*)(ls_raw + pl.off_scr);
    c.red = (double*)(ls_raw + pl.off_red);
    c.m = p.m; c.ldn = pl.ldn;
    c.rank = (C > 1) ? (int)cg::this_cluster().block_rank() : 0;
    c.col0 = c.rank * pl.NL;
    c.nloc = max(0, min(pl.NL, p.n - c.col0));
    c.tid = threadIdx.x; c.lane = c.tid & 31; c.warp = c.tid >> 5;
    c.qmv = (p.m < LS_THREADS) ? max(1, min(LS_THREADS / p.m, c.nloc)) : 1;
    c.cwmv = (c.nloc + c.qmv - 1) / c.qmv;
    c.qrm = (c.nloc > 0 && c.nloc < LS_THREADS) ? max(1, min(LS_THREADS / c.nloc, p.m)) : 1;
    c.rwrm = (p.m + c.qrm - 1) / c.qrm;
    c.par = 0; c.flip = 0;
    c.st = (uint32_t*)(ls_raw + pl.off_st);
    const bool writer = c.rank == 0 && c.tid == 0;

    // this CTA's columns of A, b, this CTA's slice of x0
    if (c.tid == 0) *c.st = 0u;
    {
        double* As = (double*)(ls_raw + pl.off_A);
        double* bs = (double*)(ls_raw + pl.off_b);
        const int total = p.m * c.nloc;
        for (int e = c.tid; e < total; e += LS_THREADS) {
            const int i = e / c.nloc, j = e - i * c.nloc;
            As[(size_t)i * c.ldn + j] = p.A[(int64_t)i * p.lda + c.col0 + j];
        }
        for (int i = c.tid; i < p.m; i += LS_THREADS) bs[i] = p.b[i];
        for (int j = c.tid; j < c.nloc; j += LS_THREADS) c.x[j] = p.x[c.col0 + j];
    }
    __syncthreads();

    // A x0 and Psi(x0)
    double sc[LS_NSC];
    {
        double a[2] = {0.0, 0.0};
        for (int j = c.tid; j < c.nloc; j += LS_THREADS) { a[0] += c.x[j]; a[1] += c.x[j] * c.x[j]; }
        ls_cta_sum<2>(c, a);
        ls_matvec(c, c.x, ls_part(c));
        for (int q = 0; q < LS_NSC; ++q) sc[q] = 0.0;
        sc[SC_SX] = a[0]; sc[SC_SQ] = a[1];
        ls_exchange<C>(c, sc, p.m, c.Ax);
    }
    double psi_x = ls_psi(p, sc);
    double L = p.L, Fprev = 0.0;
    int k = 0, trials = 0;
    uint32_t st_all = 0;
    for (; k < p.maxitrs; ++k) {
        if (writer) p.T[k] = (double)(ls_clock() - ns0);
        const double fx = ls_value(c, p.kind, c.Ax, c.r);
        const double Fk = fx + psi_x;
        if (writer) p.F[k] = Fk;
        ls_rmatvec(c);
        if (p.linesearch) L = L / p.ls_ratio;
        for (;;) {
            ++trials;
            ls_prox<C>(c, p, L, p.linesearch != 0, sc);
            ls_matvec(c, c.x1, ls_part(c));
            ls_exchange<C>(c, sc, p.m, c.Ax1);
            st_all = (uint32_t)sc[SC_ST];
            if (st_all || !p.linesearch) break;
            const double f1 = ls_value(c, p.kind, c.Ax1, nullptr);
            const bool burg = p.hkind <= ACCBPG_SMALL_H_BURG_L2;
            const double D = burg ? sc[SC_DIV] : sc[SC_DIV] + (sc[SC_SY] - sc[SC_SX]);
            if (f1 > fx + sc[SC_DOT] + L * D) L = L * p.ls_ratio;            // algorithms.py:53
            else break;
        }
        if (st_all) { ++k; break; }
        double* t = c.x; c.x = c.x1; c.x1 = t;
        t = c.Ax; c.Ax = c.Ax1; c.Ax1 = t;
        psi_x = ls_psi(p, sc);
        if (writer) p.Ls[k] = L;
        if (k > 0 && fabs(Fk - Fprev) < p.epsilon) { ++k; break; }              // algorithms.py:66
        Fprev = Fk;
    }
    if (C > 1) cg::this_cluster().sync();               // nobody leaves while its shared memory may still be read
    for (int j = c.tid; j < c.nloc; j += LS_THREADS) p.x[c.col0 + j] = c.x[j];
    if (c.tid == 0 && *c.st) atomicOr(p.status, *c.st);
    if (writer) {
        p.info[0] = (double)k; p.info[1] = (double)trials; p.info[2] = L; p.info[3] = (double)C;
    }
}

template <int C>
static int ls_launch(Ctx* c, cudaStream_t s, const LsParams& p, size_t smem) {
    static bool attr_done[kMaxDevices] = {};
    if (!(c->device >= 0 && c->device < kMaxDevices && attr_done[c->device])) {
        ACCBPG_CUDA(cudaFuncSetAttribute(linreg_bpg_small_kernel<C>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         (int)LS_SMEM_LIMIT));
        if (c->device >= 0 && c->device < kMaxDevices) attr_done[c->device] = true;
    }
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(C, 1, 1);
    cfg.blockDim = dim3(LS_THREADS, 1, 1);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = s;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = C;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = C > 1 ? 1 : 0;
    ACCBPG_CUDA(cudaLaunchKernelEx(&cfg, linreg_bpg_small_kernel<C>, p));
    return ACCBPG_OK;
}

}  // namespace accbpg

using namespace accbpg;

extern "C" {

size_t accbpg_linreg_bpg_small_smem_bytes(int64_t m, int64_t n) {
    size_t bytes = 0;
    return ls_pick_cluster(m, n, &bytes) ? bytes : 0;
}

int accbpg_linreg_bpg_small(void* ctx, void* stream, int kind, const double* A, int64_t m, int64_t n, int64_t lda,
                            const double* b, int hkind, double lamda, double delta, double* x, double L,
                            double ls_ratio, int linesearch, int maxitrs, double epsilon, double* F_out,
                            double* Ls_out, double* T_out, double* info_out) {
    Ctx* c = (Ctx*)ctx;
    cudaStream_t s = (cudaStream_t)stream;
    if (!c || !A || !b || !x || !F_out || !Ls_out || !T_out || !info_out) return arg_err("linreg_bpg_small: NULL pointer");
    ACCBPG_ON_DEVICE(c);
    if (kind != ACCBPG_LINREG_POISSON && kind != ACCBPG_LINREG_KL) return arg_err("linreg kind");
    if (hkind < ACCBPG_SMALL_H_BURG || hkind > ACCBPG_SMALL_H_SHANNON_SIMPLEX) return arg_err("linreg_bpg_small: hkind");
    size_t smem = 0;
    const int C = ls_pick_cluster(m, n, &smem);
    if (C == 0 || lda < n)
        return arg_err("linreg_bpg_small: shape does not fit a cluster's shared memory (accbpg_linreg_bpg_small_smem_bytes)");
    if (!(L > 0.0) || !(ls_ratio > 1.0) || maxitrs < 1) return arg_err("linreg_bpg_small: L, ls_ratio, maxitrs");
    LsParams p;
    p.A = A; p.b = b; p.m = (int)m; p.n = (int)n; p.lda = lda; p.kind = kind; p.hkind = hkind;
    p.lamda = lamda; p.delta = delta; p.x = x; p.L = L; p.ls_ratio = ls_ratio; p.epsilon = epsilon;
    p.linesearch = linesearch; p.maxitrs = maxitrs; p.F = F_out; p.Ls = Ls_out; p.T = T_out; p.info = info_out;
    p.status = c->d_status;
    int rc = C == 8 ? ls_launch<8>(c, s, p, smem) : C == 4 ? ls_launch<4>(c, s, p, smem)
           : C == 2 ? ls_launch<2>(c, s, p, smem) : ls_launch<1>(c, s, p, smem);
    if (rc) return rc;
    ACCBPG_LAUNCHED("linreg_bpg_small_kernel");
    return ACCBPG_OK;
}

}  // extern "C"
