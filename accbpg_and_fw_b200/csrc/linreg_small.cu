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
//
// linreg_abpg_small_kernel<C, DRV> runs ABPG (algorithms.py:94-180) or ABPG_gain (:295-420) the same way, in a plan of
// its own (x-, z-, z, x, g per column slice; b, A x-, A z-, A y, A z, A x, r replicated).  It follows the operator
// loop's carried-image scheme: A y and A x are combinations of the carried A x- and A z-, A z is the one matvec of a
// trip, A x is re-formed from x every reanchor_every iterations.  A trip is one exchange (two with the simplex kernel's
// normaliser) carrying A z and the n-sums of D(x, y), D(z, z-), dot(g, x - y), Psi(x) and the restart dot.
// On a B200 at a 1000 W power limit (profiles/linreg_small_accel_r01.json): ABPG 117 k it/s on Poisson 200 x 100 and
// 89 k on KL 1000 x 100, ABPG_gain 51 k and 39 k, 10-16x the operator-by-operator loop (DESIGN.md section 9).
#include <cooperative_groups.h>

#include "common.cuh"

namespace accbpg {

constexpr int LS_THREADS = 512;
constexpr int LS_WARPS = LS_THREADS / 32;
constexpr size_t LS_SMEM_LIMIT = 227 * 1024;       // the shared memory an sm_100 CTA may have (the kernel has no static)
// scalars in an exchange.  BPG: dot(g, x1 - x), D(x1, x), sum x, sum x1, x1.x1, status.  ABPG: dot(g, x - y), D(x, y),
// sum y, sum x, x.x, status, D(z, z-), sum z-, sum z, dot(g, x - x-) (the restart test)
constexpr int LS_NSC = 10;
enum { SC_DOT = 0, SC_DIV, SC_SY, SC_SX, SC_SQ, SC_ST, SC_DZZ, SC_SZ1, SC_SZ, SC_RDOT };

struct LsPlan {
    int NL, ldn;                  // columns per CTA, row pitch of the shared copy of A (odd: conflict-free column walks)
    size_t xstride;               // one exchange buffer: LS_NSC scalars + an m-vector
    size_t off_A, off_b, off_Ax, off_Ax1, off_r, off_xch, off_x, off_x1, off_g, off_scr, off_red, off_st, off_xsc, bytes;
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
    p.off_xsc = o; o += (size_t)LS_NSC * 8;         // the scalars of the last exchange, summed over the cluster
    p.bytes = o;
    return p;
}

// The accelerated drivers' plan: the slices x-, z-, z, x, g and the replicated m-vectors b, A x-, A z-, A y, A z, A x, r
struct LaPlan {
    int NL, ldn;
    size_t off_A, off_b, off_Ax1, off_Az1, off_Ay, off_Az, off_Ax, off_r, off_xch, off_x1, off_z1, off_z, off_x, off_g,
        off_scr, off_red, off_st, off_xsc, bytes;
};

__host__ __device__ inline LaPlan la_plan(int64_t m, int64_t n, int C) {
    LaPlan p;
    p.NL = (int)((n + C - 1) / C);
    p.ldn = p.NL | 1;
    size_t o = 0;
    p.off_A = o;   o += (size_t)m * p.ldn * 8;
    p.off_b = o;   o += (size_t)m * 8;
    p.off_Ax1 = o; o += (size_t)m * 8;
    p.off_Az1 = o; o += (size_t)m * 8;
    p.off_Ay = o;  o += (size_t)m * 8;
    p.off_Az = o;  o += (size_t)m * 8;
    p.off_Ax = o;  o += (size_t)m * 8;
    p.off_r = o;   o += (size_t)m * 8;
    p.off_xch = o; o += 2 * ((size_t)LS_NSC + (size_t)m) * 8;
    p.off_x1 = o;  o += (size_t)p.NL * 8;
    p.off_z1 = o;  o += (size_t)p.NL * 8;
    p.off_z = o;   o += (size_t)p.NL * 8;
    p.off_x = o;   o += (size_t)p.NL * 8;
    p.off_g = o;   o += (size_t)p.NL * 8;
    p.off_scr = o; o += (size_t)LS_THREADS * 8;
    p.off_red = o; o += (size_t)2 * LS_NSC * LS_WARPS * 8;
    p.off_st = o;  o += 16;
    p.off_xsc = o; o += (size_t)LS_NSC * 8;
    p.bytes = o;
    return p;
}

// smallest cluster whose plan fits; 0 when none of <= 8 CTAs does
template <class Plan>
static int ls_pick_cluster(int64_t m, int64_t n, size_t* bytes, Plan (*plan)(int64_t, int64_t, int)) {
    if (m < 1 || n < 1 || m > (1 << 20) || n > (1 << 20)) return 0;
    for (int C = 1; C <= 8; C *= 2) {
        const Plan pl = plan(m, n, C);
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
    double *Ax, *Ax1, *r, *xch, *xsc, *x, *x1, *g, *scr, *red;
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
    if (c.tid < LS_NSC) {                               // one thread per scalar; the others read it after the barrier
        const int q = c.tid;
        if (q == SC_ST) {
            uint32_t st = 0;
#pragma unroll
            for (int r = 0; r < C; ++r) st |= (uint32_t)ls_ld_cluster(src[r] + 8 * q);
            c.xsc[q] = (double)st;
        } else {
            double a = ls_ld_cluster(src[0] + 8 * q);
#pragma unroll
            for (int r = 1; r < C; ++r) a += ls_ld_cluster(src[r] + 8 * q);
            c.xsc[q] = a;
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
#pragma unroll
    for (int q = 0; q < LS_NSC; ++q) sc[q] = c.xsc[q];
}

// ---- out = h.div_prox_map(ctr, g, L) on this CTA's columns (BurgProxF / shannon_point / ShannonProxSumF +
//      DivideBySlotF in vecops.cu: same formulas, checks and status bits).  Returns this thread's status bits; the
//      simplex normaliser is summed over all n through one exchange of its own.
template <int C>
__device__ __forceinline__ uint32_t ls_step(LsCtx& c, const LsParams& p, const double* ctr, const double* g, double L,
                                            double* out) {
    const int hk = p.hkind;
    const double lamda = p.lamda;
    uint32_t st = 0;
    if (hk == ACCBPG_SMALL_H_SHANNON_SIMPLEX) {
        // y exp(-g/L), normalised by its sum over all n
        double s[1] = {0.0};
        for (int j = c.tid; j < c.nloc; j += LS_THREADS) {
            const double yj = ctr[j];
            if (!(yj > 0.0)) st |= ACCBPG_ST_Y_NOT_POS;
            const double v = yj * exp(-g[j] / L);
            out[j] = v;
            s[0] += v;
        }
        ls_cta_sum<1>(c, s);
        double t[LS_NSC] = {s[0]};
        ls_exchange<C>(c, t, 0, nullptr);
        for (int j = c.tid; j < c.nloc; j += LS_THREADS) out[j] = out[j] / t[0];
        return st;
    }
    const bool burg = hk <= ACCBPG_SMALL_H_BURG_L2;
    const double lamL = lamda / L, four_lamL = 4 * lamL, two_lamL = 2 * lamL;
    for (int j = c.tid; j < c.nloc; j += LS_THREADS) {
        const double yj = ctr[j];
        double gj = g[j], v;
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
        out[j] = v;
    }
    return st;
}

// ---- one element of D(x, y): burg_divergence adds (r - log r) - 1 to div; shannon_divergence adds x log((x+d)/(y+d))
//      to div and y to sy (its sum x term is the caller's)
__device__ __forceinline__ void ls_div_elem(bool burg, double delta, double xj, double yj, double& div, double& sy,
                                            uint32_t& st) {
    if (burg) {
        if (!(xj > 0.0) || !(yj > 0.0)) st |= ACCBPG_ST_ARG_NOT_POS;
        const double r = xj / yj;
        div += (r - log(r)) - 1.0;
    } else {
        if (!(xj >= 0.0) || !(yj >= 0.0)) st |= ACCBPG_ST_ARG_NEGATIVE;
        div += xj * log((xj + delta) / (yj + delta));
        sy += yj;
    }
}

// D(x, y) from its exchanged sums (the Shannon kernels add sum y - sum x)
__device__ __forceinline__ double ls_div(const LsParams& p, double div, double sy, double sx) {
    return p.hkind <= ACCBPG_SMALL_H_BURG_L2 ? div : div + (sy - sx);
}

// ---- BPG trial: x1 = h.div_prox_map(x, g, L) and the partial n-sums dot(g, x1 - x) (vec_dot_diff), D(x1, x),
//      sum x1 and x1.x1 (Psi of x1)
template <int C>
__device__ __forceinline__ void ls_prox(LsCtx& c, const LsParams& p, double L, bool with_div, double (&sc)[LS_NSC]) {
    const bool burg = p.hkind <= ACCBPG_SMALL_H_BURG_L2;
    uint32_t st = ls_step<C>(c, p, c.x, c.g, L, c.x1);
    double a[5] = {0.0, 0.0, 0.0, 0.0, 0.0};
    for (int j = c.tid; j < c.nloc; j += LS_THREADS) {
        const double xj = c.x1[j], yj = c.x[j];
        if (with_div) {
            a[SC_DOT] += c.g[j] * (xj - yj);
            ls_div_elem(burg, p.delta, xj, yj, a[SC_DIV], a[SC_SY], st);
        }
        a[SC_SX] += xj;
        a[SC_SQ] += xj * xj;
    }
    ls_flag(c, st);
    ls_cta_sum<5>(c, a);                                // (its barrier also publishes x1 and the status word)
#pragma unroll
    for (int q = 0; q < LS_NSC; ++q) sc[q] = q < 5 ? a[q] : 0.0;
    sc[SC_ST] = (double)*c.st;
}

// Psi(x) from the exchanged sums, in the operator path's rounding order (BurgEntropyL1 / ShannonEntropyL1: lamda * sum x;
// BurgEntropyL2: (lamda / 2) * x.x)
__device__ __forceinline__ double ls_psi(const LsParams& p, const double (&sc)[LS_NSC]) {
    if (p.hkind == ACCBPG_SMALL_H_BURG_L1 || p.hkind == ACCBPG_SMALL_H_SHANNON_L1) return p.lamda * sc[SC_SX];
    if (p.hkind == ACCBPG_SMALL_H_BURG_L2) return (p.lamda / 2) * sc[SC_SQ];
    return 0.0;
}

// ---- rank, column slice and the split of the matrix passes, for NL columns per CTA (the buffers are the caller's)
template <int C>
__device__ __forceinline__ void ls_split(LsCtx& c, const LsParams& p, int NL) {
    namespace cg = cooperative_groups;
    c.m = p.m;
    c.rank = (C > 1) ? (int)cg::this_cluster().block_rank() : 0;
    c.col0 = c.rank * NL;
    c.nloc = max(0, min(NL, p.n - c.col0));
    c.tid = threadIdx.x; c.lane = c.tid & 31; c.warp = c.tid >> 5;
    c.qmv = (p.m < LS_THREADS) ? max(1, min(LS_THREADS / p.m, c.nloc)) : 1;
    c.cwmv = (c.nloc + c.qmv - 1) / c.qmv;
    c.qrm = (c.nloc > 0 && c.nloc < LS_THREADS) ? max(1, min(LS_THREADS / c.nloc, p.m)) : 1;
    c.rwrm = (p.m + c.qrm - 1) / c.qrm;
    c.par = 0; c.flip = 0;
}

// ---- this CTA's columns of A, b and this CTA's slice of x0 into x; then A x0 into Ax (every CTA) and sum x0, x0.x0
//      into sc[SC_SX], sc[SC_SQ] (Psi(x0))
template <int C>
__device__ __forceinline__ void ls_start(LsCtx& c, const LsParams& p, double* x, double* Ax, double (&sc)[LS_NSC]) {
    if (c.tid == 0) *c.st = 0u;
    {
        double* As = const_cast<double*>(c.A);
        double* bs = const_cast<double*>(c.b);
        const int total = p.m * c.nloc;
        for (int e = c.tid; e < total; e += LS_THREADS) {
            const int i = e / c.nloc, j = e - i * c.nloc;
            As[(size_t)i * c.ldn + j] = p.A[(int64_t)i * p.lda + c.col0 + j];
        }
        for (int i = c.tid; i < p.m; i += LS_THREADS) bs[i] = p.b[i];
        for (int j = c.tid; j < c.nloc; j += LS_THREADS) x[j] = p.x[c.col0 + j];
    }
    __syncthreads();
    double a[2] = {0.0, 0.0};
    for (int j = c.tid; j < c.nloc; j += LS_THREADS) { a[0] += x[j]; a[1] += x[j] * x[j]; }
    ls_cta_sum<2>(c, a);
    ls_matvec(c, x, ls_part(c));
    for (int q = 0; q < LS_NSC; ++q) sc[q] = 0.0;
    sc[SC_SX] = a[0]; sc[SC_SQ] = a[1];
    ls_exchange<C>(c, sc, p.m, Ax);
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
    c.red = (double*)(ls_raw + pl.off_red);     c.xsc = (double*)(ls_raw + pl.off_xsc);
    c.ldn = pl.ldn;
    c.st = (uint32_t*)(ls_raw + pl.off_st);
    ls_split<C>(c, p, pl.NL);
    const bool writer = c.rank == 0 && c.tid == 0;

    // A x0 and Psi(x0)
    double sc[LS_NSC];
    ls_start<C>(c, p, c.x, c.Ax, sc);
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
            const double D = ls_div(p, sc[SC_DIV], sc[SC_SY], sc[SC_SX]);
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

// ---- ABPG / ABPG_gain (algorithms.py:94-180, :295-420) -------------------------------------------------------------

struct LaParams : LsParams {
    double gamma, G0, ls_inc, ls_dec;
    int theta_eq, restart, rule, checkdiv, reanchor;
    double* hist;                    // rows of maxitrs: F, G / Gain, Gdiv, theta, D(x,y), D(z,z-), T
    // info: [0] entries written, [1] trips, [2] cluster size, [3] Gdr unbound, [4] last G / gain
};

// Every iteration of the operator loop's default scheme (config.linear_images): the images A x- and A z- are carried,
// A y and A x are combinations of them, A z is one matvec per trip and A x is re-formed from x every reanchor
// iterations.  y, x, 1 - theta and the prox are the operator path's elementwise expressions, so only sums differ.
// Each trip is one exchange (two for the simplex kernel's normaliser); the scalar control runs in every thread.
template <int C, int DRV>
__global__ void __launch_bounds__(LS_THREADS, 1) linreg_abpg_small_kernel(LaParams p) {
    extern __shared__ __align__(16) unsigned char ls_raw[];
    namespace cg = cooperative_groups;
    constexpr bool GAIN = DRV == ACCBPG_SMALL_DRV_ABPG_GAIN;
    const unsigned long long ns0 = ls_clock();
    const LaPlan pl = la_plan(p.m, p.n, C);
    LsCtx c;
    c.A = (const double*)(ls_raw + pl.off_A);
    c.b = (const double*)(ls_raw + pl.off_b);
    c.r = (double*)(ls_raw + pl.off_r);     c.xch = (double*)(ls_raw + pl.off_xch);
    c.g = (double*)(ls_raw + pl.off_g);     c.scr = (double*)(ls_raw + pl.off_scr);
    c.red = (double*)(ls_raw + pl.off_red);     c.xsc = (double*)(ls_raw + pl.off_xsc);
    c.x = c.x1 = c.Ax = c.Ax1 = nullptr;
    c.ldn = pl.ldn;
    c.st = (uint32_t*)(ls_raw + pl.off_st);
    ls_split<C>(c, p, pl.NL);
    const bool writer = c.rank == 0 && c.tid == 0;
    double* X1 = (double*)(ls_raw + pl.off_x1);   double* Z1 = (double*)(ls_raw + pl.off_z1);
    double* Z = (double*)(ls_raw + pl.off_z);     double* X = (double*)(ls_raw + pl.off_x);
    double* Ax1 = (double*)(ls_raw + pl.off_Ax1); double* Az1 = (double*)(ls_raw + pl.off_Az1);
    double* Ay = (double*)(ls_raw + pl.off_Ay);
    double* Az = (double*)(ls_raw + pl.off_Az);   double* Ax = (double*)(ls_raw + pl.off_Ax);
    const int M = p.maxitrs;
    auto hist = [&](int row, int k) -> double& { return p.hist[(size_t)row * M + k]; };   // rows: see LaParams
    const bool burg = p.hkind <= ACCBPG_SMALL_H_BURG_L2;
    const double gamma = p.gamma, L = p.L;

    // x0, z0 = x0, A x0 = A z0, Psi(x0)
    double sc[LS_NSC];
    ls_start<C>(c, p, X1, Ax1, sc);
    for (int j = c.tid; j < c.nloc; j += LS_THREADS) Z1[j] = X1[j];
    for (int i = c.tid; i < p.m; i += LS_THREADS) Az1[i] = Ax1[i];
    double psi_x = ls_psi(p, sc);

    double theta = 1.0, G = p.G0, gdr = 0.0, fx_carry = 0.0, Fprev = 0.0, dxy = 0.0, dzz = 0.0;
    bool have_fx = false, gdr_bound = false;
    int kk = 0, k = 0, trips = 0, unbound = 0;
    uint32_t st_all = 0;
    for (; k < M; ++k) {
        if (writer) hist(6, k) = (double)(ls_clock() - ns0);
        // F[k] = f(x_k) + Psi(x_k): from the carried A x_k, or the value the last trip of ABPG_gain formed at it
        const double fx = (GAIN && have_fx) ? fx_carry : ls_value(c, p.kind, Ax1, nullptr);
        const double Fk = fx + psi_x;
        if (writer) hist(0, k) = Fk;
        const double G_1 = G, theta_1 = theta;
        if (GAIN) G = G / p.ls_dec;
        else theta = (p.theta_eq && kk > 0) ? la_solve_theta(theta, gamma, 1.0) : gamma / (kk + gamma);
        for (;;) {
            ++trips;
            if (GAIN && kk > 0) {
                if (p.theta_eq) {
                    theta = la_solve_theta(theta_1, gamma, G / G_1);
                } else {
                    const double alpha = G / G_1;                                     // algorithms.py:367
                    theta = theta_1 * ((1 + alpha * (gamma - 1)) / (gamma * alpha + theta_1));
                }
            }
            const double omt = 1 - theta, tg = la_pow(theta, gamma), tg1 = la_pow(theta, gamma - 1);
            // y = (1-theta) x- + theta z-: its image, f(y), r(A y) and g = A^T r
            for (int i = c.tid; i < p.m; i += LS_THREADS) Ay[i] = omt * Ax1[i] + theta * Az1[i];
            const double fy = ls_value(c, p.kind, Ay, c.r);
            ls_rmatvec(c);
            const double Lz = GAIN ? tg1 * G * L : tg1 * L;
            uint32_t st = ls_step<C>(c, p, Z1, c.g, Lz, Z);
            // x = (1-theta) x- + theta z and the trip's partial n-sums
            double a[LS_NSC] = {};
            for (int j = c.tid; j < c.nloc; j += LS_THREADS) {
                const double x1j = X1[j], z1j = Z1[j], zj = Z[j], gj = c.g[j];
                const double yj = omt * x1j + theta * z1j;
                const double xj = omt * x1j + theta * zj;
                X[j] = xj;
                a[SC_DOT] += gj * (xj - yj);
                ls_div_elem(burg, p.delta, xj, yj, a[SC_DIV], a[SC_SY], st);
                a[SC_SX] += xj;
                a[SC_SQ] += xj * xj;
                a[SC_RDOT] += gj * (xj - x1j);
            }
            for (int j = c.tid; j < c.nloc; j += LS_THREADS) {
                const double zj = Z[j];
                ls_div_elem(burg, p.delta, zj, Z1[j], a[SC_DZZ], a[SC_SZ1], st);
                a[SC_SZ] += zj;
            }
            ls_flag(c, st);
            ls_cta_sum<LS_NSC>(c, a);                   // (its barrier also publishes z, x and the status word)
#pragma unroll
            for (int q = 0; q < LS_NSC; ++q) sc[q] = a[q];
            sc[SC_ST] = (double)*c.st;
            ls_matvec(c, Z, ls_part(c));
            ls_exchange<C>(c, sc, p.m, Az);
            st_all = (uint32_t)sc[SC_ST];
            if (st_all) break;
            for (int i = c.tid; i < p.m; i += LS_THREADS) Ax[i] = omt * Ax1[i] + theta * Az[i];
            dxy = ls_div(p, sc[SC_DIV], sc[SC_SY], sc[SC_SX]);
            dzz = ls_div(p, sc[SC_DZZ], sc[SC_SZ1], sc[SC_SZ]);
            if (!GAIN) { gdr = dxy / dzz / tg; break; }
            if (dzz < p.epsilon) break;                 // Gdr keeps its previous value, as in the reference
            gdr = dxy / dzz / tg;
            gdr_bound = true;
            bool again;
            if (p.checkdiv) {
                again = gdr > G;
            } else {
                fx_carry = ls_value(c, p.kind, Ax, nullptr);
                again = fx_carry > fy + sc[SC_DOT] + tg * G * L * dzz;   // algorithms.py:387
            }
            if (!again) break;
            G = G * p.ls_inc;
        }
        if (st_all) { ++k; break; }
        if (GAIN && !gdr_bound) { unbound = 1; break; }  // the reference's Gdiv[k] = Gdr raises UnboundLocalError
        have_fx = GAIN && !p.checkdiv;
        if ((k + 1) % p.reanchor == 0) {                // A x from x itself; F[k+1] from the fresh image
            double t[LS_NSC] = {};
            ls_matvec(c, X, ls_part(c));
            ls_exchange<C>(c, t, p.m, Ax);
            have_fx = false;
        }
        if (writer) {
            hist(1, k) = GAIN ? G : gdr;
            if (GAIN) hist(2, k) = gdr;
            hist(3, k) = theta; hist(4, k) = dxy; hist(5, k) = dzz;
        }
        ++kk;
        // restart (algorithms.py:168, :406): ABPG only from k = 1; ABPG_gain's rule 'f' at k = 0 compares F[0] with
        // F[-1], the reference's still-zero last slot
        if (p.restart && (GAIN || k > 0)) {
            bool rs = false;
            if (p.rule == ACCBPG_SMALL_RESTART_F) rs = Fk > (k > 0 ? Fprev : (M == 1 ? Fk : 0.0));
            else if (p.rule == ACCBPG_SMALL_RESTART_G) rs = sc[SC_RDOT] > 0;
            if (rs) {
                theta = 1.0;
                kk = 0;
                for (int j = c.tid; j < c.nloc; j += LS_THREADS) Z[j] = X[j];
                for (int i = c.tid; i < p.m; i += LS_THREADS) Az[i] = Ax[i];
            }
        }
        Fprev = Fk;
        psi_x = ls_psi(p, sc);
        double* t = X1; X1 = X; X = t;
        t = Z1; Z1 = Z; Z = t;
        t = Ax1; Ax1 = Ax; Ax = t;
        t = Az1; Az1 = Az; Az = t;
        if (dzz < p.epsilon) { ++k; break; }
    }
    if (C > 1) cg::this_cluster().sync();               // nobody leaves while its shared memory may still be read
    for (int j = c.tid; j < c.nloc; j += LS_THREADS) p.x[c.col0 + j] = X1[j];
    if (c.tid == 0 && *c.st) atomicOr(p.status, *c.st);
    if (writer) {
        p.info[0] = (double)k; p.info[1] = (double)trips; p.info[2] = (double)C; p.info[3] = (double)unbound;
        p.info[4] = GAIN ? G : gdr;
    }
}

template <auto KERNEL, class P>
static int ls_launch(Ctx* c, cudaStream_t s, const P& p, int C, size_t smem) {
    static bool attr_done[kMaxDevices] = {};
    if (!(c->device >= 0 && c->device < kMaxDevices && attr_done[c->device])) {
        ACCBPG_CUDA(cudaFuncSetAttribute(KERNEL, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)LS_SMEM_LIMIT));
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
    ACCBPG_CUDA(cudaLaunchKernelEx(&cfg, KERNEL, p));
    return ACCBPG_OK;
}

template <int DRV>
static int la_launch(Ctx* c, cudaStream_t s, const LaParams& p, int C, size_t smem) {
    return C == 8 ? ls_launch<linreg_abpg_small_kernel<8, DRV>>(c, s, p, C, smem)
         : C == 4 ? ls_launch<linreg_abpg_small_kernel<4, DRV>>(c, s, p, C, smem)
         : C == 2 ? ls_launch<linreg_abpg_small_kernel<2, DRV>>(c, s, p, C, smem)
                  : ls_launch<linreg_abpg_small_kernel<1, DRV>>(c, s, p, C, smem);
}

}  // namespace accbpg

using namespace accbpg;

extern "C" {

size_t accbpg_linreg_bpg_small_smem_bytes(int64_t m, int64_t n) {
    size_t bytes = 0;
    return ls_pick_cluster(m, n, &bytes, ls_plan) ? bytes : 0;
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
    const int C = ls_pick_cluster(m, n, &smem, ls_plan);
    if (C == 0 || lda < n)
        return arg_err("linreg_bpg_small: shape does not fit a cluster's shared memory (accbpg_linreg_bpg_small_smem_bytes)");
    if (!(L > 0.0) || !(ls_ratio > 1.0) || maxitrs < 1) return arg_err("linreg_bpg_small: L, ls_ratio, maxitrs");
    LsParams p;
    p.A = A; p.b = b; p.m = (int)m; p.n = (int)n; p.lda = lda; p.kind = kind; p.hkind = hkind;
    p.lamda = lamda; p.delta = delta; p.x = x; p.L = L; p.ls_ratio = ls_ratio; p.epsilon = epsilon;
    p.linesearch = linesearch; p.maxitrs = maxitrs; p.F = F_out; p.Ls = Ls_out; p.T = T_out; p.info = info_out;
    p.status = c->d_status;
    int rc = C == 8 ? ls_launch<linreg_bpg_small_kernel<8>>(c, s, p, C, smem)
           : C == 4 ? ls_launch<linreg_bpg_small_kernel<4>>(c, s, p, C, smem)
           : C == 2 ? ls_launch<linreg_bpg_small_kernel<2>>(c, s, p, C, smem)
                    : ls_launch<linreg_bpg_small_kernel<1>>(c, s, p, C, smem);
    if (rc) return rc;
    ACCBPG_LAUNCHED("linreg_bpg_small_kernel");
    return ACCBPG_OK;
}

size_t accbpg_linreg_abpg_small_smem_bytes(int64_t m, int64_t n) {
    size_t bytes = 0;
    return ls_pick_cluster(m, n, &bytes, la_plan) ? bytes : 0;
}

int accbpg_linreg_abpg_small(void* ctx, void* stream, int driver, int kind, const double* A, int64_t m, int64_t n,
                             int64_t lda, const double* b, int hkind, double lamda, double delta, double* x, double L,
                             double gamma, int maxitrs, double epsilon, int theta_eq, int restart, int restart_rule,
                             double G0, double ls_inc, double ls_dec, int checkdiv, int reanchor_every, double* hist,
                             double* info_out) {
    Ctx* c = (Ctx*)ctx;
    cudaStream_t s = (cudaStream_t)stream;
    if (!c || !A || !b || !x || !hist || !info_out) return arg_err("linreg_abpg_small: NULL pointer");
    ACCBPG_ON_DEVICE(c);
    if (driver != ACCBPG_SMALL_DRV_ABPG && driver != ACCBPG_SMALL_DRV_ABPG_GAIN) return arg_err("linreg_abpg_small: driver");
    if (kind != ACCBPG_LINREG_POISSON && kind != ACCBPG_LINREG_KL) return arg_err("linreg kind");
    if (hkind < ACCBPG_SMALL_H_BURG || hkind > ACCBPG_SMALL_H_SHANNON_SIMPLEX) return arg_err("linreg_abpg_small: hkind");
    size_t smem = 0;
    const int C = ls_pick_cluster(m, n, &smem, la_plan);
    if (C == 0 || lda < n)
        return arg_err("linreg_abpg_small: shape does not fit a cluster's shared memory "
                       "(accbpg_linreg_abpg_small_smem_bytes)");
    auto pos = [](double v) { return isfinite(v) && v > 0.0; };
    if (!pos(L) || !pos(gamma) || !pos(G0) || !pos(ls_inc) || !pos(ls_dec))
        return arg_err("linreg_abpg_small: L, gamma, G0, ls_inc, ls_dec must be finite and > 0");
    if (maxitrs < 1 || reanchor_every < 1 || restart_rule < ACCBPG_SMALL_RESTART_NONE ||
        restart_rule > ACCBPG_SMALL_RESTART_G)
        return arg_err("linreg_abpg_small: maxitrs, reanchor_every, restart_rule");
    LaParams p = {};
    p.A = A; p.b = b; p.m = (int)m; p.n = (int)n; p.lda = lda; p.kind = kind; p.hkind = hkind;
    p.lamda = lamda; p.delta = delta; p.x = x; p.L = L; p.epsilon = epsilon; p.maxitrs = maxitrs;
    p.info = info_out; p.status = c->d_status;
    p.gamma = gamma; p.G0 = G0; p.ls_inc = ls_inc; p.ls_dec = ls_dec;
    p.theta_eq = theta_eq != 0; p.restart = restart != 0; p.rule = restart_rule; p.checkdiv = checkdiv != 0;
    p.reanchor = reanchor_every; p.hist = hist;
    int rc = driver == ACCBPG_SMALL_DRV_ABPG_GAIN ? la_launch<ACCBPG_SMALL_DRV_ABPG_GAIN>(c, s, p, C, smem)
                                                  : la_launch<ACCBPG_SMALL_DRV_ABPG>(c, s, p, C, smem);
    if (rc) return rc;
    ACCBPG_LAUNCHED("linreg_abpg_small_kernel");
    return ACCBPG_OK;
}

}  // extern "C"
