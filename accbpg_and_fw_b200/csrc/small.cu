// Small-shape D-optimal design: the WHOLE BPG loop (algorithms.py:11-72) in one CTA.
//
// At BASELINE.json configs[0] (D_opt_design(80, 200)) an iteration of the operator-by-operator path is ~12 launches and
// one host decision per line-search trip (~300 us); the arithmetic is ~25 us of one SM.  When H (m x n doubles) fits in
// shared memory next to the m x m factor, one persistent CTA of 16 warps runs every iteration of
//     BPG(DOptimalObj(H), BurgEntropySimplex(eps), L, x0, maxitrs, epsilon, linesearch, ls_ratio)
// on the device: same control flow, same stopping test, F_k and L_k written to history arrays, one launch per solve.
//
//   Gram      M = H diag(x) H^T      FP64 DMMA (m8n8k4), 16 x 16 block of the lower triangle per warp, operands from the
//                                    shared-memory copy of H                                  (functions.py:43-47)
//   factor    M = Lt D Lt^T          right-looking, one CTA barrier per column, pivot reciprocal taken one column ahead
//                                    by the thread that produces the pivot; f = -sum log d_j    (functions.py:48-51)
//   gradient  g_j = -sum_i (Lt^-1 h_j)_i^2 / d_i      blocked forward substitution IN PLACE on the shared-memory copy of H
//                                    (a warp owns 8 columns and walks the 8-row blocks: DMMA products with the rows already
//                                    solved, then the inverse of the 8 x 8 unit diagonal block); the copy of H is then
//                                    refilled from global memory (L2) by cp.async under the prox   (functions.py:52-58)
//   prox      Burg-simplex root-find (functions.py:341-356) with the CTA-wide sums of a Newton step in one barrier
//   test      f(x+) > f(x) + <g, x+ - x> + L D(x+, x)  ->  L *= ls_ratio                      (algorithms.py:46-56)
//
// dopt_abpg_small_kernel<C, DRV> runs ABPG (algorithms.py:94-180) or ABPG_gain (:295-420) on the same functions, in a
// plan with three more vectors, evaluating every point from scratch (see the kernel).  On a B200 at a 1000 W power
// limit (profiles/dopt_small_accel_r01.json): ABPG 20.8 k it/s and ABPG_gain 9.6 k it/s at 80 x 200, 2.6x and 4.0x the
// operator-by-operator loop (DESIGN.md section 9).
#include <cooperative_groups.h>

#include "dmma.cuh"

namespace accbpg {

constexpr int SM_THREADS = 512;
constexpr int SM_WARPS = SM_THREADS / 32;
constexpr int SM_MAX_M = 128;
constexpr int SM_SMEM_LIMIT = 220 * 1024;
constexpr int SM_ACC_SUMS = 5;                 // values of dopt_abpg_small_kernel's CTA-wide sum of a trip
#define kInf (__longlong_as_double(0x7ff0000000000000LL))

struct SmallPlan {
    int MP, NP, NL, ldn, lda, nblk16;
    size_t off_H, off_A, off_part, off_x, off_x1, off_g, off_d, off_rinv, off_cp, off_xd, off_red, off_acc, bytes;
};

// C = CTAs of the cluster: CTA r holds columns [r NL, (r + 1) NL) of H (NL a multiple of 8); vectors are replicated.
// acc: the plan of dopt_abpg_small_kernel, which appends three more vectors and the buffers of its wider CTA-wide sum.
__host__ __device__ inline SmallPlan small_plan(int m, int n, int C, bool acc = false) {
    SmallPlan p;
    p.MP = (m + 15) / 16 * 16;
    p.NL = ((n + C - 1) / C + 7) / 8 * 8;
    p.NP = p.NL * C;                  // vectors are padded to the cluster's column range (>= n)
    p.ldn = p.NL + 4;                 // = 4 mod 8: DMMA fragment reads (8 rows x 4 consecutive doubles) hit every bank pair once
    p.lda = p.MP + 4;
    p.nblk16 = (p.MP / 16) * (p.MP / 16 + 1) / 2;
    size_t o = 0;
    p.off_H = o;    o += (size_t)p.MP * p.ldn * 8;
    p.off_A = o;    o += (size_t)p.MP * p.lda * 8;
    p.off_part = o; o += (C > 1) ? (size_t)2 * p.nblk16 * 256 * 8 : 0;   // this CTA's partial Gram blocks, double buffered
    p.off_x = o;    o += (size_t)p.NP * 8;
    p.off_x1 = o;   o += (size_t)p.NP * 8;
    p.off_g = o;    o += (size_t)p.NP * 8;
    p.off_d = o;    o += (size_t)p.MP * 8;
    p.off_rinv = o; o += (size_t)p.MP * 8;
    p.off_cp = o;   o += (size_t)p.MP * 12 * 8;        // the unscaled panel of the factorisation, rows of 12 doubles
    p.off_xd = o;   o += (size_t)p.MP * 12 * 8;        // inverses of the 8 x 8 unit diagonal blocks, rows of 12 doubles
    p.off_red = o;  o += 256 * 8;                      // [0,128) CTA-wide reductions, [128,192) the prox group's
    p.off_acc = o;  o += acc ? (size_t)3 * p.NP * 8 + (size_t)2 * SM_ACC_SUMS * SM_WARPS * 8 : 0;
    p.bytes = o;
    return p;
}

struct SmallParams {
    const double* H; int m, n; int64_t ldh;
    double* x;                       // in: x0, out: the last iterate
    double L, ls_ratio, epsilon, eps_prox;
    int linesearch, maxitrs;
    double* F; double* Ls;           // histories, maxitrs entries each
    double* info;                    // [0] entries written (k + 1), [1] line-search trials, [2] last L, [3] Newton steps in total, [4..9] clocks per phase
    uint32_t* status;
};

struct SmallCtx {
    double *Hs, *A, *part, *xs, *x1s, *gs, *dv, *rinv, *Cp, *Xd, *red;
    int m, n, MP, NP, ldn, lda;
    int C, rank, NL, col0, nloc, nblk16, gcount;     // cluster size / rank, local column slice [col0, col0 + nloc), Gram calls so far
    int tid, lane, warp, g, t;
    int flip;
    long long tf0, tf1, tf2, tf3;        // clocks inside the factorisation: diagonal tile, its inverse, panel, trailing update
};

// ---- CTA-wide sums of two values with ONE barrier: warps leave partials in alternating buffers ([a of warp 0..15,
//      b of warp 0..15]), then EVERY warp adds them with one load and a 4-step butterfly inside each half warp (fixed
//      order: bit-reproducible, identical in every warp) and broadcasts the two totals
__device__ __forceinline__ void cta_sum2(SmallCtx& c, double& a, double& b) {
    a = warp_sum(a);
    b = warp_sum(b);
    double* s = c.red + c.flip * 64;
    c.flip ^= 1;
    if (c.lane == 0) { s[c.warp] = a; s[SM_WARPS + c.warp] = b; }
    __syncthreads();
    double v = s[c.lane];
#pragma unroll
    for (int o = SM_WARPS / 2; o >= 1; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    a = __shfl_sync(0xffffffffu, v, 0);
    b = __shfl_sync(0xffffffffu, v, SM_WARPS);
}
__device__ __forceinline__ double cta_min(SmallCtx& c, double a) {
    a = warp_min(a);
    double* s = c.red + c.flip * 64;
    c.flip ^= 1;
    if (c.lane == 0) s[c.warp] = a;
    __syncthreads();
    double r = s[0];
#pragma unroll
    for (int w = 1; w < SM_WARPS; ++w) r = fmin(r, s[w]);
    return r;
}

// ---- this CTA's columns of H (global, L2 resident after the first pass) -> shared-memory copy; rows >= m and columns
//      beyond the slice stay zero
__device__ __forceinline__ void small_fill_H(const SmallCtx& c, const double* H, int64_t ldh, bool vec) {
    if (c.nloc <= 0) return;
    if (vec) {
        const int per_row = c.nloc >> 1;                // 16-byte chunks per row (col0 and nloc are even here)
        const int total = c.m * per_row;
        for (int e = c.tid; e < total; e += SM_THREADS) {
            const int i = e / per_row, q = e - i * per_row;
            cp_async16(c.Hs + (size_t)i * c.ldn + 2 * q, H + (int64_t)i * ldh + c.col0 + 2 * q, 16);
        }
        cp_async_commit();
    } else {
        const int total = c.m * c.nloc;
        for (int e = c.tid; e < total; e += SM_THREADS) {
            const int i = e / c.nloc, j = e - i * c.nloc;
            c.Hs[(size_t)i * c.ldn + j] = H[(int64_t)i * ldh + c.col0 + j];
        }
    }
}

// ---- A <- H diag(v) H^T (lower 16 x 16 blocks; diagonal blocks are written in full).  In a cluster every CTA forms the
//      blocks over ITS columns, leaves them (packed, 256 doubles per block) in its partial buffer, and after one cluster
//      barrier every CTA adds the C partial buffers in rank order through distributed shared memory: all CTAs hold the
//      same A, bit for bit.  The partial buffers alternate between calls, so the barrier of the next call also covers
//      the reads of this one.
template <int C>
__device__ __forceinline__ void small_gram(SmallCtx& c, const double* v) {
    const int nb = c.MP >> 4;
    const int nblocks = c.nblk16;
    double* part = (C > 1) ? c.part + (size_t)(c.gcount & 1) * nblocks * 256 : nullptr;
    const double* vl = v + c.col0;
    for (int b = c.warp; b < nblocks; b += SM_WARPS) {
        int bi = (int)((sqrtf(8.0f * b + 1.0f) - 1.0f) * 0.5f);
        while ((bi + 1) * (bi + 2) / 2 <= b) ++bi;
        while (bi * (bi + 1) / 2 > b) --bi;
        const int bj = b - bi * (bi + 1) / 2;
        double acc[2][2][2];
#pragma unroll
        for (int i = 0; i < 2; ++i)
#pragma unroll
            for (int j = 0; j < 2; ++j) acc[i][j][0] = acc[i][j][1] = 0.0;
        const double* ap = c.Hs + (size_t)(bi * 16 + c.g) * c.ldn + c.t;
        const double* bp = c.Hs + (size_t)(bj * 16 + c.g) * c.ldn + c.t;
        const size_t r8 = (size_t)8 * c.ldn;
#pragma unroll 2
        for (int k0 = 0; k0 < c.NL; k0 += 4) {
            const double xv = vl[k0 + c.t];
            const double a0 = ap[k0] * xv, a1 = ap[r8 + k0] * xv;
            const double b0 = bp[k0], b1 = bp[r8 + k0];
            dmma884(acc[0][0][0], acc[0][0][1], a0, b0);
            dmma884(acc[0][1][0], acc[0][1][1], a0, b1);
            dmma884(acc[1][0][0], acc[1][0][1], a1, b0);
            dmma884(acc[1][1][0], acc[1][1][1], a1, b1);
        }
#pragma unroll
        for (int i = 0; i < 2; ++i)
#pragma unroll
            for (int j = 0; j < 2; ++j) {
                double* o = (C > 1) ? part + (size_t)b * 256 + (i * 8 + c.g) * 16 + j * 8 + 2 * c.t
                                    : c.A + (size_t)(bi * 16 + i * 8 + c.g) * c.lda + bj * 16 + j * 8 + 2 * c.t;
                o[0] = acc[i][j][0];
                o[1] = acc[i][j][1];
            }
    }
    if (C > 1) {
        namespace cg = cooperative_groups;
        cg::cluster_group cl = cg::this_cluster();
        cl.sync();
        const double* src[C];
#pragma unroll
        for (int r = 0; r < C; ++r) src[r] = cl.map_shared_rank(part, r);
        for (int e = c.tid; e < nblocks * 128; e += SM_THREADS) {          // a pair of doubles per thread and step
            const int b = e >> 7, w = (e & 127) * 2;
            int bi = (int)((sqrtf(8.0f * b + 1.0f) - 1.0f) * 0.5f);
            while ((bi + 1) * (bi + 2) / 2 <= b) ++bi;
            while (bi * (bi + 1) / 2 > b) --bi;
            const int bj = b - bi * (bi + 1) / 2;
            double2 sacc = *reinterpret_cast<const double2*>(src[0] + (size_t)b * 256 + w);
#pragma unroll
            for (int r = 1; r < C; ++r) {
                const double2 q = *reinterpret_cast<const double2*>(src[r] + (size_t)b * 256 + w);
                sacc.x += q.x;
                sacc.y += q.y;
            }
            double* o = c.A + (size_t)(bi * 16 + (w >> 4)) * c.lda + bj * 16 + (w & 15);
            o[0] = sacc.x;
            o[1] = sacc.y;
        }
    }
    ++c.gcount;
    (void)nb;
}

// reciprocal for the pivot chain: 20-bit seed and two Newton steps (4 dependent FMAs, no special-case branches; pivots of a
// positive definite matrix are normal numbers); within 1 ulp of 1/d
__device__ __forceinline__ double pivot_rcp(double d) {
    double x;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(x) : "d"(d));
    double e = fma(-d, x, 1.0);
    x = fma(x, e, x);
    e = fma(-d, x, 1.0);
    return fma(x, e, x);
}

// warp 0: eliminate the 8 x 8 diagonal tile at (j0, j0) - lane i < 8 holds row i, pivot and pivot column travel by
// shuffles - store Lt, d, 1/d, then lanes 0..7 invert the unit lower tile, a column each (-> Xd)
__device__ __forceinline__ void small_diag_tile(SmallCtx& c, int j0) {
    const int m = c.m, lda = c.lda;
    double* T = c.A + (size_t)j0 * lda + j0;
    const int i = c.lane & 7;
    double t[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) t[k] = (k <= i) ? T[(size_t)i * lda + k] : 0.0;
#pragma unroll
    for (int cc = 0; cc < 8; ++cc) {
        const double d = __shfl_sync(0xffffffffu, t[cc], cc);
        const bool live = j0 + cc < m;
        const double r = live ? pivot_rcp(d) : 0.0;
        const double ci = t[cc];
        double ck[8];
#pragma unroll
        for (int k = cc + 1; k < 8; ++k) ck[k] = __shfl_sync(0xffffffffu, ci, k);
        const double l = (i > cc) ? ci * r : 0.0;
#pragma unroll
        for (int k = cc + 1; k < 8; ++k) t[k] -= l * ck[k];      // (entries right of the diagonal are never read)
        if (c.lane == cc && live) { c.dv[j0 + cc] = d; c.rinv[j0 + cc] = r; }
        if (c.lane < 8 && i > cc) { t[cc] = l; T[(size_t)i * lda + cc] = l; }
    }
}

// inverse X of the unit lower 8 x 8 tile at (j0, j0) -> Xd (lanes 0..7 of the calling warp, a column each).  Only the
// gradient's forward substitution needs it, so it runs off the factorisation's critical path.
__device__ __forceinline__ void small_tile_inverse(const SmallCtx& c, int j0) {
    const double* T = c.A + (size_t)j0 * c.lda + j0;
    if (c.lane < 8) {
        const int cc = c.lane;
        double xcol[8];
#pragma unroll
        for (int r = 0; r < 8; ++r) xcol[r] = (r == cc) ? 1.0 : 0.0;
#pragma unroll
        for (int r = 1; r < 8; ++r) {
            double sacc = 0.0;
#pragma unroll
            for (int k = 0; k < r; ++k) sacc += T[(size_t)r * c.lda + k] * xcol[k];
            if (r > cc) xcol[r] = -sacc;
        }
#pragma unroll
        for (int r = 0; r < 8; ++r) c.Xd[(size_t)(j0 + r) * 12 + cc] = xcol[r];
    }
}

// rows below the diagonal tile of panel p, a lane per row: C[i, :] Lt_diag^T = A[i, panel] by substitution over the eight
// columns (C = Lt D, the unscaled panel -> Cp), Lt[i, :] = C[i, :] D^-1 -> A.  Needs the eliminated tile, not its inverse.
__device__ __forceinline__ void small_panel_rows(const SmallCtx& c, int j0, int row) {
    const double* T = c.A + (size_t)j0 * c.lda + j0;
    double* ar = c.A + (size_t)row * c.lda + j0;
    double t[8];
#pragma unroll
    for (int k = 0; k < 8; k += 2) {
        const double2 v = *reinterpret_cast<const double2*>(ar + k);
        t[k] = v.x; t[k + 1] = v.y;
    }
#pragma unroll
    for (int k = 1; k < 8; ++k)
#pragma unroll
        for (int q = 0; q < k; ++q) t[k] -= t[q] * T[(size_t)k * c.lda + q];
    double* cq = c.Cp + (size_t)row * 12;
#pragma unroll
    for (int k = 0; k < 8; k += 2) {
        *reinterpret_cast<double2*>(cq + k) = make_double2(t[k], t[k + 1]);
        *reinterpret_cast<double2*>(ar + k) = make_double2(t[k] * c.rinv[j0 + k], t[k + 1] * c.rinv[j0 + k + 1]);
    }
}

__device__ __forceinline__ void small_trailing_tile(const SmallCtx& c, int j0, int I, int K) {
    double* o = c.A + (size_t)(I * 8 + c.g) * c.lda + K * 8 + 2 * c.t;
    double acc0 = o[0], acc1 = o[1];
    const double* lp = c.A + (size_t)(I * 8 + c.g) * c.lda + j0 + c.t;
    const double* cp = c.Cp + (size_t)(K * 8 + c.g) * 12 + c.t;
    dmma884(acc0, acc1, -lp[0], cp[0]);
    dmma884(acc0, acc1, -lp[4], cp[4]);
    o[0] = acc0;
    o[1] = acc1;
}

// (look-ahead) the diagonal tile of panel p + 1 is updated first and eliminated by warp 0 while the other warps apply
// panel p to the rest of the trailing matrix
__device__ __forceinline__ double small_factor(SmallCtx& c, bool& bad) {
    const int m = c.m, lda = c.lda, MP = c.MP;
    double* A = c.A;
    double* Cp = c.Cp;
    for (int i = m + c.tid; i < MP; i += SM_THREADS) { c.dv[i] = 1.0; c.rinv[i] = 0.0; }
    const int npan = (m + 7) >> 3, ntl = MP >> 3;
    long long tq = clock64();
    if (c.warp == 0) small_diag_tile(c, 0);
    __syncthreads();
    { const long long now = clock64(); c.tf0 += now - tq; tq = now; }
    for (int p = 0; p < npan; ++p) {
        const int j0 = 8 * p;
        // panel: the rows below the diagonal tile, a lane per row (warps 0..); one more warp inverts the tile meanwhile
        {
            const int rows = MP - (j0 + 8);
            const int pw = (rows + 31) >> 5;            // warps that hold rows
            if (c.warp < pw) {
                const int row = j0 + 8 + c.tid;
                if (row < MP) small_panel_rows(c, j0, row);
            } else if (c.warp == pw) {
                small_tile_inverse(c, j0);
            }
        }
        const int nt = ntl - (p + 1);
        if (nt <= 0) break;
        __syncthreads();
        { const long long now = clock64(); c.tf2 += now - tq; tq = now; }
        const int ntile = nt * (nt + 1) / 2;
        if (c.warp == 0) {
            small_trailing_tile(c, j0, p + 1, p + 1);
            __syncwarp();
            if (p + 1 < npan) small_diag_tile(c, j0 + 8);
        } else {
            for (int e = c.warp; e < ntile; e += SM_WARPS - 1) {            // tiles 1 .. ntile-1 over warps 1 .. 15
                int ii = (int)((sqrtf(8.0f * e + 1.0f) - 1.0f) * 0.5f);
                while ((ii + 1) * (ii + 2) / 2 <= e) ++ii;
                while (ii * (ii + 1) / 2 > e) --ii;
                const int kk = e - ii * (ii + 1) / 2;
                small_trailing_tile(c, j0, p + 1 + ii, p + 1 + kk);
            }
        }
        __syncthreads();
        { const long long now = clock64(); c.tf3 += now - tq; tq = now; }
    }
    __syncthreads();
    double s = 0.0, z = 0.0;
    bool b = false;
    for (int i = c.tid; i < m; i += SM_THREADS) {
        const double d = c.dv[i];
        if (!(d > 0.0)) b = true;
        s += log(d);
    }
    z = b ? 1.0 : 0.0;
    cta_sum2(c, s, z);
    bad = z > 0.0;
    return -s;
}

// ---- inverses of the 8 x 8 unit lower diagonal blocks of Lt -> Xd (rows of 12 doubles)
__device__ __forceinline__ void small_diag_inverses(const SmallCtx& c) {
    const int nblk = c.MP >> 3;
    for (int e = c.tid; e < nblk * 8; e += SM_THREADS) {
        const int I = e >> 3, cc = e & 7;
        const double* Lb = c.A + (size_t)(I * 8) * c.lda + I * 8;
        double xcol[8];
#pragma unroll
        for (int r = 0; r < 8; ++r) xcol[r] = (r == cc) ? 1.0 : 0.0;
#pragma unroll
        for (int r = 1; r < 8; ++r) {
            double s = 0.0;
#pragma unroll
            for (int k = 0; k < r; ++k) s += Lb[(size_t)r * c.lda + k] * xcol[k];
            if (r > cc) xcol[r] = -s;
        }
#pragma unroll
        for (int r = 0; r < 8; ++r) c.Xd[(size_t)(I * 8 + r) * 12 + cc] = xcol[r];
    }
}

// ---- g_j = -sum_i (Lt^-1 h_j)_i^2 / d_i : forward substitution in place on Hs.  A warp owns NB = 1 or 2 blocks of 8
//      columns and walks them together (the fragments of Lt are loaded once for both, and the blocks' DMMA chains are
//      independent)
template <int NB>
__device__ __forceinline__ void small_gradient_blocks(const SmallCtx& c, int cb0) {
    const int nblk = c.MP >> 3;
    double n0[NB], n1[NB];
    double* Hc[NB];
#pragma unroll
    for (int b = 0; b < NB; ++b) { n0[b] = n1[b] = 0.0; Hc[b] = c.Hs + (cb0 + b * SM_WARPS) * 8; }
    for (int I = 0; I < nblk; ++I) {
        double s0[NB], s1[NB], u0[NB], u1[NB];
#pragma unroll
        for (int b = 0; b < NB; ++b) s0[b] = s1[b] = u0[b] = u1[b] = 0.0;
        const double* ap = c.A + (size_t)(I * 8 + c.g) * c.lda + c.t;
        const size_t boff = (size_t)c.t * c.ldn + c.g;
        const int kend = I * 8;
        for (int k0 = 0; k0 + 8 <= kend; k0 += 8) {     // two accumulators per block: no DMMA waits for its predecessor
            const double a0 = ap[k0], a1 = ap[k0 + 4];
#pragma unroll
            for (int b = 0; b < NB; ++b) {
                dmma884(s0[b], s1[b], a0, Hc[b][boff + (size_t)k0 * c.ldn]);
                dmma884(u0[b], u1[b], a1, Hc[b][boff + (size_t)(k0 + 4) * c.ldn]);
            }
        }
        double* hp[NB];
#pragma unroll
        for (int b = 0; b < NB; ++b) {
            hp[b] = Hc[b] + (size_t)(I * 8 + c.g) * c.ldn + 2 * c.t;
            const double r0 = hp[b][0] - (s0[b] + u0[b]), r1 = hp[b][1] - (s1[b] + u1[b]);
            hp[b][0] = r0;
            hp[b][1] = r1;
        }
        __syncwarp();
        const double* xp = c.Xd + (size_t)(I * 8 + c.g) * 12 + c.t;
        const double x0 = xp[0], x4 = xp[4];
        const size_t roff = (size_t)(I * 8 + c.t) * c.ldn + c.g;
        double w0[NB], w1[NB];
#pragma unroll
        for (int b = 0; b < NB; ++b) {
            w0[b] = w1[b] = 0.0;
            dmma884(w0[b], w1[b], x0, Hc[b][roff]);
            dmma884(w0[b], w1[b], x4, Hc[b][roff + (size_t)4 * c.ldn]);
        }
        __syncwarp();
        const double ri = c.rinv[I * 8 + c.g];
#pragma unroll
        for (int b = 0; b < NB; ++b) {
            hp[b][0] = w0[b];
            hp[b][1] = w1[b];
            n0[b] += w0[b] * w0[b] * ri;
            n1[b] += w1[b] * w1[b] * ri;
        }
        __syncwarp();
    }
#pragma unroll
    for (int b = 0; b < NB; ++b) {
        // rows live in the lane groups g = 0..7: add them in a fixed tree
#pragma unroll
        for (int o = 4; o < 32; o <<= 1) {
            n0[b] += __shfl_xor_sync(0xffffffffu, n0[b], o);
            n1[b] += __shfl_xor_sync(0xffffffffu, n1[b], o);
        }
        if (c.g == 0) {
            c.gs[c.col0 + (cb0 + b * SM_WARPS) * 8 + 2 * c.t] = -n0[b];
            c.gs[c.col0 + (cb0 + b * SM_WARPS) * 8 + 2 * c.t + 1] = -n1[b];
        }
    }
}
// NBMAX = 1: every warp walks one block at a time (same values; fewer registers, for a kernel that holds more state)
template <int C, int NBMAX = 2>
__device__ __forceinline__ void small_gradient(const SmallCtx& c) {
    const int ncb = c.NL >> 3;
    for (int cb = c.warp; cb < ncb; cb += NBMAX * SM_WARPS) {
        if (NBMAX == 2 && cb + SM_WARPS < ncb) small_gradient_blocks<NBMAX>(c, cb);
        else small_gradient_blocks<1>(c, cb);
    }
    if (C > 1) {
        // every CTA needs the whole gradient for the (replicated) prox: each one stores its slice into the other CTAs'
        // vectors through distributed shared memory; the cluster barrier that publishes it follows in the caller
        namespace cg = cooperative_groups;
        cg::cluster_group cl = cg::this_cluster();
        __syncthreads();
#pragma unroll
        for (int r = 1; r < C; ++r) {
            double* dst = cl.map_shared_rank(c.gs, (c.rank + r) % C);
            for (int i = c.tid; i < c.NL; i += SM_THREADS) dst[c.col0 + i] = c.gs[c.col0 + i];
        }
    }
}

// ---- out <- argmin <g, x> + L D(x, ctr) on the simplex (Burg kernel, g in c.gs); returns the Newton steps taken.
//      Only the warps that hold elements (n / 32 of them, at most 16) run the root-find, on a named barrier of their own:
//      the sums of a Newton step cost one barrier among those warps and the idle warps do not compete for issue slots.
__device__ __forceinline__ void grp_bar(int nthreads) { asm volatile("bar.sync 1, %0;" ::"r"(nthreads) : "memory"); }
__device__ __forceinline__ void grp_sum2(const SmallCtx& c, int nw, int& gf, double& a, double& b) {
    a = warp_sum(a);
    b = warp_sum(b);
    double* s = c.red + 128 + gf * 32;
    gf ^= 1;
    if (c.lane == 0) { s[c.warp] = a; s[SM_WARPS + c.warp] = b; }
    grp_bar(nw * 32);
    double v = ((c.lane & (SM_WARPS - 1)) < nw) ? s[c.lane] : 0.0;
#pragma unroll
    for (int o = SM_WARPS / 2; o >= 1; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    a = __shfl_sync(0xffffffffu, v, 0);
    b = __shfl_sync(0xffffffffu, v, SM_WARPS);
}
__device__ __forceinline__ int small_prox(SmallCtx& c, const double* ctr, double* out, double L, double eps,
                                          uint32_t& st) {
    const int n = c.n;
    const int nw = min(SM_WARPS, (n + 31) >> 5);
    int nnewton = 0;
    if (c.warp < nw) {
        int gf = 0;
        double lo = kInf;
        for (int i = c.tid; i < n; i += SM_THREADS) {
            const double yi = ctr[i];
            if (!(yi > 0.0)) st |= ACCBPG_ST_ARG_NOT_POS;
            const double v = __ddiv_rn(__dsub_rn(c.gs[i], __dmul_rn(L, -1.0 / yi)), L);      // no FMA contraction: NumPy's rounding
            out[i] = v;
            lo = fmin(lo, v);
        }
        lo = warp_min(lo);
        {
            double* s = c.red + 128 + gf * 32;
            gf ^= 1;
            if (c.lane == 0) s[c.warp] = lo;
            grp_bar(nw * 32);
            double v = (c.lane < nw) ? s[c.lane] : kInf;
            lo = warp_min(v);
        }
        const double cmin = -lo;
        double cc = cmin + 1.0;
        int nbis = 0;
        double s1, s2;
        auto sums = [&](double q) {
            double a = 0.0, b = 0.0;
            for (int i = c.tid; i < n; i += SM_THREADS) {
                const double tq = out[i] + q;
                a += 1.0 / tq;
                b += -1.0 / __dmul_rn(tq, tq);
            }
            grp_sum2(c, nw, gf, a, b);
            s1 = a; s2 = b;
        };
        for (;;) {                                            // functions.py:344-346
            sums(cc);
            if (s1 - 1.0 < 0.0 && nbis < 2000) { cc = (cmin + cc) / 2.0; ++nbis; }
            else break;
        }
        double fc = s1 - 1.0;
        while (fabs(fc) > eps) {                              // functions.py:348-354
            const double cn = cc - fc / s2;
            if (cc - cn == 0.0) break;
            cc = cn;
            sums(cc);
            fc = s1 - 1.0;
            if (++nnewton >= 200) { st |= ACCBPG_ST_NEWTON_MAXIT; break; }
        }
        for (int i = c.tid; i < n; i += SM_THREADS) out[i] = 1.0 / (out[i] + cc);
    }
    return nnewton;
}

// ---- the buffers of a plan, this CTA's rank and column slice, the thread's place in the CTA
template <int C>
__device__ __forceinline__ void small_ctx(SmallCtx& c, const SmallPlan& pl, unsigned char* sm_raw, int m, int n) {
    namespace cg = cooperative_groups;
    c.Hs = (double*)(sm_raw + pl.off_H);   c.A = (double*)(sm_raw + pl.off_A);
    c.part = (double*)(sm_raw + pl.off_part);
    c.xs = (double*)(sm_raw + pl.off_x);   c.x1s = (double*)(sm_raw + pl.off_x1);
    c.gs = (double*)(sm_raw + pl.off_g);   c.dv = (double*)(sm_raw + pl.off_d);
    c.rinv = (double*)(sm_raw + pl.off_rinv); c.Cp = (double*)(sm_raw + pl.off_cp);
    c.Xd = (double*)(sm_raw + pl.off_xd);  c.red = (double*)(sm_raw + pl.off_red);
    c.m = m; c.n = n; c.MP = pl.MP; c.NP = pl.NP; c.ldn = pl.ldn; c.lda = pl.lda;
    c.C = C; c.rank = (C > 1) ? (int)cg::this_cluster().block_rank() : 0;
    c.NL = pl.NL; c.col0 = c.rank * pl.NL; c.nloc = min(pl.NL, n - c.col0); c.nblk16 = pl.nblk16; c.gcount = 0;
    if (c.nloc < 0) c.nloc = 0;
    c.tid = threadIdx.x; c.lane = c.tid & 31; c.warp = c.tid >> 5; c.g = c.lane >> 2; c.t = c.lane & 3;
    c.flip = 0;
    c.tf0 = c.tf1 = c.tf2 = c.tf3 = 0;
}

template <int C>
__global__ void __launch_bounds__(SM_THREADS, 1) dopt_bpg_small_kernel(SmallParams p) {
    extern __shared__ __align__(16) unsigned char sm_raw[];
    namespace cg = cooperative_groups;
    const SmallPlan pl = small_plan(p.m, p.n, C);
    SmallCtx c;
    small_ctx<C>(c, pl, sm_raw, p.m, p.n);
    const bool vec = ((reinterpret_cast<uintptr_t>(p.H) & 15u) == 0) && (p.ldh % 2 == 0) && (p.n % 2 == 0);
    const bool writer = c.rank == 0;
    uint32_t st = 0;

    for (size_t e = c.tid; e < pl.bytes / 8; e += SM_THREADS) ((double*)sm_raw)[e] = 0.0;
    __syncthreads();
    if (C > 1) cg::this_cluster().sync();               // no CTA's shared memory is written remotely before it is cleared
    small_fill_H(c, p.H, p.ldh, vec);
    for (int i = c.tid; i < p.n; i += SM_THREADS) {
        const double v = p.x[i];
        if (v < 0.0) st |= ACCBPG_ST_X_NEGATIVE;
        c.xs[i] = v;
    }
    if (vec) cp_async_wait<0>();
    __syncthreads();

    bool bad = false;
    long long tp0 = 0, tp1 = 0, tp2 = 0, tp3 = 0, tp4 = 0, tp5 = 0;   // clocks per phase: diag inverses, gradient, prox, div/dot, Gram, factor
    long long tc = clock64();
#define SM_LAP(v) { const long long now_ = clock64(); v += now_ - tc; tc = now_; }
    small_gram<C>(c, c.xs);
    __syncthreads();
    double fx = small_factor(c, bad);
    double L = p.L;
    int k = 0, trials = 0, newton = 0;
    double fprev = 0.0;
    if (bad) st |= ACCBPG_ST_NOT_PD;
    for (; k < p.maxitrs && !bad; ++k) {
        if (writer && c.tid == 0) p.F[k] = fx;
        // gradient at x from the factor in A
        tc = clock64();
        small_gradient<C>(c);
        if (C > 1) cg::this_cluster().sync();           // the other CTAs' slices of the gradient have arrived
        else __syncthreads();
        small_fill_H(c, p.H, p.ldh, vec);                        // refill the copy of H under the prox
        SM_LAP(tp1);
        if (p.linesearch) L = L / p.ls_ratio;
        double f1 = 0.0;
        for (;;) {
            newton += small_prox(c, c.xs, c.x1s, L, p.eps_prox, st);
            ++trials;
            __syncthreads();                            // x1 complete
            SM_LAP(tp2);
            double dsum = 0.0, dot = 0.0;
            for (int i = c.tid; i < p.n; i += SM_THREADS) {
                const double xi = c.x1s[i], yi = c.xs[i];
                if (!(xi > 0.0)) st |= ACCBPG_ST_ARG_NOT_POS;
                const double r = xi / yi;
                dsum += __dsub_rn(__dsub_rn(r, log(r)), 1.0);
                dot += __dmul_rn(c.gs[i], __dsub_rn(xi, yi));
            }
            if (vec) cp_async_wait<0>();
            cta_sum2(c, dsum, dot);                     // (its barrier also publishes the refilled H)
            SM_LAP(tp3);
            small_gram<C>(c, c.x1s);
            __syncthreads();
            SM_LAP(tp4);
            f1 = small_factor(c, bad);
            SM_LAP(tp5);
            if (bad) { st |= ACCBPG_ST_NOT_PD; break; }
            if (!p.linesearch) break;
            if (f1 > __dadd_rn(__dadd_rn(fx, dot), __dmul_rn(L, dsum))) L = L * p.ls_ratio;            // algorithms.py:53
            else break;
        }
        if (bad) { ++k; break; }
        for (int i = c.tid; i < p.n; i += SM_THREADS) c.xs[i] = c.x1s[i];
        if (writer && c.tid == 0) p.Ls[k] = L;
        const double fk = fx;
        fx = f1;
        __syncthreads();
        if (k > 0 && fabs(fk - fprev) < p.epsilon) { ++k; break; }       // algorithms.py:70
        fprev = fk;
    }
    if (C > 1) cg::this_cluster().sync();               // nobody leaves while its shared memory may still be read
    if (writer)
        for (int i = c.tid; i < p.n; i += SM_THREADS) p.x[i] = c.xs[i];
    if (st) atomicOr(p.status, st);
    if (writer && c.tid == 0) {
        p.info[0] = (double)k; p.info[1] = (double)trials; p.info[2] = L; p.info[3] = (double)newton;
        p.info[4] = (double)tp0; p.info[5] = (double)tp1; p.info[6] = (double)tp2; p.info[7] = (double)tp3;
        p.info[8] = (double)tp4; p.info[9] = (double)tp5;
        p.info[10] = (double)c.tf0; p.info[11] = (double)c.tf1; p.info[12] = (double)c.tf2; p.info[13] = (double)c.tf3;
    }
}

// ---- ABPG / ABPG_gain (algorithms.py:94-180, :295-420) on the same machinery ---------------------------------------

struct SmallAccParams {
    const double* H; int m, n; int64_t ldh;
    double* x;                       // in: x0, out: the last iterate
    double L, gamma, epsilon, eps_prox, G0, ls_inc, ls_dec;
    int maxitrs, theta_eq, restart, rule, checkdiv;
    double* hist;                    // rows of maxitrs: F, G / Gain, Gdiv, theta, D(x,y), D(z,z-), T
    double* info;                    // [0] entries written, [1] trips, [2] cluster size, [3] Gdr unbound, [4] last G / gain
    uint32_t* status;
};

// ---- CTA-wide sums of K <= SM_ACC_SUMS values with one barrier: warps leave their partials in one of two alternating
//      buffers, every thread adds them in warp order (the same bits in every thread, and in every CTA given the same
//      inputs)
template <int K>
__device__ __forceinline__ void cta_sumk(const SmallCtx& c, double* red, int& flip, double (&v)[K]) {
    double* s = red + flip * (SM_ACC_SUMS * SM_WARPS);
    flip ^= 1;
#pragma unroll
    for (int q = 0; q < K; ++q) {
        v[q] = warp_sum(v[q]);
        if (c.lane == 0) s[q * SM_WARPS + c.warp] = v[q];
    }
    __syncthreads();
#pragma unroll
    for (int q = 0; q < K; ++q) {
        double a = s[q * SM_WARPS];
#pragma unroll
        for (int w = 1; w < SM_WARPS; ++w) a = __dadd_rn(a, s[q * SM_WARPS + w]);
        v[q] = a;
    }
}

// ---- f(v) = -log det(H diag(v) H^T) from scratch: waits for this CTA's refill of its slice of H (only this CTA reads
//      it), then Gram matrix and factorisation; the factor stays in c.A for small_gradient
template <int C>
__device__ __forceinline__ double small_value(SmallCtx& c, const double* v, bool vec, bool& bad) {
    if (vec) cp_async_wait<0>();
    __syncthreads();                                    // v complete, the refilled H visible
    small_gram<C>(c, v);
    __syncthreads();
    return small_factor(c, bad);
}

// Every point is evaluated from scratch, as the reference does; carrying the Gram images M(x-), M(z-) and M(z) next to H
// would not fit one SM at 80 x 200.  An iteration starts with f(x_k) = F[k] when no trip has formed it, then each trip:
//   1. y = (1-theta) x- + theta z-; Gram, factor, f(y); gradient g at y in place on the copy of H, whose refill starts
//   2. z = div_prox_map(z-, g, theta^(gamma-1) [G] L)
//   3. x = (1-theta) x- + theta z; D(x, y), D(z, z-), dot(g, x - y), the restart dot dot(g, x - x-) and the status in
//      one CTA-wide sum
//   4. ABPG_gain without checkdiv, after the refill: Gram, factor, f(x) for the line search (:387); the accepted trip's
//      value is F[k+1]
// The scalar and elementwise expressions round like the host's Python / NumPy arithmetic and accbpg_vec_axpby (explicit
// round-to-nearest operations: this file is compiled with FMA contraction).  Every CTA takes every decision from the
// same bits: the vectors are replicated and the Gram matrix is summed in rank order.  What a decision needs after a
// Gram pass is reduced to a few values before it (the restart tests, the line search's right-hand side), so the scalar
// control does not add to the register pressure of the passes.
template <int C, int DRV>
__global__ void __launch_bounds__(SM_THREADS, 1) dopt_abpg_small_kernel(SmallAccParams p) {
    extern __shared__ __align__(16) unsigned char sm_raw[];
    namespace cg = cooperative_groups;
    constexpr bool GAIN = DRV == ACCBPG_SMALL_DRV_ABPG_GAIN;
    const unsigned long long ns0 = ls_clock();
    const SmallPlan pl = small_plan(p.m, p.n, C, true);
    SmallCtx c;
    small_ctx<C>(c, pl, sm_raw, p.m, p.n);
    double* const X1 = c.xs;                            // x-
    double* const Z1 = c.x1s;                           // z-
    double* const Y = (double*)(sm_raw + pl.off_acc);
    double* const Z = Y + pl.NP;
    double* const X = Z + pl.NP;
    double* const red = X + pl.NP;
    int rflip = 0;
    const bool vec = ((reinterpret_cast<uintptr_t>(p.H) & 15u) == 0) && (p.ldh % 2 == 0) && (p.n % 2 == 0);
    const bool writer = c.rank == 0 && c.tid == 0;
    const int n = p.n, M = p.maxitrs;
    auto hist = [&](int row, int k) -> double& { return p.hist[(size_t)row * M + k]; };   // rows: see SmallAccParams
    uint32_t st = 0;

    for (size_t e = c.tid; e < pl.bytes / 8; e += SM_THREADS) ((double*)sm_raw)[e] = 0.0;
    __syncthreads();
    if (C > 1) cg::this_cluster().sync();               // no CTA's shared memory is written remotely before it is cleared
    small_fill_H(c, p.H, p.ldh, vec);
    for (int i = c.tid; i < n; i += SM_THREADS) {       // x0 and z0 = x0
        const double v = p.x[i];
        if (v < 0.0) st |= ACCBPG_ST_X_NEGATIVE;
        X1[i] = v;
        Z1[i] = v;
    }
    bool stop;
    {
        double s0 = st ? 1.0 : 0.0, s1 = 0.0;           // a negative entry of x0 ends the solve before f(x0)
        cta_sum2(c, s0, s1);
        stop = s0 > 0.0;
    }

    double theta = 1.0, G = p.G0, gdr = 0.0, fx = 0.0, Fprev = 0.0;
    bool have_fx = false, gdr_bound = false;
    int kk = 0, k = 0, trips = 0, unbound = 0, newton = 0;
    for (; k < M && !stop; ++k) {
        if (writer) hist(6, k) = (double)(ls_clock() - ns0);
        if (!have_fx) {                                 // F[k] = f(x_k) from scratch
            bool bad = false;
            fx = small_value<C>(c, X1, vec, bad);
            if (bad) { st |= ACCBPG_ST_NOT_PD; break; }
        }
        if (writer) hist(0, k) = fx;
        // restart rule 'f' (algorithms.py:168, :406): F[k] > F[k-1]; ABPG_gain's at k = 0 compares with F[-1], the
        // reference's still-zero last slot
        const bool rs_f = fx > (k > 0 ? Fprev : (M == 1 ? fx : 0.0));
        Fprev = fx;
        const double G_1 = G, theta_1 = theta;
        if (GAIN) G = __ddiv_rn(G, p.ls_dec);
        else theta = (p.theta_eq && kk > 0) ? la_solve_theta(theta, p.gamma, 1.0)
                                            : __ddiv_rn(p.gamma, __dadd_rn((double)kk, p.gamma));
        bool rs_g = false, dzz_small = false;
        for (;;) {
            ++trips;
            have_fx = false;
            if (GAIN && kk > 0) {
                if (p.theta_eq) {
                    theta = la_solve_theta(theta_1, p.gamma, __ddiv_rn(G, G_1));
                } else {
                    const double alpha = __ddiv_rn(G, G_1);                           // algorithms.py:367
                    theta = __dmul_rn(theta_1, __ddiv_rn(__dadd_rn(1.0, __dmul_rn(alpha, __dsub_rn(p.gamma, 1.0))),
                                                         __dadd_rn(__dmul_rn(p.gamma, alpha), theta_1)));
                }
            }
            // 1. y, f(y), g = grad f(y); the copy of H is refilled under steps 2 and 3
            {
                const double omt = __dsub_rn(1.0, theta);
                for (int i = c.tid; i < n; i += SM_THREADS)
                    Y[i] = __dadd_rn(__dmul_rn(omt, X1[i]), __dmul_rn(theta, Z1[i]));
            }
            bool bad = false;
            const double fy = small_value<C>(c, Y, vec, bad);
            if (bad) { st |= ACCBPG_ST_NOT_PD; stop = true; break; }
            small_gradient<C, 1>(c);
            if (C > 1) cg::this_cluster().sync();       // the other CTAs' slices of the gradient have arrived
            else __syncthreads();
            small_fill_H(c, p.H, p.ldh, vec);
            // 2. z
            {
                const double tg1 = la_pow(theta, __dsub_rn(p.gamma, 1.0));
                const double Lz = GAIN ? __dmul_rn(__dmul_rn(tg1, G), p.L) : __dmul_rn(tg1, p.L);
                newton += small_prox(c, Z1, Z, Lz, p.eps_prox, st);
            }
            __syncthreads();                            // z complete
            // 3. x and the trip's sums: D(x, y), D(z, z-), dot(g, x - y), dot(g, x - x-), status
            double a[SM_ACC_SUMS] = {0.0, 0.0, 0.0, 0.0, 0.0};
            {
                const double omt = __dsub_rn(1.0, theta);
                for (int i = c.tid; i < n; i += SM_THREADS) {
                    const double x1i = X1[i], z1i = Z1[i], zi = Z[i], yi = Y[i], gi = c.gs[i];
                    const double xi = __dadd_rn(__dmul_rn(omt, x1i), __dmul_rn(theta, zi));
                    X[i] = xi;
                    if (!(xi > 0.0) || !(zi > 0.0)) st |= ACCBPG_ST_ARG_NOT_POS;
                    const double r = __ddiv_rn(xi, yi), q = __ddiv_rn(zi, z1i);
                    a[0] = __dadd_rn(a[0], __dsub_rn(__dsub_rn(r, log(r)), 1.0));
                    a[1] = __dadd_rn(a[1], __dsub_rn(__dsub_rn(q, log(q)), 1.0));
                    a[2] = __dadd_rn(a[2], __dmul_rn(gi, __dsub_rn(xi, yi)));
                    a[3] = __dadd_rn(a[3], __dmul_rn(gi, __dsub_rn(xi, x1i)));
                }
            }
            a[4] = st ? 1.0 : 0.0;
            cta_sumk<SM_ACC_SUMS>(c, red, rflip, a);    // (its barrier also publishes x)
            if (a[4] > 0.0) { stop = true; break; }
            const double tg = la_pow(theta, p.gamma);
            if (writer) { hist(3, k) = theta; hist(4, k) = a[0]; hist(5, k) = a[1]; }
            rs_g = a[3] > 0.0;
            dzz_small = a[1] < p.epsilon;
            if (GAIN && dzz_small) break;               // Gdr keeps its previous value, as in the reference
            gdr = __ddiv_rn(__ddiv_rn(a[0], a[1]), tg);
            if (!GAIN) break;
            gdr_bound = true;
            bool again;
            if (p.checkdiv) {
                again = gdr > G;
            } else {
                const double rhs = __dadd_rn(__dadd_rn(fy, a[2]), __dmul_rn(__dmul_rn(__dmul_rn(tg, G), p.L), a[1]));
                fx = small_value<C>(c, X, vec, bad);    // 4.
                if (bad) { st |= ACCBPG_ST_NOT_PD; stop = true; break; }
                have_fx = true;
                again = fx > rhs;                       // algorithms.py:387
            }
            if (!again) break;
            G = __dmul_rn(G, p.ls_inc);
        }
        if (stop) { ++k; break; }
        if (GAIN && !gdr_bound) { unbound = 1; break; }  // the reference's Gdiv[k] = Gdr raises UnboundLocalError
        if (writer) {
            hist(1, k) = GAIN ? G : gdr;
            if (GAIN) hist(2, k) = gdr;
        }
        ++kk;
        // restart (algorithms.py:168, :406): ABPG only from k = 1, ABPG_gain from k = 0
        bool rs = false;
        if (p.restart && (GAIN || k > 0))
            rs = p.rule == ACCBPG_SMALL_RESTART_F ? rs_f : p.rule == ACCBPG_SMALL_RESTART_G ? rs_g : false;
        if (rs) { theta = 1.0; kk = 0; }
        for (int i = c.tid; i < n; i += SM_THREADS) {  // x- <- x, z- <- z (x on a restart)
            const double xi = X[i];
            X1[i] = xi;
            Z1[i] = rs ? xi : Z[i];
        }
        if (dzz_small) { ++k; break; }
    }
    if (vec) cp_async_wait<0>();                        // a refill still in flight when a status bit ended the solve
    if (C > 1) cg::this_cluster().sync();               // nobody leaves while its shared memory may still be read
    if (c.rank == 0)
        for (int i = c.tid; i < n; i += SM_THREADS) p.x[i] = X1[i];
    if (st) atomicOr(p.status, st);
    if (writer) {
        p.info[0] = (double)k; p.info[1] = (double)trips; p.info[2] = (double)C; p.info[3] = (double)unbound;
        p.info[4] = GAIN ? G : gdr; p.info[5] = (double)newton;
    }
}

// cluster size for a shape: the largest of {preferred, 2, 1} whose plan fits one SM's shared memory (a cluster also
// admits shapes whose H does not fit a single CTA).  ACCBPG_SMALL_CLUSTER = 1 / 2 / 4 overrides the preference.
// acc: the plan of dopt_abpg_small_kernel.
static int small_pick_cluster(int m, int64_t n, size_t* bytes, bool acc = false) {
    if (m < 1 || m > SM_MAX_M || n < 2 || n > 65536 || n <= m) return 0;
    static int pref = 0;
    if (pref == 0) { const char* e = getenv("ACCBPG_SMALL_CLUSTER"); pref = e ? atoi(e) : 4; if (pref != 1 && pref != 2 && pref != 4) pref = 4; }
    const int cand[3] = {pref, pref > 2 ? 2 : 1, 1};
    for (int q = 0; q < 3; ++q) {
        const int C = cand[q];
        if (C > 1 && n < 32 * C) continue;              // too few columns to be worth splitting
        const SmallPlan pl = small_plan(m, (int)n, C, acc);
        if (pl.bytes <= (size_t)SM_SMEM_LIMIT) { if (bytes) *bytes = pl.bytes; return C; }
    }
    return 0;
}

template <auto KERNEL, class P>
static int small_launch(Ctx* c, cudaStream_t s, const P& p, int C, size_t smem) {
    static bool attr_done[kMaxDevices] = {};
    if (!(c->device >= 0 && c->device < kMaxDevices && attr_done[c->device])) {
        ACCBPG_CUDA(cudaFuncSetAttribute(KERNEL, cudaFuncAttributeMaxDynamicSharedMemorySize, SM_SMEM_LIMIT));
        if (c->device >= 0 && c->device < kMaxDevices) attr_done[c->device] = true;
    }
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(C, 1, 1);
    cfg.blockDim = dim3(SM_THREADS, 1, 1);
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
static int small_acc_launch(Ctx* c, cudaStream_t s, const SmallAccParams& p, int C, size_t smem) {
    return C == 4 ? small_launch<dopt_abpg_small_kernel<4, DRV>>(c, s, p, C, smem)
         : C == 2 ? small_launch<dopt_abpg_small_kernel<2, DRV>>(c, s, p, C, smem)
                  : small_launch<dopt_abpg_small_kernel<1, DRV>>(c, s, p, C, smem);
}

}  // namespace accbpg

using namespace accbpg;

extern "C" {

size_t accbpg_dopt_bpg_small_smem_bytes(int m, int64_t n) {
    size_t bytes = 0;
    return small_pick_cluster(m, n, &bytes) ? bytes : 0;
}

int accbpg_dopt_bpg_small(void* ctx, void* stream, const double* H, int m, int64_t n, int64_t ldh, double* x, double L,
                          double ls_ratio, int linesearch, int maxitrs, double epsilon, double eps_prox, double* F_out,
                          double* Ls_out, double* info_out) {
    Ctx* c = (Ctx*)ctx;
    cudaStream_t s = (cudaStream_t)stream;
    if (!c || !H || !x || !F_out || !Ls_out || !info_out) return arg_err("dopt_bpg_small: NULL pointer");
    ACCBPG_ON_DEVICE(c);
    size_t smem = 0;
    const int C = small_pick_cluster(m, n, &smem);
    if (C == 0 || ldh < n) return arg_err("dopt_bpg_small: shape does not fit one SM (accbpg_dopt_bpg_small_smem_bytes)");
    if (!(L > 0.0) || !(ls_ratio > 1.0) || maxitrs < 1 || !(eps_prox > 0.0)) return arg_err("dopt_bpg_small: L, ls_ratio, maxitrs, eps");
    SmallParams p;
    p.H = H; p.m = m; p.n = (int)n; p.ldh = ldh; p.x = x; p.L = L; p.ls_ratio = ls_ratio; p.epsilon = epsilon;
    p.eps_prox = eps_prox; p.linesearch = linesearch; p.maxitrs = maxitrs; p.F = F_out; p.Ls = Ls_out; p.info = info_out;
    p.status = c->d_status;
    int rc = C == 4 ? small_launch<dopt_bpg_small_kernel<4>>(c, s, p, C, smem)
           : C == 2 ? small_launch<dopt_bpg_small_kernel<2>>(c, s, p, C, smem)
                    : small_launch<dopt_bpg_small_kernel<1>>(c, s, p, C, smem);
    if (rc) return rc;
    ACCBPG_LAUNCHED("dopt_bpg_small_kernel");
    return ACCBPG_OK;
}

size_t accbpg_dopt_abpg_small_smem_bytes(int m, int64_t n) {
    size_t bytes = 0;
    return small_pick_cluster(m, n, &bytes, true) ? bytes : 0;
}

int accbpg_dopt_abpg_small(void* ctx, void* stream, int driver, const double* H, int m, int64_t n, int64_t ldh,
                           double* x, double L, double gamma, int maxitrs, double epsilon, double eps_prox,
                           int theta_eq, int restart, int restart_rule, double G0, double ls_inc, double ls_dec,
                           int checkdiv, double* hist, double* info_out) {
    Ctx* c = (Ctx*)ctx;
    cudaStream_t s = (cudaStream_t)stream;
    if (!c || !H || !x || !hist || !info_out) return arg_err("dopt_abpg_small: NULL pointer");
    ACCBPG_ON_DEVICE(c);
    if (driver != ACCBPG_SMALL_DRV_ABPG && driver != ACCBPG_SMALL_DRV_ABPG_GAIN) return arg_err("dopt_abpg_small: driver");
    size_t smem = 0;
    const int C = small_pick_cluster(m, n, &smem, true);
    if (C == 0 || ldh < n)
        return arg_err("dopt_abpg_small: shape does not fit one SM (accbpg_dopt_abpg_small_smem_bytes)");
    auto pos = [](double v) { return isfinite(v) && v > 0.0; };
    if (!pos(L) || !pos(gamma) || !pos(G0) || !pos(ls_inc) || !pos(ls_dec) || !pos(eps_prox))
        return arg_err("dopt_abpg_small: L, gamma, G0, ls_inc, ls_dec, eps_prox must be finite and > 0");
    if (maxitrs < 1 || restart_rule < ACCBPG_SMALL_RESTART_NONE || restart_rule > ACCBPG_SMALL_RESTART_G)
        return arg_err("dopt_abpg_small: maxitrs, restart_rule");
    SmallAccParams p = {};
    p.H = H; p.m = m; p.n = (int)n; p.ldh = ldh; p.x = x; p.L = L; p.gamma = gamma; p.epsilon = epsilon;
    p.eps_prox = eps_prox; p.G0 = G0; p.ls_inc = ls_inc; p.ls_dec = ls_dec; p.maxitrs = maxitrs;
    p.theta_eq = theta_eq != 0; p.restart = restart != 0; p.rule = restart_rule; p.checkdiv = checkdiv != 0;
    p.hist = hist; p.info = info_out; p.status = c->d_status;
    int rc = driver == ACCBPG_SMALL_DRV_ABPG_GAIN ? small_acc_launch<ACCBPG_SMALL_DRV_ABPG_GAIN>(c, s, p, C, smem)
                                                  : small_acc_launch<ACCBPG_SMALL_DRV_ABPG>(c, s, p, C, smem);
    if (rc) return rc;
    ACCBPG_LAUNCHED("dopt_abpg_small_kernel");
    return ACCBPG_OK;
}

}  // extern "C"
