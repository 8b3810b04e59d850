// D-optimal design objective on sm_100a:  f(x) = -log det(H diag(x) H^T),  g_j = -h_j^T M^{-1} h_j
// (reference: DOptimalObj.func_grad, accbpg/functions.py:43-59).
//
//   K1  gram     M = H diag(x) H^T     FP64 DMMA (mma.sync m8n8k4) SYRK, lower 128x128 tiles, split over the
//                                      n (column) dimension, partials reduced in a fixed order (deterministic)
//   K2+K3 factor M = L L^T, L^{-1}     chol.cu: right-looking 64-block Cholesky whose launches also carry the block
//                                      forward substitution for L^{-1}; -log det from the pivots
//   K4  grad     g_j = -||Linv h_j||^2 DMMA triangular GEMM Linv*H streamed over column panels of H; the epilogue
//                                      squares and column-reduces the 128x128 tile, so M^{-1}H never exists in HBM
//
// Blackwell's tcgen05 tensor path has no FP64 kind, so FP64 tensor work is issued as warp-level DMMA.8x8x4
// (every f64 mma.sync shape lowers to that SASS on sm_100a) fed from shared memory through a 4-stage cp.async pipeline.
#include <cuda.h>
#include <cstdlib>
#include <map>
#include <tuple>
#include <vector>
#include "dmma.cuh"

namespace accbpg {

// ------------------------------------------------------------------------------------------ K1: SYRK
// Lower 128x128 tiles only.  Off-diagonal tiles use all 16 warps; in a diagonal tile the six warp tiles strictly above
// the diagonal are skipped, the four on the diagonal also skip their own strictly-upper 16x16 quarter (TMA kernel), and
// the ten that remain are numbered so that the four SM sub-partitions carry equal-ish DMMA counts (table below): a
// diagonal tile costs 9/16 of a full one (and stages its 128 rows of H once, as both operands).  The column range is
// split differently for the two kinds of tile so that every CTA carries about the same work.
struct SyrkParams {
    const double* H;
    const double* x;
    double* P;          // [split][mp][mp] partial tiles (lower tiles only are written)
    int m, mp, nt;
    int n_off;          // number of strictly-lower tiles
    int s_off, s_diag;  // column splits of an off-diagonal / a diagonal tile
    int diag_first;     // CTA order: the longer kind first
    int64_t n, ldh, kchunk_off, kchunk_diag;
    uint32_t* status;
};

// Warp -> warp tile of a diagonal CTA tile.  Warp id mod 4 is the SM sub-partition.  The six tiles below the diagonal
// cost 16 DMMAs per k-step, the four on it 10 (their strictly-upper 8x8 mma tiles are skipped; 12 in the cp.async
// fallback), so sub-partitions 0 and 1 get one full + two diagonal tiles (36) and sub-partitions 2 and 3 two full ones
// (32): a diagonal CTA tile costs 36/64 of a full one.
__constant__ signed char kDiagWm[16] = {1, 2, 2, 3, 0, 2, 3, 3, 1, 3, -1, -1, -1, -1, -1, -1};
__constant__ signed char kDiagWn[16] = {0, 0, 1, 1, 0, 2, 0, 2, 1, 3, -1, -1, -1, -1, -1, -1};

template <bool ALIGNED16>
__global__ void __launch_bounds__(GEMM_THREADS, 1) syrk_dmma_kernel(SyrkParams p) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    double* smem = reinterpret_cast<double*>(smem_raw);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int g = lane >> 2, t = lane & 3;

    // ---- which tile, which column chunk
    int b = blockIdx.x;
    const int n_off_ctas = p.n_off * p.s_off, n_diag_ctas = p.nt * p.s_diag;
    bool diag;
    if (p.diag_first) { diag = b < n_diag_ctas; if (!diag) b -= n_diag_ctas; }
    else              { diag = b >= n_off_ctas; if (diag) b -= n_off_ctas; }
    int bi, bj, split;
    int64_t kchunk;
    if (diag) {
        bi = bj = b % p.nt;
        split = b / p.nt;
        kchunk = p.kchunk_diag;
    } else {
        const int tt = b % p.n_off;                   // strictly-lower tile index -> (bi, bj), bi > bj
        split = b / p.n_off;
        bi = (int)((sqrt(8.0 * tt + 1.0) + 1.0) * 0.5);
        while (bi * (bi - 1) / 2 > tt) --bi;
        while ((bi + 1) * bi / 2 <= tt) ++bi;
        bj = tt - bi * (bi - 1) / 2;
        kchunk = p.kchunk_off;
    }
    int wm = warp >> 2, wn = warp & 3;
    if (diag) { wm = kDiagWm[warp]; wn = kDiagWn[warp]; }
    const bool active = wm >= 0;

    const int64_t k_begin = (int64_t)split * kchunk;
    int64_t k_end = k_begin + kchunk;
    if (k_end > p.n) k_end = p.n;
    const int KT = (k_end > k_begin) ? (int)((k_end - k_begin + BK - 1) / BK) : 0;

    double acc[MI][NI][2];
#pragma unroll
    for (int i = 0; i < MI; ++i)
#pragma unroll
        for (int j = 0; j < NI; ++j) acc[i][j][0] = acc[i][j][1] = 0.0;

    // Per-thread copy descriptors of the fast path (aligned, k-slab fully inside the chunk): the same 16-byte column
    // chunk of rows lr and lr+64 of the A block and of the B block.  Pointers advance by BK per k-slab.
    const int ch = tid & 7, lr = tid >> 3;
    const double* ga[2];
    const double* gb[2];
    int ba[2], bb[2];
#pragma unroll
    for (int i = 0; i < 2; ++i) {
        const int ra = bi * BM + lr + 64 * i, rb = bj * BN + lr + 64 * i;
        ba[i] = ra < p.m ? 16 : 0;
        bb[i] = rb < p.m ? 16 : 0;
        ga[i] = p.H + (int64_t)(ba[i] ? ra : 0) * p.ldh + k_begin + ch * 2;
        gb[i] = p.H + (int64_t)(bb[i] ? rb : 0) * p.ldh + k_begin + ch * 2;
    }
    const int soff = lr * A_LD + ch * 2;
    const int KT_full = (k_end > k_begin) ? (int)((k_end - k_begin) / BK) : 0;
    const int b_off = diag ? 0 : BM * A_LD;          // a diagonal tile reads its B operand from the A slab

    auto load_stage = [&](int stage, int kt) {
        double* As = smem + stage * KMAJOR_STAGE_DOUBLES;
        double* Bs = As + BM * A_LD;
        double* Xs = Bs + BN * A_LD;
        if (ALIGNED16 && kt < KT_full) {
            const int64_t ko = (int64_t)kt * BK;
#pragma unroll
            for (int i = 0; i < 2; ++i) {
                cp_async16(As + soff + i * 64 * A_LD, ga[i] + ko, ba[i]);
                if (!diag) cp_async16(Bs + soff + i * 64 * A_LD, gb[i] + ko, bb[i]);
            }
            if (tid < 8) cp_async16(Xs + tid * 2, p.x + k_begin + ko + tid * 2, 16);
            return;
        }
        const int64_t k0 = k_begin + (int64_t)kt * BK;
        load_kmajor_slab<ALIGNED16>(As, p.H, p.ldh, bi * BM, p.m, k0, k_end, tid);
        if (!diag) load_kmajor_slab<ALIGNED16>(Bs, p.H, p.ldh, bj * BN, p.m, k0, k_end, tid);
        if (ALIGNED16) {
            if (tid < 8) {
                int64_t gk = k0 + tid * 2;
                int64_t left = (k_end - gk) * 8;
                int bytes = left > 0 ? (left >= 16 ? 16 : 8) : 0;
                cp_async16(Xs + tid * 2, bytes ? (p.x + gk) : p.x, bytes);
            }
        } else {
            if (tid < 16) {
                int64_t gk = k0 + tid;
                int bytes = gk < k_end ? 8 : 0;
                cp_async8(Xs + tid, bytes ? (p.x + gk) : p.x, bytes);
            }
        }
    };

#pragma unroll
    for (int s = 0; s < STAGES - 1; ++s) {
        if (s < KT) load_stage(s, s);
        cp_async_commit();
    }

    bool neg = false;
    for (int kt = 0; kt < KT; ++kt) {
        cp_async_wait<STAGES - 2>();
        __syncthreads();
        {
            const int nk = kt + STAGES - 1;
            if (nk < KT) load_stage(nk % STAGES, nk);
            cp_async_commit();
        }
        if (active) {
            const double* As = smem + (kt % STAGES) * KMAJOR_STAGE_DOUBLES;
            const double* Xs = As + (BM + BN) * A_LD;
            const double* ap = As + (wm * 32 + g) * A_LD + t;
            const double* bp = As + b_off + (wn * 32 + g) * A_LD + t;
#pragma unroll
            for (int kk = 0; kk < BK / 4; ++kk) {
                const double xv = Xs[kk * 4 + t];
                neg |= (xv < 0.0);
                double a[MI], bq[NI];
#pragma unroll
                for (int i = 0; i < MI; ++i) a[i] = ap[i * 8 * A_LD + kk * 4];
#pragma unroll
                for (int j = 0; j < NI; ++j) bq[j] = bp[j * 8 * A_LD + kk * 4] * xv;      // diag(x) fused into the operand
#pragma unroll
                for (int i = 0; i < MI; ++i)
#pragma unroll
                    for (int j = 0; j < NI; ++j) dmma884(acc[i][j][0], acc[i][j][1], a[i], bq[j]);
            }
        }
    }
    cp_async_wait<0>();
    if (neg) atomicOr(p.status, ACCBPG_ST_X_NEGATIVE);
    if (!active) return;

    // partial tile -> workspace (mp is a multiple of 128: no bounds checks, 16-byte stores)
    double* P = p.P + (size_t)split * p.mp * p.mp;
#pragma unroll
    for (int i = 0; i < MI; ++i) {
        int row = bi * BM + wm * 32 + i * 8 + g;
#pragma unroll
        for (int j = 0; j < NI; ++j) {
            int col = bj * BN + wn * 32 + j * 8 + 2 * t;
            double2 v = make_double2(acc[i][j][0], acc[i][j][1]);
            *reinterpret_cast<double2*>(P + (size_t)row * p.mp + col) = v;
        }
    }
}

// ------------------------------------------------------------------------------------------ K1, TMA mainloop
// Same tiling and work split as syrk_dmma_kernel, with the operand traffic taken off the warps: one elected thread
// issues a 2-D TMA box (128 rows x 16 columns of H, 128-byte swizzle) per operand and a 1-D box of x per k-slab,
// completion is signalled on per-stage mbarriers (full / empty), and there is no CTA-wide barrier in the main loop.
// With the 128-byte swizzle the 16-byte chunk index of (row, k) is (k/2) ^ (row & 7).  A DMMA fragment read touches
// rows g = 0..3 and 32 contiguous bytes per row in a half warp, which would be a 2-way conflict under the natural row
// order; mma row g of tile i is therefore mapped to row 8i + 2(g&3) + (g>>2) of the warp tile (and the same for the
// columns of the output): a half warp then touches rows 0,2,4,6 (or 1,3,5,7) of an 8-row group and its eight
// (row, chunk) pairs land on eight distinct chunks, while every mma tile still covers 8 consecutive rows, so the
// diagonal warp tiles can drop their strictly-upper 8x8 mma tiles.
constexpr int TMA_STAGES = 6;
constexpr int TMA_PREFETCH = 4;                          // slabs in flight ahead of the consumers
constexpr int TMA_STAGE_BYTES = 2 * BM * BK * 8 + 1024;  // A box, B box, x slab (padded to keep 1024-byte alignment)
constexpr int TMA_SMEM = TMA_STAGES * TMA_STAGE_BYTES + 1024 /* alignment slack */ + 256 /* mbarriers */;

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
// consumer release of a stage it has only read: the reads are complete once the DMMAs that use them have issued, so no
// release fence is needed in front of the arrival (a release arrive shows up as membar stalls, one per warp and slab)
__device__ __forceinline__ void mbar_arrive_relaxed(uint32_t bar) {
    asm volatile("mbarrier.arrive.relaxed.cta.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
// bounded wait: a protocol error traps instead of hanging the GPU
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    uint32_t ok = 0;
    for (int spin = 0; spin < (1 << 21); ++spin) {
        asm volatile("{\n .reg .pred p;\n mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n selp.u32 %0, 1, 0, p;\n}\n"
                     : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
        if (ok) return;
    }
    __trap();
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const void* tmap, int c0, int c1, uint32_t bar) {
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
                 ::"r"(dst), "l"(tmap), "r"(c0), "r"(c1), "r"(bar) : "memory");
}
__device__ __forceinline__ void tma_load_1d(uint32_t dst, const void* tmap, int c0, uint32_t bar) {
    asm volatile("cp.async.bulk.tensor.1d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2}], [%3];"
                 ::"r"(dst), "l"(tmap), "r"(c0), "r"(bar) : "memory");
}
__device__ __forceinline__ double lds_f64(uint32_t addr) {
    double v;
    asm volatile("ld.shared.f64 %0, [%1];" : "=d"(v) : "r"(addr));
    return v;
}

__global__ void __launch_bounds__(GEMM_THREADS, 1)
syrk_tma_kernel(SyrkParams p, const __grid_constant__ CUtensorMap tmH, const __grid_constant__ CUtensorMap tmX) {
    extern __shared__ unsigned char smem_raw[];
    const uint32_t smem0 = ((uint32_t)__cvta_generic_to_shared(smem_raw) + 1023u) & ~1023u;      // 1024-byte aligned
    const uint32_t bars = smem0 + TMA_STAGES * TMA_STAGE_BYTES;      // full[0..S), empty[0..S): 8 bytes each
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int g = lane >> 2, t = lane & 3;

    int b = blockIdx.x;
    const int n_off_ctas = p.n_off * p.s_off, n_diag_ctas = p.nt * p.s_diag;
    bool diag;
    if (p.diag_first) { diag = b < n_diag_ctas; if (!diag) b -= n_diag_ctas; }
    else              { diag = b >= n_off_ctas; if (diag) b -= n_off_ctas; }
    int bi, bj, split;
    int64_t kchunk;
    if (diag) {
        bi = bj = b % p.nt;
        split = b / p.nt;
        kchunk = p.kchunk_diag;
    } else {
        const int tt = b % p.n_off;
        split = b / p.n_off;
        bi = (int)((sqrt(8.0 * tt + 1.0) + 1.0) * 0.5);
        while (bi * (bi - 1) / 2 > tt) --bi;
        while ((bi + 1) * bi / 2 <= tt) ++bi;
        bj = tt - bi * (bi - 1) / 2;
        kchunk = p.kchunk_off;
    }
    int wm = warp >> 2, wn = warp & 3;
    if (diag) { wm = kDiagWm[warp]; wn = kDiagWn[warp]; }
    const bool active = wm >= 0;
    const int n_active = diag ? 10 : 16;
    const bool diag_warp = diag && active && (wm == wn);

    const int64_t k_begin = (int64_t)split * kchunk;             // multiple of BK: chunk edges fall on slab edges
    int64_t k_end = k_begin + kchunk;
    if (k_end > p.n) k_end = p.n;
    const int KT = (k_end > k_begin) ? (int)((k_end - k_begin + BK - 1) / BK) : 0;

    if (tid == 0) {
        for (int s = 0; s < TMA_STAGES; ++s) {
            mbar_init(bars + 8 * s, 1);                          // full: the producer's arrive.expect_tx
            mbar_init(bars + 8 * (TMA_STAGES + s), n_active);    // empty: one arrival per consuming warp
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();

    const uint32_t stage_tx = (diag ? 1u : 2u) * BM * BK * 8 + BK * 8;
    auto issue = [&](int s) {                                    // one thread: arm the stage and launch its copies
        const int st = s % TMA_STAGES;
        const uint32_t base = smem0 + st * TMA_STAGE_BYTES, full = bars + 8 * st;
        const int kcol = (int)(k_begin + (int64_t)s * BK);
        mbar_arrive_expect_tx(full, stage_tx);
        tma_load_2d(base, &tmH, kcol, bi * BM, full);
        if (!diag) tma_load_2d(base + BM * BK * 8, &tmH, kcol, bj * BN, full);
        tma_load_1d(base + 2 * BM * BK * 8, &tmX, kcol, full);
    };
    if (tid == 0) {
        const int pre = KT < TMA_PREFETCH ? KT : TMA_PREFETCH;
        for (int s = 0; s < pre; ++s) issue(s);
    }

    double acc[MI][NI][2];
#pragma unroll
    for (int i = 0; i < MI; ++i)
#pragma unroll
        for (int j = 0; j < NI; ++j) acc[i][j][0] = acc[i][j][1] = 0.0;

    // per-thread byte offset inside a stage, with the swizzle term folded in
    //   element (row, k = 4kk + t):  row*128 + ((2kk + t/2) ^ (row & 7))*16 + (t & 1)*8 = base ^ (kk << 5)
    const int pg = 2 * (g & 3) + (g >> 2);                        // mma row g -> row pg of its 8-row group
    const int ra = (active ? wm : 0) * 32 + pg, rb = (active ? wn : 0) * 32 + pg;
    const uint32_t offA = ra * 128 + ((((t >> 1) ^ pg)) << 4) + (t & 1) * 8;
    const uint32_t offB = rb * 128 + ((((t >> 1) ^ pg)) << 4) + (t & 1) * 8 + (diag ? 0 : BM * BK * 8);

    bool neg = false;
    const bool check_x = (warp == 0);      // one warp sees every x of the chunk; the sign test stays off the FP64 pipe
    for (int s = 0; s < KT; ++s) {
        const int st = s % TMA_STAGES;
        const uint32_t base = smem0 + st * TMA_STAGE_BYTES;
        if (tid == 0) {                                          // keep TMA_PREFETCH slabs in flight
            const int sn = s + TMA_PREFETCH;
            if (sn < KT) {
                if (sn >= TMA_STAGES) mbar_wait(bars + 8 * (TMA_STAGES + sn % TMA_STAGES), ((sn / TMA_STAGES) + 1) & 1);
                issue(sn);
            }
        }
        if (active) {
            mbar_wait(bars + 8 * st, (s / TMA_STAGES) & 1);
            const uint32_t xs = base + 2 * BM * BK * 8 + t * 8;
            if (diag_warp) {
#pragma unroll
                for (int kk = 0; kk < BK / 4; ++kk) {
                    const double xv = lds_f64(xs + kk * 32);
                    if (check_x) neg |= (__double2hiint(xv) < 0) & (((__double2hiint(xv) & 0x7fffffff) | __double2loint(xv)) != 0);
                    double a[MI], bq[NI];
#pragma unroll
                    for (int i = 0; i < MI; ++i) a[i] = lds_f64(base + ((offA ^ (kk << 5)) + i * 8 * 128));
#pragma unroll
                    for (int j = 0; j < NI; ++j) bq[j] = lds_f64(base + ((offB ^ (kk << 5)) + j * 8 * 128)) * xv;
#pragma unroll
                    for (int i = 0; i < MI; ++i)
#pragma unroll
                        for (int j = 0; j < NI; ++j)
                            if (i >= j)                  // 8x8 mma tiles strictly above the diagonal are never read
                                dmma884(acc[i][j][0], acc[i][j][1], a[i], bq[j]);
                }
            } else {
#pragma unroll
                for (int kk = 0; kk < BK / 4; ++kk) {
                    const double xv = lds_f64(xs + kk * 32);
                    if (check_x) neg |= (__double2hiint(xv) < 0) & (((__double2hiint(xv) & 0x7fffffff) | __double2loint(xv)) != 0);
                    double a[MI], bq[NI];
#pragma unroll
                    for (int i = 0; i < MI; ++i) a[i] = lds_f64(base + ((offA ^ (kk << 5)) + i * 8 * 128));
#pragma unroll
                    for (int j = 0; j < NI; ++j) bq[j] = lds_f64(base + ((offB ^ (kk << 5)) + j * 8 * 128)) * xv;
#pragma unroll
                    for (int i = 0; i < MI; ++i)
#pragma unroll
                        for (int j = 0; j < NI; ++j) dmma884(acc[i][j][0], acc[i][j][1], a[i], bq[j]);
                }
            }
            __syncwarp();
            if (lane == 0) mbar_arrive_relaxed(bars + 8 * (TMA_STAGES + st));
        }
    }
    if (neg) atomicOr(p.status, ACCBPG_ST_X_NEGATIVE);
    if (!active) return;

    // partial tile -> workspace; rows and columns follow the permuted mma mapping
    double* P = p.P + (size_t)split * p.mp * p.mp;
#pragma unroll
    for (int i = 0; i < MI; ++i) {
        const int row = bi * BM + wm * 32 + 8 * i + pg;
#pragma unroll
        for (int j = 0; j < NI; ++j) {
#pragma unroll
            for (int e = 0; e < 2; ++e) {
                const int nn = 2 * t + e;
                const int col = bj * BN + wn * 32 + 8 * j + 2 * (nn & 3) + (nn >> 2);
                P[(size_t)row * p.mp + col] = acc[i][j][e];
            }
        }
    }
}

// M[i][j] = M[j][i] = sum_s P[s][i][j]  (i >= j), splits added in index order
__global__ void __launch_bounds__(256) syrk_reduce_kernel(const double* P, int s_off, int s_diag, int m, int mp,
                                                          double* M) {
    int j = blockIdx.x * 32 + (threadIdx.x & 31);
    int i = blockIdx.y * 8 + (threadIdx.x >> 5);
    if (i >= m || j > i) return;
    const int splits = ((i >> 7) == (j >> 7)) ? s_diag : s_off;
    const size_t off = (size_t)i * mp + j, sz = (size_t)mp * mp;
    double s = 0.0;
    for (int k = 0; k < splits; ++k) s += __ldcg(P + k * sz + off);
    M[(size_t)i * m + j] = s;
    M[(size_t)j * m + i] = s;
}

// ------------------------------------------------------------------------------------------ K1 + cross-GPU sum
// Column-sharded runs: the Gram matrix is the sum of the ranks' local ones.  Instead of an NCCL all-reduce after the
// split reduction, the reduction itself continues across the GPUs through NVLink peer memory (buffers from
// torch.distributed._symmetric_memory, every rank's mapped into every other rank's address space):
//   A  syrk_reduce_push_kernel: split sums stored into slot `rank` of every rank's receive buffer (remote stores);
//      the last CTA raises this rank's flag word on every rank
//   B  gram_sum_received_kernel: wait for the `world` flags, sum the received lower triangles in rank order -> M
// Every rank sums the same numbers in the same order: all ranks hold the same bits.  Flags carry a call counter (epoch),
// so nothing is ever reset; the receive buffer is double-buffered on the epoch's parity (a rank can be one call ahead of
// a peer that is still summing, never two); waits are bounded and trap on a protocol error.

constexpr int kMaxPeers = 16;
struct PeerGram {
    double* recv[kMaxPeers];                    // every rank's receive buffer: [2 (epoch parity)][world (sender)][m*m]
    unsigned long long* flags[kMaxPeers];       // every rank's flag words: [world (sender)], last epoch received
    int rank, world;
    unsigned long long epoch;
    int64_t total;                              // m*m
};


// Split reduction of the SYRK partials with the result pushed over NVLink: every thread sums the partial tiles of one
// lower-triangle element and stores it into slot `rank` of EVERY rank's receive buffer (posted remote stores, 256-byte
// runs along j); the last CTA to finish raises this rank's flag word on every rank.
__global__ void __launch_bounds__(256) syrk_reduce_push_kernel(const double* P, int s_off, int s_diag, int m, int mp,
                                                               PeerGram g, unsigned int* counter) {
    __shared__ bool sh_last;
    const int j = blockIdx.x * 32 + (threadIdx.x & 31);
    const int i = blockIdx.y * 8 + (threadIdx.x >> 5);
    if (i < m && j <= i) {
        const int splits = ((i >> 7) == (j >> 7)) ? s_diag : s_off;
        const size_t off = (size_t)i * mp + j, sz = (size_t)mp * mp;
        double s = 0.0;
        for (int k = 0; k < splits; ++k) s += __ldcg(P + k * sz + off);
        const size_t dst = ((size_t)(g.epoch & 1) * g.world + g.rank) * g.total + (size_t)i * m + j;
        for (int r = 0; r < g.world; ++r) {
            int q = g.rank + r;                    // start with the own buffer, then round-robin over the peers
            if (q >= g.world) q -= g.world;
            g.recv[q][dst] = s;
        }
    }
    __threadfence_system();                        // this CTA's remote stores are performed before its ticket
    __syncthreads();
    if (threadIdx.x == 0) {
        unsigned int t = atomicAdd(counter, 1u);
        sh_last = (t == gridDim.x * gridDim.y - 1);
        if (sh_last) *counter = 0u;
    }
    __syncthreads();
    if (sh_last) {
        __threadfence_system();
        if (threadIdx.x < g.world) st_release_sys(g.flags[threadIdx.x] + g.rank, g.epoch);
    }
}

// Waits until every rank's matrix of this epoch has arrived in the local receive buffer, then sums the `world` lower
// triangles in rank order (all ranks form bit-identical sums) and writes M with its mirror.
__global__ void __launch_bounds__(256) gram_sum_received_kernel(PeerGram g, int m, double* M) {
    if (threadIdx.x < g.world) {
        peer_flag_wait(g.flags[g.rank] + threadIdx.x, g.epoch);
    }
    __syncthreads();
    const int j = blockIdx.x * 32 + (threadIdx.x & 31);
    const int i = blockIdx.y * 8 + (threadIdx.x >> 5);
    if (i < m && j <= i) {
        const double* src = g.recv[g.rank] + (size_t)(g.epoch & 1) * g.world * g.total + (size_t)i * m + j;
        double s = 0.0;
        for (int r = 0; r < g.world; ++r) s += __ldcg(src + (size_t)r * g.total);   // L2: the slots are rewritten by peers
        M[(size_t)i * m + j] = s;
        M[(size_t)j * m + i] = s;
    }
}

// ------------------------------------------------------------------------------------------ K4: gradient
struct TrmmParams {
    const double* Linv;   // [mp][mp], zero above the diagonal
    const double* H;
    double* part;         // [nib][npad] partial column sums of squares
    int m, mp, nib;
    int64_t n, ldh, npad;
    // optional gate (persistent kernel only): tiles of a row block start once its rows of L^-1 are final in the data-flow
    // Cholesky chain that is still running (DfGate of dmma.cuh); ascending: walk row blocks lightest (= earliest) first
    const int* gate_fX = nullptr;
    const int* gate_fLi = nullptr;
    int gate_nb = 0, gate_epoch = 0, ascending = 0;
    // tail filler (persistent kernel only): the ascending list leaves out the last `hold0` panels of row block 0, the
    // descending list ends with them (`ext_cnt` = hold0 there).  A tile of the heaviest row blocks takes 50-67 us at
    // m = 500 against 17 us for row block 0, so the last wave of the gradient ends on short tiles instead of long ones.
    int hold0 = 0, ext_cnt = 0;
};

template <bool ALIGNED16>
__global__ void __launch_bounds__(GEMM_THREADS, 1) trmm_colnorm_kernel(TrmmParams p) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    double* smem = reinterpret_cast<double*>(smem_raw);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int g = lane >> 2, t = lane & 3;
    const int wm = warp >> 2, wn = warp & 3;
    const int ib = p.nib - 1 - blockIdx.x;            // heavy row blocks first
    const int64_t j0 = (int64_t)blockIdx.y * BN;
    int kmax = (ib + 1) * BM;                         // Linv is lower triangular: k <= row
    const int m16 = (p.m + BK - 1) / BK * BK;
    if (kmax > m16) kmax = m16;
    const int KT = kmax / BK;
    // inside the diagonal block of Linv a warp's 32 rows end at column ib*128 + wm*32 + 31: it stops issuing there
    // (each sub-partition hosts one warp of every wm, so the four pipes stay evenly loaded)
    const int klim = ib * BM + wm * 32 + 32;

    double acc[MI][NI][2];
#pragma unroll
    for (int i = 0; i < MI; ++i)
#pragma unroll
        for (int j = 0; j < NI; ++j) acc[i][j][0] = acc[i][j][1] = 0.0;

    auto load_stage = [&](int stage, int kt) {
        double* As = smem + stage * NN_STAGE_DOUBLES;
        double* Bs = As + BM * A_LD;
        // A: Linv rows ib*128.., cols k0..k0+15 (padded buffer: always in range, 16-byte aligned)
        load_kmajor_slab<true>(As, p.Linv, p.mp, ib * BM, p.mp, (int64_t)kt * BK, p.mp, tid);
        // B: H rows k0..k0+15 (rows >= m read as zero), cols j0..j0+127
        load_nmajor_slab<ALIGNED16>(Bs, p.H, p.ldh, kt * BK, p.m, j0, p.n, tid);
    };

#pragma unroll
    for (int s = 0; s < STAGES - 1; ++s) {
        if (s < KT) load_stage(s, s);
        cp_async_commit();
    }
    for (int kt = 0; kt < KT; ++kt) {
        cp_async_wait<STAGES - 2>();
        __syncthreads();
        {
            int nk = kt + STAGES - 1;
            if (nk < KT) load_stage(nk % STAGES, nk);
            cp_async_commit();
        }
        const double* As = smem + (kt % STAGES) * NN_STAGE_DOUBLES;
        int k4 = (klim - kt * BK) >> 2;
        k4 = k4 < 0 ? 0 : (k4 > BK / 4 ? BK / 4 : k4);
        mma_nn_slab(acc, As, As + BM * A_LD, wm, wn, g, t, k4);
    }
    cp_async_wait<0>();
    __syncthreads();      // pipeline buffers are dead: reuse the front of smem for the column exchange

    // epilogue: column sums of squares over this tile's 128 rows, fixed order
    double* colx = smem;                              // [4][128]
#pragma unroll
    for (int j = 0; j < NI; ++j) {
#pragma unroll
        for (int e = 0; e < 2; ++e) {
            double s = 0.0;
#pragma unroll
            for (int i = 0; i < MI; ++i) s = fma(acc[i][j][e], acc[i][j][e], s);
            s += __shfl_xor_sync(0xffffffffu, s, 4);
            s += __shfl_xor_sync(0xffffffffu, s, 8);
            s += __shfl_xor_sync(0xffffffffu, s, 16);
            if (g == 0) colx[wm * BN + wn * 32 + j * 8 + 2 * t + e] = s;
        }
    }
    __syncthreads();
    if (tid < BN) {
        int64_t col = j0 + tid;
        if (col < p.n)
            p.part[(size_t)ib * p.npad + col] = ((colx[tid] + colx[BN + tid]) + colx[2 * BN + tid]) + colx[3 * BN + tid];
    }
}

// ------------------------------------------------------------------------------------------ K4, TMA mainloop
// The stage layout of trmm_persistent_kernel; same tile and triangular stop as trmm_colnorm_kernel.  A (rows of Linv)
// arrives as one swizzled 2-D TMA box per k-slab, read with the permuted row mapping of syrk_tma_kernel (the column sums
// do not care which row is which); B (16 rows of the H panel, 1 KB each) arrives as sixteen 1-D bulk copies into rows
// padded to BT_LD doubles, so the B fragments keep the conflict-free padded addressing.  Rows k >= m of the last slab
// are not copied: Linv is zero in those columns, so whatever finite values the (zero-initialised) stage holds there
// contribute nothing.
constexpr int TRT_STAGES = 6;
constexpr int TRT_A_BYTES = BM * BK * 8;                                  // 16 KB, 1024-byte aligned
constexpr int TRT_B_BYTES = ((BK * BT_LD * 8 + 1023) / 1024) * 1024;      // 16 x 132 doubles, padded to 17 KB
constexpr int TRT_STAGE_BYTES = TRT_A_BYTES + TRT_B_BYTES;

__device__ __forceinline__ void bulk_load_1d(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(dst), "l"(src), "r"(bytes), "r"(bar) : "memory");
}

template <int K4>
__device__ __forceinline__ void trmm_tma_slab(double (&acc)[MI][NI][2], uint32_t base, const uint32_t (&offA)[2],
                                              uint32_t offB) {
#pragma unroll
    for (int kk = 0; kk < K4; ++kk) {
        double a[MI], bq[NI];
#pragma unroll
        for (int i = 0; i < MI; ++i) a[i] = lds_f64(base + ((offA[i & 1] ^ (kk << 5)) + (i >> 1) * 16 * 128));
#pragma unroll
        for (int j = 0; j < NI; ++j) bq[j] = lds_f64(base + offB + (kk * 4 * BT_LD + j * 8) * 8);
#pragma unroll
        for (int i = 0; i < MI; ++i)
#pragma unroll
            for (int j = 0; j < NI; ++j) dmma884(acc[i][j][0], acc[i][j][1], a[i], bq[j]);
    }
}

// ------------------------------------------------------------------------------------------ K4, persistent
// One CTA per SM walks a list of (row block, column panel) tiles fetched from a device counter, heaviest row blocks
// first, and the TMA ring keeps running across tile boundaries: the pipeline fill of a tile hides under the DMMAs of
// the previous one (a tile is only 8-32 k-slabs long at m = 500).  Each stage carries a small descriptor (row block,
// panel, k-slab, last-slab flag) written by the producer next to the data.  `first_tile` / `tile_limit` restrict a launch
// to part of the list, `grid` to part of the SMs.
struct TrmmTileMeta { int ib, panel, slab, flags; };      // flags: 1 = last slab of its tile, 2 = no more tiles
constexpr int TRP_SMEM = TRT_STAGES * TRT_STAGE_BYTES + 1024 + 256 + 4 * BN * 8 + TRT_STAGES * 16;
constexpr int TRP_THREADS = GEMM_THREADS + 32;          // 16 consuming warps + one producer warp

__global__ void __launch_bounds__(TRP_THREADS, 1)
trmm_persistent_kernel(TrmmParams p, const __grid_constant__ CUtensorMap tmL, int* tile_counter, int first_tile,
                       int tile_limit) {
    extern __shared__ unsigned char smem_raw[];
    const uint32_t smem0 = ((uint32_t)__cvta_generic_to_shared(smem_raw) + 1023u) & ~1023u;
    unsigned char* smem_gen = smem_raw + (smem0 - (uint32_t)__cvta_generic_to_shared(smem_raw));
    const uint32_t bars = smem0 + TRT_STAGES * TRT_STAGE_BYTES;
    double* colx = reinterpret_cast<double*>(smem_gen + TRT_STAGES * TRT_STAGE_BYTES + 256);      // [4][128]
    TrmmTileMeta* meta = reinterpret_cast<TrmmTileMeta*>(colx + 4 * BN);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int g = lane >> 2, t = lane & 3;
    const int wm = warp >> 2, wn = warp & 3;
    const int64_t npanels = (p.n + BN - 1) / BN;
    const int m16 = (p.m + BK - 1) / BK * BK;

    for (int st = 0; st < TRT_STAGES; ++st) {
        double* bz = reinterpret_cast<double*>(smem_gen + st * TRT_STAGE_BYTES + TRT_A_BYTES);
        for (int e = tid; e < BK * BT_LD; e += TRP_THREADS) bz[e] = 0.0;
    }
    if (tid == 0) {
        for (int s = 0; s < TRT_STAGES; ++s) {
            mbar_init(bars + 8 * s, 1);
            mbar_init(bars + 8 * (TRT_STAGES + s), GEMM_THREADS / 32);
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    __syncthreads();

    // ---- producer state (thread 0 only)
    int pr_ib = 0, pr_panel = 0, pr_slab = 0, pr_KT = 0;      // current tile being issued (pr_slab == pr_KT: need a new one)
    int issued = 0;                                           // stages issued so far (data or the final marker)
    bool pr_done = false;
    int pr_ready = -1;                                        // gated launch: row blocks <= pr_ready are known to be final
    auto gate_wait = [&](const int* f) {
        unsigned long long t0 = 0;
        unsigned spin = 0;
        for (;;) {
            int v;
            asm volatile("ld.acquire.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(f) : "memory");
            if ((v >> 8) == p.gate_epoch && (v & 255) >= 1) return;
            __nanosleep(200);
            if ((++spin & 0xffu) == 0) {
                unsigned long long now;
                asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(now));
                if (t0 == 0) t0 = now;
                else if (now - t0 > 2000000000ULL) __trap();
            }
        }
    };
    auto produce_one = [&]() {
        const int st = issued % TRT_STAGES;
        if (issued >= TRT_STAGES) mbar_wait(bars + 8 * (TRT_STAGES + st), ((issued / TRT_STAGES) + 1) & 1);
        const uint32_t full = bars + 8 * st;
        if (pr_slab == pr_KT) {                               // fetch the next tile
            const int tile = first_tile + atomicAdd(tile_counter, 1);
            if (tile >= tile_limit) {
                meta[st].flags = 2;
                mbar_arrive(full);
                pr_done = true;
                ++issued;
                return;
            }
            if (p.ascending) {
                const int first0 = (int)npanels - p.hold0;                 // tiles of row block 0 in this list
                if (tile < first0) { pr_ib = 0; pr_panel = tile; }
                else { const int t2 = tile - first0; pr_ib = 1 + (int)(t2 / npanels); pr_panel = (int)(t2 % npanels); }
            } else if (p.ext_cnt > 0 && tile >= tile_limit - p.ext_cnt) {   // the held-back panels of row block 0, last
                pr_ib = 0;
                pr_panel = (int)npanels - (tile_limit - tile);
            } else {
                pr_ib = p.nib - 1 - (int)(tile / npanels);                 // default: heaviest first
                pr_panel = (int)(tile % npanels);
            }
            if (p.gate_fX != nullptr && pr_ib > pr_ready) {   // rows of this row block of L^-1 final?  (64-row block rows 2ib, 2ib+1)
                for (int J = 2 * pr_ib; J <= 2 * pr_ib + 1 && J < p.gate_nb; ++J) {
                    gate_wait(p.gate_fX + J);
                    for (int r = 0; r < J; ++r) gate_wait(p.gate_fLi + J * p.gate_nb + r);
                }
                asm volatile("fence.proxy.async;" ::: "memory");      // generic-proxy acquire before the TMA reads of L^-1
                pr_ready = pr_ib;
            }
            int kmax = (pr_ib + 1) * BM;
            if (kmax > m16) kmax = m16;
            pr_KT = kmax / BK;
            pr_slab = 0;
        }
        const uint32_t base = smem0 + st * TRT_STAGE_BYTES;
        const int k0 = pr_slab * BK;
        const int64_t j0 = (int64_t)pr_panel * BN;
        int64_t ncols = p.n - j0;
        if (ncols > BN) ncols = BN;
        const uint32_t row_bytes = (uint32_t)ncols * 8;
        int rows = p.m - k0;
        rows = rows > BK ? BK : rows;
        meta[st].ib = pr_ib; meta[st].panel = pr_panel; meta[st].slab = pr_slab;
        meta[st].flags = (pr_slab + 1 == pr_KT) ? 1 : 0;
        mbar_arrive_expect_tx(full, TRT_A_BYTES + (uint32_t)rows * row_bytes);
        tma_load_2d(base, &tmL, k0, pr_ib * BM, full);
        const double* src = p.H + (int64_t)k0 * p.ldh + j0;
        for (int r = 0; r < rows; ++r)
            bulk_load_1d(base + TRT_A_BYTES + r * BT_LD * 8, src + (int64_t)r * p.ldh, row_bytes, full);
        ++pr_slab;
        ++issued;
    };

    if (warp == GEMM_THREADS / 32) {                          // the producer warp: one lane feeds the ring and leaves
        if (lane == 0)
            while (!pr_done) produce_one();
        return;
    }

    double acc[MI][NI][2];
#pragma unroll
    for (int i = 0; i < MI; ++i)
#pragma unroll
        for (int j = 0; j < NI; ++j) acc[i][j][0] = acc[i][j][1] = 0.0;
    uint32_t offA[2];
#pragma unroll
    for (int pq = 0; pq < 2; ++pq) {
        const int ra = wm * 32 + 2 * g + pq;
        offA[pq] = ra * 128 + ((((t >> 1) ^ (ra & 7))) << 4) + (t & 1) * 8;
    }
    const uint32_t offB = TRT_A_BYTES + (t * BT_LD + wn * 32 + g) * 8;

    for (int gs = 0;; ++gs) {
        const int st = gs % TRT_STAGES;
        mbar_wait(bars + 8 * st, (gs / TRT_STAGES) & 1);
        const TrmmTileMeta mt = meta[st];
        if (mt.flags & 2) break;
        const uint32_t base = smem0 + st * TRT_STAGE_BYTES;
        int k4 = (mt.ib * BM + wm * 32 + 32 - mt.slab * BK) >> 2;      // this warp's rows end at its own diagonal
        k4 = k4 < 0 ? 0 : (k4 > BK / 4 ? BK / 4 : k4);
        if (k4 == BK / 4) trmm_tma_slab<BK / 4>(acc, base, offA, offB);
        else if (k4 == 3) trmm_tma_slab<3>(acc, base, offA, offB);
        else if (k4 == 2) trmm_tma_slab<2>(acc, base, offA, offB);
        else if (k4 == 1) trmm_tma_slab<1>(acc, base, offA, offB);
        __syncwarp();
        if (lane == 0) mbar_arrive(bars + 8 * (TRT_STAGES + st));
        if (mt.flags & 1) {                                   // tile finished: column sums of squares, fixed order
#pragma unroll
            for (int j = 0; j < NI; ++j) {
#pragma unroll
                for (int e = 0; e < 2; ++e) {
                    double sq = 0.0;
#pragma unroll
                    for (int i = 0; i < MI; ++i) { sq = fma(acc[i][j][e], acc[i][j][e], sq); acc[i][j][e] = 0.0; }
                    sq += __shfl_xor_sync(0xffffffffu, sq, 4);
                    sq += __shfl_xor_sync(0xffffffffu, sq, 8);
                    sq += __shfl_xor_sync(0xffffffffu, sq, 16);
                    if (g == 0) colx[wm * BN + wn * 32 + j * 8 + 2 * t + e] = sq;
                }
            }
            asm volatile("bar.sync 1, %0;" ::"n"(GEMM_THREADS) : "memory");       // the 16 consuming warps only
            if (tid < BN) {
                const int64_t col = (int64_t)mt.panel * BN + tid;
                if (col < p.n)
                    p.part[(size_t)mt.ib * p.npad + col] =
                        ((colx[tid] + colx[BN + tid]) + colx[2 * BN + tid]) + colx[3 * BN + tid];
            }
            asm volatile("bar.sync 1, %0;" ::"n"(GEMM_THREADS) : "memory");
        }
    }
}

__global__ void __launch_bounds__(256) grad_finalize_kernel(const double* part, int nib, int64_t npad, int64_t n,
                                                            double* g) {
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; j < n; j += stride) {
        double s = 0.0;
        for (int b = 0; b < nib; ++b) s += __ldcg(part + (size_t)b * npad + j);
        g[j] = -s;
    }
}

// Gram matrix of a simplex vertex s (s = fill everywhere, s[i] = radius; functions_lmo.py:153-158) without a pass over H:
//   H diag(s) H^T = fill * (H H^T) + (radius - fill) * h_i h_i^T
// G = H H^T of the local columns is formed once per solve; the column index comes from the device slot the LMO wrote.
__global__ void __launch_bounds__(256) vertex_gram_kernel(const double* __restrict__ H, int m, int64_t n, int64_t ldh,
                                                          const double* __restrict__ G, double fill,
                                                          const double* __restrict__ d_idx, int64_t col_offset,
                                                          double radius, double* __restrict__ out) {
    const int64_t col = (int64_t)(*d_idx) - col_offset;
    const bool mine = (col >= 0 && col < n);
    const double w = radius - fill;
    const int64_t total = (int64_t)m * m, stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += stride) {
        const int r = (int)(e / m), c = (int)(e - (int64_t)r * m);
        double v = fill * G[e];
        if (mine) v = fma(w * __ldg(H + (int64_t)r * ldh + col), __ldg(H + (int64_t)c * ldh + col), v);
        out[e] = v;
    }
}

// ------------------------------------------------------------------------------------------ host side plan
struct DoptPlan {
    int mp, nt, n_off, nib;
    int s_off, s_diag, smax, diag_first;
    int64_t kchunk_off, kchunk_diag, npad;
    size_t off_P, off_Linv, off_Y, off_part, off_M, off_L, off_W, off_M2, off_W2, off_aux, off_aux2, total;
};

// Relative cost of a diagonal tile: 36/64 by DMMA count; its sub-partitions host only 2-3 active warps instead of 4,
// which hides less latency, so the effective figure is a little higher (calibrated on B200; ACCBPG_DIAG_COST overrides).
static double syrk_diag_cost() {
    static double v = -1.0;
    if (v < 0.0) { const char* e = getenv("ACCBPG_DIAG_COST"); v = e ? atof(e) : 0.5625; }
    return v;
}

// Makespan (in k-slab units) of the SYRK grid under in-order dispatch onto `sms` single-CTA SMs.
static double syrk_makespan(int n_off, int nt, int64_t ktiles, int s_off, int s_diag, int sms, int* diag_first) {
    const double ovh = 2.0, diag_cost = syrk_diag_cost();
    const double d_off = n_off ? (double)((ktiles + s_off - 1) / s_off) + ovh : 0.0;
    const double d_diag = (double)((ktiles + s_diag - 1) / s_diag) * diag_cost + ovh;
    const int c_off = n_off * s_off, c_diag = nt * s_diag;
    *diag_first = d_diag > d_off;
    std::vector<double> sm(sms, 0.0);      // min-heap emulated by a linear scan: sms <= a few hundred
    auto put = [&](int count, double d) {
        for (int i = 0; i < count; ++i) {
            int best = 0;
            for (int q = 1; q < sms; ++q) if (sm[q] < sm[best]) best = q;
            sm[best] += d;
        }
    };
    if (*diag_first) { put(c_diag, d_diag); put(c_off, d_off); }
    else             { put(c_off, d_off); put(c_diag, d_diag); }
    double mx = 0.0;
    for (double v : sm) mx = v > mx ? v : mx;
    return mx;
}

static DoptPlan make_plan(int m, int64_t n, int sm_count) {
    static std::map<std::tuple<int, int64_t, int>, DoptPlan> cache;
    auto key = std::make_tuple(m, n, sm_count);
    auto it = cache.find(key);
    if (it != cache.end()) return it->second;
    DoptPlan pl;
    pl.nt = (m + BM - 1) / BM;
    pl.mp = pl.nt * BM;
    pl.n_off = pl.nt * (pl.nt - 1) / 2;
    pl.nib = pl.nt;
    pl.npad = (n + 1) / 2 * 2;
    const int64_t ktiles = (n + BK - 1) / BK;
    int64_t max_splits = ktiles / 32;                 // at least 32 k-slabs (512 columns) per CTA
    if (max_splits < 1) max_splits = 1;
    if (max_splits > 64) max_splits = 64;
    pl.smax = (int)max_splits;                        // workspace is sized for the largest split count
    double best = 1e300;
    pl.s_off = pl.s_diag = 1; pl.diag_first = 0;
    for (int so = 1; so <= max_splits; ++so) {
        for (int d = -2; d <= 2; ++d) {
            int sd = (int)(syrk_diag_cost() * so + 0.5) + d;
            if (sd < 1 || sd > max_splits) continue;
            if ((int64_t)(pl.n_off * so + pl.nt * sd) > 6LL * sm_count) continue;
            int df = 0;
            double mk = syrk_makespan(pl.n_off, pl.nt, ktiles, so, sd, sm_count, &df);
            if (mk < best * (1.0 - 1e-9)) { best = mk; pl.s_off = so; pl.s_diag = sd; pl.diag_first = df; }
        }
    }
    pl.kchunk_off = (ktiles + pl.s_off - 1) / pl.s_off * BK;
    pl.kchunk_diag = (ktiles + pl.s_diag - 1) / pl.s_diag * BK;
    // layout: the m-only buffers first (their offsets do not depend on n_local), then the n-dependent ones
    const size_t mm = ((size_t)m * m * 8 + 255) / 256 * 256;
    size_t a = 0;
    pl.off_M = a;    a += mm;
    pl.off_L = a;    a += mm;
    pl.off_W = a;    a += mm;      // trailing matrix of the factorisation
    pl.off_M2 = a;   a += mm;      // second set: the value-only evaluation that runs on the side stream
    pl.off_W2 = a;   a += mm;
    pl.off_Linv = a; a += (size_t)pl.mp * pl.mp * 8;
    pl.off_Y = a;    a += (size_t)pl.mp * pl.mp * 8;      // running sums of the block forward substitution
    {   // progress counters + published diagonal inverses of the data-flow Cholesky chain, one set per concurrent chain
        const size_t ab = (chol_df_aux_bytes(m) + 255) / 256 * 256;
        pl.off_aux = a;  a += ab;
        pl.off_aux2 = a; a += ab;
    }
    pl.off_P = a;    a += (size_t)pl.smax * pl.mp * pl.mp * 8;
    pl.off_part = a; a += (size_t)pl.nib * pl.npad * 8;
    pl.total = a;
    cache[key] = pl;
    return pl;
}

static int device_sm_count() {
    int dev = 0, sms = 148;
    if (cudaGetDevice(&dev) == cudaSuccess) cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    return sms;
}

static bool g_attr_done[kMaxDevices] = {};       // the attribute is per device
static int ensure_smem_attrs() {
    int dev = 0;
    ACCBPG_CUDA(cudaGetDevice(&dev));
    if (dev >= 0 && dev < kMaxDevices && g_attr_done[dev]) return ACCBPG_OK;
    ACCBPG_CUDA(cudaFuncSetAttribute(syrk_dmma_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, KMAJOR_SMEM));
    ACCBPG_CUDA(cudaFuncSetAttribute(syrk_dmma_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, KMAJOR_SMEM));
    ACCBPG_CUDA(cudaFuncSetAttribute(syrk_tma_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, TMA_SMEM));
    ACCBPG_CUDA(cudaFuncSetAttribute(trmm_persistent_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, TRP_SMEM));
    ACCBPG_CUDA(cudaFuncSetAttribute(trmm_colnorm_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, NN_SMEM));
    ACCBPG_CUDA(cudaFuncSetAttribute(trmm_colnorm_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, NN_SMEM));
    if (dev >= 0 && dev < kMaxDevices) g_attr_done[dev] = true;
    return ACCBPG_OK;
}

static inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

// cuTensorMapEncodeTiled through the runtime's driver entry point (the library links no libcuda symbol directly)
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn encode_tiled_fn() {
    static EncodeTiledFn fn = nullptr;
    static bool tried = false;
    if (!tried) {
        tried = true;
        void* ptr = nullptr;
        cudaDriverEntryPointQueryResult qr = cudaDriverEntryPointSymbolNotFound;
        cudaError_t e = cudaGetDriverEntryPointByVersion("cuTensorMapEncodeTiled", &ptr, 12000, cudaEnableDefault, &qr);
        if (e == cudaSuccess && qr == cudaDriverEntryPointSuccess && ptr) fn = (EncodeTiledFn)ptr;
        if (getenv("ACCBPG_VERBOSE"))
            fprintf(stderr, "[accbpg] cuTensorMapEncodeTiled entry point: rc %d, query %d, ptr %p\n", (int)e, (int)qr, ptr);
    }
    return fn;
}

// A operand of trmm_persistent_kernel: L^-1 (mp x mp, ld mp) in 128-row x 16-column boxes with the 128-byte swizzle.
// False when the driver has no tensor-map entry point or the encoding fails.
static bool encode_linv_tmap(CUtensorMap* tmL, const double* Linv, int mp) {
    EncodeTiledFn fn = encode_tiled_fn();
    if (!fn) return false;
    cuuint64_t dimL[2] = {(cuuint64_t)mp, (cuuint64_t)mp};
    cuuint64_t strL[1] = {(cuuint64_t)mp * 8};
    cuuint32_t boxL[2] = {BK, BM};
    cuuint32_t one[2] = {1, 1};
    return fn(tmL, CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 2, (void*)Linv, dimL, strL, boxL, one, CU_TENSOR_MAP_INTERLEAVE_NONE,
              CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

// 2-D FP64 tensor map (no swizzle, zero fill outside) over a row-major matrix with `cols` columns, `rows` rows and leading
// dimension `ld`, box = box_cols x box_rows; for the other translation units (fw.cu).  `out` points to a CUtensorMap.
bool encode_tmap_f64_2d(void* out, const double* base, uint64_t cols, uint64_t rows, uint64_t ld, uint32_t box_cols,
                        uint32_t box_rows) {
    EncodeTiledFn fn = encode_tiled_fn();
    if (!fn || !aligned16(base) || (ld % 2) != 0 || (box_cols % 2) != 0 || box_cols > 256 || box_rows > 256) return false;
    cuuint64_t dim[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
    cuuint64_t str[1] = {(cuuint64_t)ld * 8};
    cuuint32_t box[2] = {box_cols, box_rows};
    cuuint32_t one[2] = {1, 1};
    return fn((CUtensorMap*)out, CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 2, (void*)base, dim, str, box, one,
              CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
              CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

// the same matrix seen as `groups` row groups of `rows` rows each (row g * rows + r of the matrix): one 3-D box moves
// box_rows rows of every group.  Only valid when groups * rows rows exist.
bool encode_tmap_f64_3d(void* out, const double* base, uint64_t cols, uint64_t rows, uint64_t groups, uint64_t ld,
                        uint32_t box_cols, uint32_t box_rows, uint32_t box_groups) {
    EncodeTiledFn fn = encode_tiled_fn();
    if (!fn || !aligned16(base) || (ld % 2) != 0 || (box_cols % 2) != 0 || box_cols > 256 || box_rows > 256 || box_groups > 256)
        return false;
    cuuint64_t dim[3] = {(cuuint64_t)cols, (cuuint64_t)rows, (cuuint64_t)groups};
    cuuint64_t str[2] = {(cuuint64_t)ld * 8, (cuuint64_t)rows * ld * 8};
    cuuint32_t box[3] = {box_cols, box_rows, box_groups};
    cuuint32_t one[3] = {1, 1, 1};
    return fn((CUtensorMap*)out, CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 3, (void*)base, dim, str, box, one,
              CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
              CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

size_t dopt_linv_offset(int m, int64_t n, int sm_count, int* mp_out) {
    DoptPlan pl = make_plan(m, n, sm_count);
    if (mp_out) *mp_out = pl.mp;
    return pl.off_Linv;
}

}  // namespace accbpg

using namespace accbpg;

extern "C" {

size_t accbpg_dopt_workspace_bytes(int m, int64_t n_local) {
    if (m < 1 || n_local < 1) return 0;
    return make_plan(m, n_local, device_sm_count()).total;
}

// the SYRK proper: partial tiles of every column split into the workspace
static int syrk_partials(Ctx* c, cudaStream_t s, const double* H, int m, int64_t n, int64_t ldh, const double* x, void* ws) {
    if (m < 1 || n < 1 || ldh < n) return arg_err("dopt_gram: shape");
    int rc = ensure_smem_attrs();
    if (rc) return rc;
    DoptPlan pl = make_plan(m, n, c->sm_count);
    SyrkParams p;
    p.H = H; p.x = x; p.P = (double*)((char*)ws + pl.off_P);
    p.m = m; p.mp = pl.mp; p.nt = pl.nt; p.n_off = pl.n_off; p.s_off = pl.s_off; p.s_diag = pl.s_diag;
    p.diag_first = pl.diag_first; p.n = n; p.ldh = ldh; p.kchunk_off = pl.kchunk_off; p.kchunk_diag = pl.kchunk_diag;
    p.status = c->d_status;
    dim3 grid(pl.n_off * pl.s_off + pl.nt * pl.s_diag);
    bool al = aligned16(H) && aligned16(x) && (ldh % 2 == 0);
    bool launched = false;
    if (al && encode_tiled_fn() && n < (1LL << 31)) {
        CUtensorMap tmH, tmX;
        cuuint64_t dimH[2] = {(cuuint64_t)n, (cuuint64_t)m};
        cuuint64_t strH[1] = {(cuuint64_t)ldh * 8};
        cuuint32_t boxH[2] = {BK, BM};
        cuuint32_t one[2] = {1, 1};
        cuuint64_t dimX[1] = {(cuuint64_t)n};
        cuuint32_t boxX[1] = {BK};
        CUresult r1 = encode_tiled_fn()(&tmH, CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 2, (void*)H, dimH, strH, boxH, one,
                                        CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                                        CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        CUresult r2 = encode_tiled_fn()(&tmX, CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 1, (void*)x, dimX, strH /* unused for rank 1 */, boxX, one,
                                        CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE,
                                        CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        static bool said = false;
        if (!said && getenv("ACCBPG_VERBOSE")) {
            said = true;
            fprintf(stderr, "[accbpg] SYRK: TMA mainloop, encode rc %d %d, grid %u (s_off %d, s_diag %d, diag_first %d)\n", (int)r1,
                    (int)r2, grid.x, pl.s_off, pl.s_diag, pl.diag_first);
        }
        if (r1 == CUDA_SUCCESS && r2 == CUDA_SUCCESS) {
            ProfScope ps(P_SYRK, s);
            syrk_tma_kernel<<<grid, GEMM_THREADS, TMA_SMEM, s>>>(p, tmH, tmX);
            launched = true;
        }
    }
    if (!launched) {
        static bool said2 = false;
        if (!said2 && getenv("ACCBPG_VERBOSE")) {
            said2 = true;
            fprintf(stderr, "[accbpg] SYRK: cp.async mainloop (aligned %d), grid %u (s_off %d, s_diag %d)\n", (int)al, grid.x, pl.s_off,
                    pl.s_diag);
        }
        ProfScope ps(P_SYRK, s);
        if (al) syrk_dmma_kernel<true><<<grid, GEMM_THREADS, KMAJOR_SMEM, s>>>(p);
        else    syrk_dmma_kernel<false><<<grid, GEMM_THREADS, KMAJOR_SMEM, s>>>(p);
    }
    ACCBPG_LAUNCHED("syrk_dmma_kernel");
    return ACCBPG_OK;
}

int accbpg_dopt_gram(void* ctx, void* stream, const double* H, int m, int64_t n, int64_t ldh, const double* x,
                     void* ws, double* M) {
    Ctx* c = (Ctx*)ctx;
    cudaStream_t s = (cudaStream_t)stream;
    if (!c || !H || !x || !ws || !M) return arg_err("dopt_gram: NULL pointer");
    ACCBPG_ON_DEVICE(c);
    int rc = syrk_partials(c, s, H, m, n, ldh, x, ws);
    if (rc) return rc;
    DoptPlan pl = make_plan(m, n, c->sm_count);
    const double* Pp = (const double*)((char*)ws + pl.off_P);
    dim3 rg((m + 31) / 32, (m + 7) / 8);
    {
        ProfScope ps(P_SYRK_REDUCE, s);
        syrk_reduce_kernel<<<rg, 256, 0, s>>>(Pp, pl.s_off, pl.s_diag, m, pl.mp, M);
    }
    ACCBPG_LAUNCHED("syrk_reduce_kernel");
    return ACCBPG_OK;
}

int accbpg_dopt_gram_allreduce(void* ctx, void* stream, const double* H, int m, int64_t n, int64_t ldh, const double* x,
                               void* ws, int rank, int world, void* const* peer_recv, void* const* peer_flags,
                               uint64_t epoch, double* M) {
    Ctx* c = (Ctx*)ctx;
    cudaStream_t s = (cudaStream_t)stream;
    if (!c || !H || !x || !ws || !M || !peer_recv || !peer_flags) return arg_err("dopt_gram_allreduce: NULL pointer");
    ACCBPG_ON_DEVICE(c);
    if (world < 1 || world > kMaxPeers || rank < 0 || rank >= world) return arg_err("dopt_gram_allreduce: rank / world");
    if (m < 1 || n < 1 || ldh < n || epoch < 1) return arg_err("dopt_gram_allreduce: shape / epoch");
    PeerGram g;
    for (int r = 0; r < world; ++r) {
        g.recv[r] = (double*)peer_recv[r];
        g.flags[r] = (unsigned long long*)peer_flags[r];
        if (!g.recv[r] || !g.flags[r]) return arg_err("dopt_gram_allreduce: NULL peer pointer");
    }
    g.rank = rank; g.world = world; g.epoch = epoch;
    g.total = (int64_t)m * m;
    // the SYRK itself: partial tiles into the workspace (the pushing split reduction replaces syrk_reduce_kernel)
    int rc = syrk_partials(c, s, H, m, n, ldh, x, ws);
    if (rc) return rc;
    DoptPlan pl = make_plan(m, n, c->sm_count);
    const double* P = (const double*)((char*)ws + pl.off_P);
    dim3 rg((m + 31) / 32, (m + 7) / 8);
    {
        ProfScope ps(P_GRAM_PUSH, s);
        syrk_reduce_push_kernel<<<rg, 256, 0, s>>>(P, pl.s_off, pl.s_diag, m, pl.mp, g, c->d_counter + 16);
        ACCBPG_LAUNCHED("syrk_reduce_push_kernel");
    }
    {
        ProfScope ps(P_GRAM_SUM, s);          // includes the wait for the slowest rank's push
        gram_sum_received_kernel<<<rg, 256, 0, s>>>(g, m, M);
        ACCBPG_LAUNCHED("gram_sum_received_kernel");
    }
    return ACCBPG_OK;
}

int accbpg_dopt_vertex_gram(void* ctx, void* stream, const double* H, int m, int64_t n, int64_t ldh, const double* G,
                            double fill, const double* d_idx, int64_t col_offset, double radius, double* out) {
    Ctx* c = (Ctx*)ctx;
    cudaStream_t s = (cudaStream_t)stream;
    if (!c || !H || !G || !d_idx || !out) return arg_err("dopt_vertex_gram: NULL pointer");
    ACCBPG_ON_DEVICE(c);
    if (m < 1 || n < 1 || ldh < n) return arg_err("dopt_vertex_gram: shape");
    int grid = grid_for(c, (int64_t)m * m, 256, 2, 8);
    vertex_gram_kernel<<<grid, 256, 0, s>>>(H, m, n, ldh, G, fill, d_idx, col_offset, radius, out);
    ACCBPG_LAUNCHED("vertex_gram_kernel");
    return ACCBPG_OK;
}

int accbpg_dopt_factor(void* ctx, void* stream, int m, const double* M, double* L, int want_inverse, void* ws,
                       double* d_out) {
    Ctx* c = (Ctx*)ctx;
    cudaStream_t s = (cudaStream_t)stream;
    if (!c || !M || !ws || !d_out) return arg_err("dopt_factor: NULL pointer");
    ACCBPG_ON_DEVICE(c);
    if (m < 1) return arg_err("dopt_factor: m");
    if (M == L) return arg_err("dopt_factor: in-place factorisation is not supported");
    // the factor scratch lives in the m-only head of the workspace (independent of n_local)
    DoptPlan pl = make_plan(m, 2, c->sm_count);
    double* W = (double*)((char*)ws + pl.off_W);
    if (M == W || L == W) return arg_err("dopt_factor: M / L alias the factor scratch");
    return chol_factor_inv(c, s, m, pl.mp, M, L, want_inverse ? 1 : 0, (double*)((char*)ws + pl.off_Linv), W,
                           (double*)((char*)ws + pl.off_Y), c->d_slots + 248, d_out, (char*)ws + pl.off_aux);
}

int accbpg_dopt_grad(void* ctx, void* stream, const double* H, int m, int64_t n, int64_t ldh, void* ws, double* g) {
    Ctx* c = (Ctx*)ctx;
    cudaStream_t s = (cudaStream_t)stream;
    if (!c || !H || !ws || !g) return arg_err("dopt_grad: NULL pointer");
    ACCBPG_ON_DEVICE(c);
    if (m < 1 || n < 1 || ldh < n) return arg_err("dopt_grad: shape");
    int rc = ensure_smem_attrs();
    if (rc) return rc;
    DoptPlan pl = make_plan(m, n, c->sm_count);
    double* Linv = (double*)((char*)ws + pl.off_Linv);      // left there by accbpg_dopt_factor(want_inverse = 1)
    double* part = (double*)((char*)ws + pl.off_part);
    TrmmParams p;
    p.Linv = Linv; p.H = H; p.part = part; p.m = m; p.mp = pl.mp; p.nib = pl.nib;
    p.n = n; p.ldh = ldh; p.npad = pl.npad;
    int64_t npanels = (n + BN - 1) / BN;
    if (npanels > 65535) return arg_err("dopt_grad: n_local too large for one launch (max 65535*128 columns)");
    const int64_t ntiles = (int64_t)pl.nib * npanels;
    if (ntiles >= (1LL << 30)) return arg_err("dopt_grad: m x n_local too large for one launch (2^30 128x128 tiles)");
    const bool al = aligned16(H) && (ldh % 2 == 0);
    CUtensorMap tmL;
    if (al && (n % 2 == 0) && encode_linv_tmap(&tmL, Linv, pl.mp)) {
        int* counter = (int*)(c->d_counter + 8);      // a second ticket word of the context
        ACCBPG_CUDA(cudaMemsetAsync(counter, 0, sizeof(int), s));
        const int pgrid = (int)(ntiles < c->sm_count ? ntiles : c->sm_count);
        ProfScope ps(P_TRMM, s);
        trmm_persistent_kernel<<<pgrid, TRP_THREADS, TRP_SMEM, s>>>(p, tmL, counter, 0, (int)ntiles);
    } else {
        const dim3 grid(pl.nib, (unsigned)npanels);
        ProfScope ps(P_TRMM, s);
        if (al) trmm_colnorm_kernel<true><<<grid, GEMM_THREADS, NN_SMEM, s>>>(p);
        else    trmm_colnorm_kernel<false><<<grid, GEMM_THREADS, NN_SMEM, s>>>(p);
    }
    ACCBPG_LAUNCHED("trmm_colnorm_kernel");
    int fg = grid_for(c, n, 256, 2, 8);
    {
        ProfScope ps(P_GRAD_FIN, s);
        grad_finalize_kernel<<<fg, 256, 0, s>>>(part, pl.nib, pl.npad, n, g);
    }
    ACCBPG_LAUNCHED("grad_finalize_kernel");
    return ACCBPG_OK;
}

// Factor M (with the inverse) and form the gradient, with the triangular GEMM started before the Cholesky chain has
// finished: the rows of row block ib of L^{-1} are final once block column 2ib+1 has retired, and the chain keeps only
// a few SMs busy.  With the data-flow chain, the first n_early row blocks are one persistent launch on a second stream
// (on the SMs the chains do not need: `reserve` below) whose producer waits on the chain's progress counters before it
// loads a row block of L^{-1}, lowest row blocks first; the remaining row blocks follow on the main stream after the
// chain, heaviest first, on all SMs.  Same results as accbpg_dopt_factor + accbpg_dopt_grad, which is the route taken
// whenever the overlap cannot run (one launch per block column in the chain, unaligned or odd-width H, one row block).
static int overlap_enabled() {          // read on every call: tools/bench_configs.py times the kernels one by one with it off
    const char* e = getenv("ACCBPG_OVERLAP");
    return (e && e[0] == '0') ? 0 : 1;
}

static int dopt_factor_grad(Ctx* c, cudaStream_t s, const double* H, int m, int64_t n, int64_t ldh, const double* M,
                            void* ws, double* d_f_out, double* g) {
    DoptPlan pl = make_plan(m, n, c->sm_count);
    const int64_t npanels = (n + BN - 1) / BN;
    const int64_t ntiles = (int64_t)pl.nib * npanels;
    const bool al = aligned16(H) && (ldh % 2 == 0) && (n % 2 == 0);
    static int early_env = -2;
    if (early_env == -2) { const char* e = getenv("ACCBPG_EARLY_BLOCKS"); early_env = e ? atoi(e) : -1; }
    int n_early = pl.nib / 2 < 4 ? pl.nib / 2 : 4;            // row blocks 0 .. n_early-1 start under the chain
    if (early_env >= 0) n_early = early_env < pl.nib - 1 ? early_env : pl.nib - 1;
    double* Linv = (double*)((char*)ws + pl.off_Linv);
    double* part = (double*)((char*)ws + pl.off_part);
    CUtensorMap tmL;
    if (!overlap_enabled() || !al || !chol_df_enabled(m) || n_early < 1 || ntiles >= (1LL << 30) ||
        !encode_linv_tmap(&tmL, Linv, pl.mp)) {
        int rc = accbpg_dopt_factor(c, s, m, M, nullptr, 1, ws, d_f_out);
        if (rc) return rc;
        return accbpg_dopt_grad(c, s, H, m, n, ldh, ws, g);
    }
    int rc = ensure_smem_attrs();
    if (rc) return rc;
    TrmmParams p;
    p.Linv = Linv; p.H = H; p.part = part; p.m = m; p.mp = pl.mp; p.nib = pl.nib; p.n = n; p.ldh = ldh; p.npad = pl.npad;
    int* counters = (int*)(c->d_counter + 8);                 // words 8 (late launch) and 9 (early launch) of the ticket block
    ACCBPG_CUDA(cudaMemsetAsync(counters, 0, 2 * sizeof(int), s));
    // SMs left to the Cholesky chains while they run.  Up to 8 block columns each chain is a spine CTA (an SM of its own)
    // and DF_SMALL_WORKERS workers at two per SM; two chains run at once (f(x) on the side stream, this one), so 2 * (1 +
    // 8) SMs and two spare (500x50000 ABPG: 1.116 -> 1.085 ms per iteration against 52, B200).  Larger chains keep 52.
    static int reserve_env = -2;
    if (reserve_env == -2) { const char* e = getenv("ACCBPG_CHAIN_SMS"); reserve_env = e ? atoi(e) : -1; }
    const int reserve = reserve_env >= 0 ? reserve_env
                                         : ((m + 63) / 64 <= 8 ? 2 * (1 + DF_SMALL_WORKERS / 2) + 2 : 52);
    int early_grid = c->sm_count - reserve;
    if (early_grid < 1) early_grid = 1;
    if ((int64_t)early_grid > npanels) early_grid = (int)npanels;
    // side2 must not start before the main stream has reached this point (counters, earlier readers of part)
    ACCBPG_CUDA(cudaEventRecord(c->ev_fork, s));
    ACCBPG_CUDA(cudaStreamWaitEvent(c->side2, c->ev_fork, 0));
    ProfScope ps_all(P_TRINV, s);                             // chain + triangular GEMM as one interval
    DfGate gate;
    rc = chol_factor_inv(c, s, m, pl.mp, M, nullptr, 1, Linv, (double*)((char*)ws + pl.off_W),
                         (double*)((char*)ws + pl.off_Y), c->d_slots + 248, d_f_out, (char*)ws + pl.off_aux, &gate);
    if (rc) return rc;
    TrmmParams pe = p;
    pe.gate_fX = gate.fX; pe.gate_fLi = gate.fLi; pe.gate_nb = gate.nb; pe.gate_epoch = gate.epoch; pe.ascending = 1;
    // panels of row block 0 kept for the end of the late launch (ACCBPG_TRMM_HOLD, per cent of the panels; only when the
    // tiles are long against the whole gradient, i.e. few tiles per SM: at m = 2000 a tile is 0.2 % of an SM's share)
    static int hold_pct = -1;
    if (hold_pct < 0) { const char* e = getenv("ACCBPG_TRMM_HOLD"); hold_pct = e ? atoi(e) : 35; if (hold_pct < 0 || hold_pct > 90) hold_pct = 0; }
    int hold0 = 0;
    if (n_early >= 2 && ntiles < 64LL * c->sm_count) hold0 = (int)(npanels * hold_pct / 100);
    pe.hold0 = hold0;
    trmm_persistent_kernel<<<early_grid, TRP_THREADS, TRP_SMEM, c->side2>>>(pe, tmL, counters + 1, 0, (int)(n_early * npanels) - hold0);
    ACCBPG_LAUNCHED("trmm_persistent_kernel");
    ACCBPG_CUDA(cudaEventRecord(c->ev_early_done, c->side2));
    const int limit = (int)((pl.nib - n_early) * npanels) + hold0;
    const int pgrid = (int)((int64_t)c->sm_count < (int64_t)limit ? c->sm_count : limit);
    TrmmParams pl2 = p;
    pl2.ext_cnt = hold0;
    trmm_persistent_kernel<<<pgrid, TRP_THREADS, TRP_SMEM, s>>>(pl2, tmL, counters, 0, limit);
    ACCBPG_LAUNCHED("trmm_persistent_kernel");
    ACCBPG_CUDA(cudaStreamWaitEvent(s, c->ev_early_done, 0));
    int fg = grid_for(c, n, 256, 2, 8);
    grad_finalize_kernel<<<fg, 256, 0, s>>>(part, pl.nib, pl.npad, n, g);
    ACCBPG_LAUNCHED("grad_finalize_kernel");
    return ACCBPG_OK;
}

int accbpg_dopt_func_grad(void* ctx, void* stream, const double* H, int m, int64_t n, int64_t ldh, const double* x,
                          int flag, void* ws, double* d_f_out, double* g) {
    Ctx* c = (Ctx*)ctx;
    if (!c || !ws) return arg_err("dopt_func_grad: NULL pointer");
    ACCBPG_ON_DEVICE(c);
    if (flag < 0 || flag > 2) return arg_err("dopt_func_grad: flag");
    if (flag >= 1 && !g) return arg_err("dopt_func_grad: gradient buffer is NULL");
    DoptPlan pl = make_plan(m, n, c->sm_count);
    double* M = (double*)((char*)ws + pl.off_M);
    int rc = accbpg_dopt_gram(ctx, stream, H, m, n, ldh, x, ws, M);
    if (rc) return rc;
    if (flag >= 1) return dopt_factor_grad(c, (cudaStream_t)stream, H, m, n, ldh, M, ws, d_f_out ? d_f_out : (c->d_slots + 249), g);
    return accbpg_dopt_factor(ctx, stream, m, M, NULL, 0, ws, d_f_out ? d_f_out : (c->d_slots + 249));
}

// -log det M (value only) on the context's side stream, started after the work queued so far on s; ev_join marks
// its end.  Uses the second set of factor buffers (off_W2, off_aux2), so it can run next to a factorisation on s.
static int value_on_side(Ctx* c, cudaStream_t s, const DoptPlan& pl, int m, const double* M, void* ws, double* d_out) {
    ACCBPG_CUDA(cudaEventRecord(c->ev_fork, s));
    ACCBPG_CUDA(cudaStreamWaitEvent(c->side, c->ev_fork, 0));
    int rc = chol_factor_inv(c, c->side, m, pl.mp, M, NULL, 0, NULL, (double*)((char*)ws + pl.off_W2), NULL,
                             c->d_slots + 246, d_out, (char*)ws + pl.off_aux2);
    if (rc) return rc;
    ACCBPG_CUDA(cudaEventRecord(c->ev_join, c->side));
    return ACCBPG_OK;
}

// f(xf) and (f(yg), grad f(yg)) in one call: the two Gram matrices are formed back to back on the main stream, then
// the value-only Cholesky runs on the context's side stream while the main stream factors M(yg), inverts L and
// streams the gradient.  Both chains are latency bound on a handful of SMs, so they overlap almost completely.
int accbpg_dopt_pair(void* ctx, void* stream, const double* H, int m, int64_t n, int64_t ldh, const double* xf,
                     const double* yg, int flag_y, void* ws, double* d_fx_out, double* d_fy_out, double* g) {
    Ctx* c = (Ctx*)ctx;
    cudaStream_t s = (cudaStream_t)stream;
    if (!c || !ws || !xf || !yg || !d_fx_out) return arg_err("dopt_pair: NULL pointer");
    ACCBPG_ON_DEVICE(c);
    if (flag_y < 1 || flag_y > 2 || !g) return arg_err("dopt_pair: flag_y must be 1 or 2 with a gradient buffer");
    DoptPlan pl = make_plan(m, n, c->sm_count);
    double* M1 = (double*)((char*)ws + pl.off_M);
    double* M2 = (double*)((char*)ws + pl.off_M2);
    int rc = accbpg_dopt_gram(ctx, stream, H, m, n, ldh, xf, ws, M2);
    if (rc) return rc;
    rc = value_on_side(c, s, pl, m, M2, ws, d_fx_out);
    if (rc) return rc;
    rc = accbpg_dopt_gram(ctx, stream, H, m, n, ldh, yg, ws, M1);
    if (rc) return rc;
    rc = dopt_factor_grad(c, s, H, m, n, ldh, M1, ws, d_fy_out ? d_fy_out : (c->d_slots + 249), g);
    if (rc) return rc;
    ACCBPG_CUDA(cudaStreamWaitEvent(s, c->ev_join, 0));
    return ACCBPG_OK;
}

// Same, starting from Gram matrices the caller already holds (M is linear in x, so the drivers can form
// M((1-t)x + t z) = (1-t)M(x) + t M(z) instead of running another SYRK).  Mx may be NULL (gradient side only).
int accbpg_dopt_pair_from_gram(void* ctx, void* stream, const double* H, int m, int64_t n, int64_t ldh,
                               const double* Mx, const double* My, int flag_y, void* ws, double* d_fx_out,
                               double* d_fy_out, double* g) {
    Ctx* c = (Ctx*)ctx;
    cudaStream_t s = (cudaStream_t)stream;
    if (!c || !ws || !My) return arg_err("dopt_pair_from_gram: NULL pointer");
    ACCBPG_ON_DEVICE(c);
    if (flag_y < 0 || flag_y > 2 || (flag_y >= 1 && !g)) return arg_err("dopt_pair_from_gram: flag_y / gradient buffer");
    if (Mx && !d_fx_out) return arg_err("dopt_pair_from_gram: d_fx_out is NULL");
    DoptPlan pl = make_plan(m, n, c->sm_count);
    int rc;
    if (Mx) {
        rc = value_on_side(c, s, pl, m, Mx, ws, d_fx_out);
        if (rc) return rc;
    }
    if (flag_y >= 1) rc = dopt_factor_grad(c, s, H, m, n, ldh, My, ws, d_fy_out ? d_fy_out : (c->d_slots + 249), g);
    else rc = accbpg_dopt_factor(ctx, stream, m, My, NULL, 0, ws, d_fy_out ? d_fy_out : (c->d_slots + 249));
    if (rc) return rc;
    if (Mx) ACCBPG_CUDA(cudaStreamWaitEvent(s, c->ev_join, 0));
    return ACCBPG_OK;
}

}  // extern "C"
