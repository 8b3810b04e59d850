// FP64 tensor-core (DMMA.8x8x4) tile machinery shared by the SYRK and the triangular GEMM: 128x128 CTA tile,
// 16 warps (4 x 4, four per SM sub-partition so the DMMA pipe always has a ready warp), warp tile 32x32 = 4x4
// mma.sync.m8n8k4 tiles, k-slabs of 16 staged through a 4-deep cp.async pipeline into padded (bank-conflict-free)
// shared memory.
#pragma once
#include "common.cuh"

namespace accbpg {

constexpr int BM = 128;            // CTA tile rows
constexpr int BN = 128;            // CTA tile cols
constexpr int BK = 16;             // k-slab per pipeline stage
constexpr int STAGES = 4;
constexpr int GEMM_THREADS = 512;  // 16 warps: 4 (rows) x 4 (cols)
constexpr int A_LD = BK + 4;       // 20 doubles: (g*20 + t) mod 16 distinct over a half warp -> conflict-free LDS.64
constexpr int BT_LD = BN + 4;      // 132 doubles for a k-major B tile: (t*132 + g) mod 16 distinct
constexpr int MI = 4, NI = 4;       // warp tile 32 x 32

constexpr int KMAJOR_STAGE_DOUBLES = BM * A_LD + BN * A_LD + BK;   // A[i][k], B[j][k], x[k]      (SYRK)
constexpr int KMAJOR_SMEM = STAGES * KMAJOR_STAGE_DOUBLES * 8;
constexpr int NN_STAGE_DOUBLES = BM * A_LD + BK * BT_LD;           // A[i][k], B[k][j]            (GEMM "NN")
constexpr int NN_SMEM = STAGES * NN_STAGE_DOUBLES * 8;

#ifdef __CUDACC__
__device__ __forceinline__ void cp_async16(void* smem, const void* gmem, int src_bytes) {
    unsigned sa = (unsigned)__cvta_generic_to_shared(smem);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;\n" ::"r"(sa), "l"(gmem), "r"(src_bytes) : "memory");
}
__device__ __forceinline__ void cp_async8(void* smem, const void* gmem, int src_bytes) {
    unsigned sa = (unsigned)__cvta_generic_to_shared(smem);
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8, %2;\n" ::"r"(sa), "l"(gmem), "r"(src_bytes) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;\n" ::"n"(N) : "memory"); }

__device__ __forceinline__ void dmma884(double& c0, double& c1, double a, double b) {
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n"
                 : "+d"(c0), "+d"(c1)
                 : "d"(a), "d"(b));
}

// [128 rows x 16 k] slab, k contiguous in global memory -> smem rows of A_LD doubles; rows >= row_limit and
// columns >= k_limit are zero-filled (cp.async src-size 0).  row0 / k0 are offsets relative to `src`.
template <bool ALIGNED16>
__device__ __forceinline__ void load_kmajor_slab(double* dst, const double* src, int64_t ld, int row0, int row_limit,
                                                 int64_t k0, int64_t k_limit, int tid) {
    if (ALIGNED16) {
#pragma unroll
        for (int i = 0; i < (BM * BK / 2) / GEMM_THREADS; ++i) {
            int c = tid + i * GEMM_THREADS;
            int row = c >> 3, ch = c & 7;
            int grow = row0 + row;
            int64_t gcol = k0 + ch * 2;
            int64_t left = (k_limit - gcol) * 8;
            int bytes = (grow < row_limit && left > 0) ? (left >= 16 ? 16 : 8) : 0;
            const double* s = bytes ? (src + (int64_t)grow * ld + gcol) : src;
            cp_async16(dst + row * A_LD + ch * 2, s, bytes);
        }
    } else {
#pragma unroll
        for (int i = 0; i < (BM * BK) / GEMM_THREADS; ++i) {
            int c = tid + i * GEMM_THREADS;
            int row = c >> 4, col = c & 15;
            int grow = row0 + row;
            int64_t gcol = k0 + col;
            int bytes = (grow < row_limit && gcol < k_limit) ? 8 : 0;
            const double* s = bytes ? (src + (int64_t)grow * ld + gcol) : src;
            cp_async8(dst + row * A_LD + col, s, bytes);
        }
    }
}

// [16 k x 128 cols] slab, columns contiguous in global memory -> smem rows of BT_LD doubles, zero-filled outside
// k < k_limit, col < col_limit.
template <bool ALIGNED16>
__device__ __forceinline__ void load_nmajor_slab(double* dst, const double* src, int64_t ld, int k0, int k_limit,
                                                 int64_t col0, int64_t col_limit, int tid) {
    if (ALIGNED16) {
#pragma unroll
        for (int i = 0; i < (BK * BN / 2) / GEMM_THREADS; ++i) {
            int c = tid + i * GEMM_THREADS;
            int kr = c >> 6, ch = c & 63;
            int gk = k0 + kr;
            int64_t gcol = col0 + ch * 2;
            int64_t left = (col_limit - gcol) * 8;
            int bytes = (gk < k_limit && left > 0) ? (left >= 16 ? 16 : 8) : 0;
            const double* s = bytes ? (src + (int64_t)gk * ld + gcol) : src;
            cp_async16(dst + kr * BT_LD + ch * 2, s, bytes);
        }
    } else {
#pragma unroll
        for (int i = 0; i < (BK * BN) / GEMM_THREADS; ++i) {
            int c = tid + i * GEMM_THREADS;
            int kr = c >> 7, col = c & 127;
            int gk = k0 + kr;
            int64_t gcol = col0 + col;
            int bytes = (gk < k_limit && gcol < col_limit) ? 8 : 0;
            const double* s = bytes ? (src + (int64_t)gk * ld + gcol) : src;
            cp_async8(dst + kr * BT_LD + col, s, bytes);
        }
    }
}

// one k-slab of the "NN" product: acc += A_s[128 x 16] * B_s[16 x 128], first K4 4-wide steps of the slab only (the
// triangular GEMM stops each warp at its own diagonal).  With four warps per sub-partition the fragment loads of one
// warp hide under the DMMAs of the others: no register double buffering.
template <int K4>
__device__ __forceinline__ void mma_nn_steps(double (&acc)[MI][NI][2], const double* ap, const double* bp) {
#pragma unroll
    for (int kk = 0; kk < K4; ++kk) {
        double a[MI], b[NI];
#pragma unroll
        for (int i = 0; i < MI; ++i) a[i] = ap[i * 8 * A_LD + kk * 4];
#pragma unroll
        for (int j = 0; j < NI; ++j) b[j] = bp[kk * 4 * BT_LD + j * 8];
#pragma unroll
        for (int i = 0; i < MI; ++i)
#pragma unroll
            for (int j = 0; j < NI; ++j) dmma884(acc[i][j][0], acc[i][j][1], a[i], b[j]);
    }
}
__device__ __forceinline__ void mma_nn_slab(double (&acc)[MI][NI][2], const double* As, const double* Bs, int wm, int wn,
                                            int g, int t, int k4_count) {
    const double* ap = As + (wm * 32 + g) * A_LD + t;
    const double* bp = Bs + t * BT_LD + wn * 32 + g;
    if (k4_count >= BK / 4) mma_nn_steps<BK / 4>(acc, ap, bp);      // the common case, fully unrolled
    else if (k4_count == 3) mma_nn_steps<3>(acc, ap, bp);
    else if (k4_count == 2) mma_nn_steps<2>(acc, ap, bp);
    else if (k4_count == 1) mma_nn_steps<1>(acc, ap, bp);
}
#endif  // __CUDACC__

// defined in chol.cu (host side, stream ordered)
// progress flags of the data-flow chain, for consumers of L^-1 that start before the chain has finished: block row J of
// L^-1 is final once fX[J] and fLi[J*nb + r], r < J, carry `epoch` in their upper 24 bits and a count >= 1
struct DfGate { const int* fX; const int* fLi; int nb; int epoch; };
int chol_factor_inv(Ctx* c, cudaStream_t s, int m, int mp, const double* M, double* L, int want_inv, double* Linv,
                    double* W, double* Y, double* acc, double* d_out, void* aux = nullptr, DfGate* gate = nullptr);
// data-flow form (two launches for the whole chain): used by chol_factor_inv when `aux` is given and chol_df_enabled(m)
// (64 < m <= 4096); otherwise one launch per block column
size_t chol_df_aux_bytes(int m);
bool chol_df_enabled(int m);
// worker CTAs of a data-flow chain with at most 8 block columns (m <= 512), where the spine bounds the chain; two per SM
constexpr int DF_SMALL_WORKERS = 16;

}  // namespace accbpg
