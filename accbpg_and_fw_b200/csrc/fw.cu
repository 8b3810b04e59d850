// D_opt_FW / D_opt_FW_away on the device (reference: accbpg/D_opt_alg.py:9-88, :91-185).
//
// The reference loop is O(mn) per iteration: argmax / masked argmin over w, a scalar step rule, a rank-one
// (Sherman-Morrison) update of Hinv = (V X V^T)^{-1}, and one GEMV-T pass over V that refreshes every w_j.
// Here the whole iteration stays on the GPU: five stream-ordered kernels per iteration, the scalar decision is
// taken by the last block of the selection kernel, histories (F, SP, SN, T) are written to device arrays and a
// stop flag turns the remaining launches of a batch into no-ops, so the host only looks at the control block once
// per batch.  F_k: D_opt_FW tracks det by the O(1) update (D_opt_alg.py:52,80); D_opt_FW_away recomputes
// log det(Hinv) by LU every iteration (:136) -- the same quantity follows the determinant-lemma increment, tracked
// here in a compensated (two-sum) accumulator; agreement with the per-iteration LU is ~1e-13 relative over
// thousands of iterations (tests/test_fw_*.py).
// Compiled with -fmad=false: the step-size formulas round as in NumPy.
#include <cooperative_groups.h>
#include <cuda.h>
#include "common.cuh"

namespace accbpg {

enum FwCtrl {
    C_STOP = 0,      // 1.0 once the optimality test fired
    C_KSTOP = 1,     // iteration index at which it fired
    C_LOGDET_HI = 2, // log det(V X V^T), compensated accumulator
    C_LOGDET_LO = 3,
    C_WMAX = 4, C_IMAX = 5,
    C_WMIN = 6, C_JMIN = 7,
    C_MODE = 8,      // 0 toward vertex i, 1 away from vertex j
    C_T = 9,         // step
    C_CS = 10,       // signed rank-one coefficient: Hinv <- (Hinv - cs*u u^T)/den
    C_DEN = 11,      // 1 - t (toward) or 1 + t (away)
    C_IDX = 12,      // chosen column (global index)
    C_TSIGN = 13,    // +t (toward) or -t (away): x[idx] += tsign
    C_NITER = 14,    // iterations executed (number of history entries written)
};

constexpr int FW_THREADS = 256;
#define FW_INF (__longlong_as_double(0x7ff0000000000000LL))

__device__ __forceinline__ void fw_arg_combine(double& v, long long& i, double v2, long long i2) {
    if (v2 < v || (v2 == v && i2 < i)) { v = v2; i = i2; }
}
__device__ __forceinline__ void fw_block_argmin(double& v, long long& i, double* shv, long long* shi) {
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = blockDim.x >> 5;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        double v2 = __shfl_xor_sync(0xffffffffu, v, o);
        long long i2 = __shfl_xor_sync(0xffffffffu, i, o);
        fw_arg_combine(v, i, v2, i2);
    }
    __syncthreads();
    if (lane == 0) { shv[wid] = v; shi[wid] = i; }
    __syncthreads();
    v = (lane < nw) ? shv[lane] : FW_INF;
    i = (lane < nw) ? shi[lane] : 0x7fffffffffffffffLL;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        double v2 = __shfl_xor_sync(0xffffffffu, v, o);
        long long i2 = __shfl_xor_sync(0xffffffffu, i, o);
        fw_arg_combine(v, i, v2, i2);
    }
}

// ---------------------------------------------------------------------------------------------------------------
// Selection (D_opt_alg.py:59-61 / :145-147) in ONE sweep over (w, x), carried as three candidates:
//   amax   (-w_i, i)  minimised            -> i = argmax w, first occurrence
//   smin   (w_i, i) over the support x_i > thr, minimised -> the masked argmin while some support entry is below w_max
//   fmask  first index outside the support -> decides the tie when every support entry equals w_max
//                                            (then (w - w_max)*[x > thr] is 0 everywhere and np.argmin returns the first index)
// thr = 1e-8 with away steps (:147), 0 without (:60).
struct FwCand {                  // 64 bytes; the column-sharded loop all-gathers one per rank
    double amax; long long imax;
    double smin; long long imin; double xmin;      // support minimum of w, its index, x there
    long long fmask; double wmask; double xmask;   // first index outside the support, w and x there
};
constexpr long long FW_NOIDX = 0x7fffffffffffffffLL;
__device__ __forceinline__ void fw_cand_init(FwCand& c) {
    c.amax = FW_INF; c.imax = FW_NOIDX; c.smin = FW_INF; c.imin = FW_NOIDX; c.xmin = 0.0;
    c.fmask = FW_NOIDX; c.wmask = 0.0; c.xmask = 0.0;
}
__device__ __forceinline__ void fw_smin_combine(FwCand& c, double v2, long long i2, double x2) {
    if (v2 < c.smin || (v2 == c.smin && i2 < c.imin)) { c.smin = v2; c.imin = i2; c.xmin = x2; }
}
__device__ __forceinline__ void fw_mask_combine(FwCand& c, long long i2, double w2, double x2) {
    if (i2 < c.fmask) { c.fmask = i2; c.wmask = w2; c.xmask = x2; }
}
__device__ __forceinline__ void fw_cand_add(FwCand& c, double wi, double xi, long long i, double thr) {
    fw_arg_combine(c.amax, c.imax, -wi, i);
    if (xi > thr) fw_smin_combine(c, wi, i, xi);
    else fw_mask_combine(c, i, wi, xi);
}
__device__ __forceinline__ void fw_cand_merge(FwCand& c, const FwCand& o) {
    fw_arg_combine(c.amax, c.imax, o.amax, o.imax);
    fw_smin_combine(c, o.smin, o.imin, o.xmin);
    fw_mask_combine(c, o.fmask, o.wmask, o.xmask);
}
__device__ __forceinline__ void fw_cand_warp(FwCand& c) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        FwCand q;
        q.amax = __shfl_xor_sync(0xffffffffu, c.amax, o);
        q.imax = __shfl_xor_sync(0xffffffffu, c.imax, o);
        q.smin = __shfl_xor_sync(0xffffffffu, c.smin, o);
        q.imin = __shfl_xor_sync(0xffffffffu, c.imin, o);
        q.xmin = __shfl_xor_sync(0xffffffffu, c.xmin, o);
        q.fmask = __shfl_xor_sync(0xffffffffu, c.fmask, o);
        q.wmask = __shfl_xor_sync(0xffffffffu, c.wmask, o);
        q.xmask = __shfl_xor_sync(0xffffffffu, c.xmask, o);
        fw_cand_merge(c, q);
    }
}
// block-wide merge; the result is valid in warp 0 (every lane)
__device__ __forceinline__ void fw_cand_block(FwCand& c, FwCand* sh /* >= 32 */) {
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = blockDim.x >> 5;
    fw_cand_warp(c);
    __syncthreads();
    if (lane == 0) sh[wid] = c;
    __syncthreads();
    if (wid == 0) {
        if (lane < nw) c = sh[lane]; else fw_cand_init(c);
        fw_cand_warp(c);
    }
}

// Column-sharded loop over NVLink peer memory (accbpg_fw_run_peer): every rank's receive buffers, mapped everywhere.
constexpr int FW_MAX_PEERS = 16;
struct FwPeer {
    FwCand* rec[FW_MAX_PEERS];                 // [2 (epoch parity)][world (sender)] selection records
    double* col[FW_MAX_PEERS];                 // [2 (epoch parity)][m] the chosen column, written by its owner
    unsigned long long* flags[FW_MAX_PEERS];   // [world] last record epoch per sender, [world] = last column epoch
    int rank, world;                           // world == 0: not in use
};

struct FwParams {
    FwPeer peer;
    const double* V; int m; int64_t n, ldv;
    double* x; double* w; double* Hinv; double* u; double* v;
    double* ctrl;
    double* hist_F; double* hist_SP; double* hist_SN; double* hist_T;
    FwCand* parts;            // one candidate record per selecting CTA
    unsigned int* counter;
    int away; double eps;
    int k;                    // iteration whose decision the tail of this kernel takes
    int nblk;                 // column blocks of the pass
    int width;                // columns per block (even, <= 128): chosen so that the blocks fill whole waves of SMs
    int nr1;                  // leading CTAs that update Hinv instead (they start first, so they read the step's
                              // coefficients long before the tail of the same launch replaces them)
    int decide;               // tail of the selecting kernels: 0 nothing, 1 merge + take the decision of iteration k,
                              // 2 merge only and write the record to cand_out (column-sharded: the ranks' records
                              // are exchanged before accbpg_fw_decide)
    FwCand* cand_out;
    int64_t col_offset;       // global index of local column 0
    int sharded;              // decide: the chosen column may live on another rank (then v <- 0 here)
    int reverse;              // pass kernel: walk the column blocks from the end
    int early;                // pass kernel: rows of V fetched before the dependency wait, always FWP_EARLY (a launch
                              // parameter rather than the constant: compiled in, it costs fw_pass_kernel<true> two
                              // registers and a different schedule)
};

// The decision of iteration p.k from the merged candidates (thread 0 of the last CTA), then the gather of the chosen
// column by the whole CTA.  D_opt_alg.py:52-82 / :136-179.
__device__ __forceinline__ void fw_decide(const FwParams& p, const FwCand& cd, int* sh_go, long long* sh_idx, int k_it = -1) {
    const int kk = k_it >= 0 ? k_it : p.k;          // the persistent loop passes its iteration explicitly
    if (threadIdx.x == 0) {
        double* c = p.ctrl;
        const double md = (double)p.m;
        const double wmax = -cd.amax;
        const long long imax = cd.imax;
        long long jmin = cd.imin;
        double wj = cd.smin, xj = cd.xmin;
        if (p.away && !(cd.imin != FW_NOIDX && cd.smin < wmax) && cd.fmask < cd.imin) {
            // argmin((w - w_max) * [x > 1e-8]) is the support minimum unless that ties with the zeros of the mask:
            // then every entry is 0 and np.argmin returns the first index overall
            jmin = cd.fmask; wj = cd.wmask; xj = cd.xmask;
        }
        if (jmin == FW_NOIDX) { jmin = 0; wj = wmax; xj = 1.0; }      // empty support cannot happen on the simplex
        const double logdet = c[C_LOGDET_HI] + c[C_LOGDET_LO];
        const double eps_pos = wmax / md - 1.0;
        const double eps_neg = 1.0 - wj / md;
        p.hist_F[kk] = -logdet;                   // D_opt_alg.py:52 (-log det M) / :136 (log det Hinv)
        p.hist_SP[kk] = eps_pos;
        p.hist_SN[kk] = eps_neg;
        unsigned long long ns;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(ns));
        p.hist_T[kk] = (double)ns;
        c[C_WMAX] = wmax; c[C_IMAX] = (double)imax;
        c[C_WMIN] = wj; c[C_JMIN] = (double)jmin;
        c[C_NITER] = (double)(kk + 1);
        int go = 1;
        if (eps_pos <= p.eps && eps_neg <= p.eps) {   // :72-73 / :159-160
            c[C_STOP] = 1.0; c[C_KSTOP] = (double)kk;
            go = 0;
        } else {
            double t, cs, den, inc, tsign;
            long long chosen;
            int mode;
            if (!p.away) {                                            // :75-82
                t = (wmax / md - 1.0) / (wmax - 1.0);
                double q = 1.0 + t * (wmax - 1.0);
                cs = t / q; den = 1.0 - t; chosen = imax; mode = 0; tsign = t;
                inc = (md - 1.0) * log(1.0 - t) + log(q);
            } else if (eps_pos >= eps_neg) {                          // :162-170
                t = (wmax / md - 1.0) / (wmax - 1.0);
                double q = 1.0 - t + t * wmax;
                cs = t / q; den = 1.0 - t; chosen = imax; mode = 0; tsign = t;
                inc = (md - 1.0) * log1p(-t) + log(q);
            } else {                                                  // :171-179 away step
                t = fmin((1.0 - wj / md) / (wj - 1.0), xj / (1.0 - xj));
                double q = 1.0 + t - t * wj;
                cs = -(t / q); den = 1.0 + t; chosen = jmin; mode = 1; tsign = -t;
                inc = (md - 1.0) * log1p(t) + log(q);
            }
            // compensated accumulation of log det(V X V^T)
            double hi = c[C_LOGDET_HI];
            double s = hi + inc;
            double bb = s - hi;
            double err = (hi - (s - bb)) + (inc - bb);
            c[C_LOGDET_HI] = s;
            c[C_LOGDET_LO] += err;
            c[C_MODE] = (double)mode; c[C_T] = t; c[C_CS] = cs; c[C_DEN] = den;
            c[C_IDX] = (double)chosen; c[C_TSIGN] = tsign;
            *sh_idx = chosen;
        }
        *sh_go = go;
    }
    __syncthreads();
    if (*sh_go) {
        const long long col = *sh_idx - p.col_offset;
        const bool mine = (col >= 0 && col < p.n);
        if (p.peer.world > 0) {
            // peer memory: the owner stores the column into every rank's receive slot of this epoch's parity and
            // releases the column flag; nobody else writes
            if (mine) {
                const unsigned long long epoch = (unsigned long long)p.k + 1ULL;
                const size_t slot = (size_t)(epoch & 1ULL) * p.m;
                for (int r = threadIdx.x; r < p.m; r += blockDim.x) {
                    const double val = p.V[(int64_t)r * p.ldv + col];
                    for (int q = 0; q < p.peer.world; ++q) p.peer.col[q][slot + r] = val;
                }
                __threadfence_system();
                __syncthreads();
                if ((int)threadIdx.x < p.peer.world)
                    st_release_sys(p.peer.flags[threadIdx.x] + p.peer.world, epoch);
            }
            return;
        }
        // column-sharded: ranks that do not own the column contribute zeros; the caller sums v over the ranks
        for (int r = threadIdx.x; r < p.m; r += blockDim.x) p.v[r] = mine ? p.V[(int64_t)r * p.ldv + col] : 0.0;
    }
}

// publish this CTA's candidates; the last of `nparts` CTAs merges them in index order and decides
__device__ __forceinline__ void fw_select_tail(const FwParams& p, FwCand& cd, int part, int nparts, FwCand* sh_c,
                                               bool* sh_last, int* sh_go, long long* sh_idx) {
    fw_cand_block(cd, sh_c);
    if (threadIdx.x == 0) p.parts[part] = cd;
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) {
        unsigned int tk = atomicAdd(p.counter, 1u);
        bool last = (tk == (unsigned)nparts - 1);
        *sh_last = last;
        if (last) *p.counter = 0u;
    }
    __syncthreads();
    if (!*sh_last) return;
    __threadfence();
    fw_cand_init(cd);
    for (int b = threadIdx.x; b < nparts; b += blockDim.x) {
        FwCand q;
        q.amax = ld_cg(&p.parts[b].amax); q.imax = __ldcg(&p.parts[b].imax);
        q.smin = ld_cg(&p.parts[b].smin); q.imin = __ldcg(&p.parts[b].imin); q.xmin = ld_cg(&p.parts[b].xmin);
        q.fmask = __ldcg(&p.parts[b].fmask); q.wmask = ld_cg(&p.parts[b].wmask); q.xmask = ld_cg(&p.parts[b].xmask);
        fw_cand_merge(cd, q);
    }
    fw_cand_block(cd, sh_c);
    if (threadIdx.x == 0) sh_c[0] = cd;
    __syncthreads();
    cd = sh_c[0];
    if (p.decide == 2) {
        if (p.peer.world > 0) {
            // record of iteration p.k -> slot `rank` of every rank's receive buffer, then this rank's flag word there
            if ((int)threadIdx.x < p.peer.world) {
                const unsigned long long epoch = (unsigned long long)p.k + 1ULL;
                p.peer.rec[threadIdx.x][(size_t)(epoch & 1ULL) * p.peer.world + p.peer.rank] = cd;
                __threadfence_system();
                st_release_sys(p.peer.flags[threadIdx.x] + p.peer.rank, epoch);
            }
        } else if (threadIdx.x == 0) {
            *p.cand_out = cd;
        }
        return;
    }
    fw_decide(p, cd, sh_go, sh_idx);
}

// column-sharded decision: merge the ranks' records in rank order, decide, gather the column if it lives here
__global__ void __launch_bounds__(FW_THREADS) fw_decide_kernel(FwParams p, const FwCand* recs, int world) {
    __shared__ int sh_go;
    __shared__ long long sh_idx;
    if (ld_cg(&p.ctrl[C_STOP]) != 0.0) return;
    FwCand cd;
    fw_cand_init(cd);
    for (int r = 0; r < world; ++r) {
        FwCand q;
        q.amax = ld_cg(&recs[r].amax); q.imax = __ldcg(&recs[r].imax);
        q.smin = ld_cg(&recs[r].smin); q.imin = __ldcg(&recs[r].imin); q.xmin = ld_cg(&recs[r].xmin);
        q.fmask = __ldcg(&recs[r].fmask); q.wmask = ld_cg(&recs[r].wmask); q.xmask = ld_cg(&recs[r].xmask);
        fw_cand_merge(cd, q);
    }
    fw_decide(p, cd, &sh_go, &sh_idx);
}

// the same over peer memory: wait for every rank's record of iteration p.k in the local receive buffer
__global__ void __launch_bounds__(FW_THREADS) fw_decide_peer_kernel(FwParams p) {
    __shared__ int sh_go;
    __shared__ long long sh_idx;
    asm volatile("griddepcontrol.wait;" ::: "memory");
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    if (ld_cg(&p.ctrl[C_STOP]) != 0.0) return;
    const unsigned long long epoch = (unsigned long long)p.k + 1ULL;
    if ((int)threadIdx.x < p.peer.world) peer_flag_wait(p.peer.flags[p.peer.rank] + threadIdx.x, epoch);
    __syncthreads();
    const FwCand* recs = p.peer.rec[p.peer.rank] + (size_t)(epoch & 1ULL) * p.peer.world;
    FwCand cd;
    fw_cand_init(cd);
    for (int r = 0; r < p.peer.world; ++r) {
        FwCand q;
        q.amax = ld_cg(&recs[r].amax); q.imax = __ldcg(&recs[r].imax);
        q.smin = ld_cg(&recs[r].smin); q.imin = __ldcg(&recs[r].imin); q.xmin = ld_cg(&recs[r].xmin);
        q.fmask = __ldcg(&recs[r].fmask); q.wmask = ld_cg(&recs[r].wmask); q.xmask = ld_cg(&recs[r].xmask);
        fw_cand_merge(cd, q);
    }
    fw_decide(p, cd, &sh_go, &sh_idx);
}

// standalone selection + decision (first iteration of a batch)
__global__ void __launch_bounds__(FW_THREADS) fw_select_kernel(FwParams p) {
    __shared__ FwCand sh_c[32];
    __shared__ bool sh_last;
    __shared__ int sh_go;
    __shared__ long long sh_idx;
    asm volatile("griddepcontrol.wait;" ::: "memory");
    if (p.decide != 2 && ld_cg(&p.ctrl[C_STOP]) != 0.0) return;
    const double thr = p.away ? 1.0e-8 : 0.0;
    FwCand cd;
    fw_cand_init(cd);
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < p.n; i += stride)
        fw_cand_add(cd, p.w[i], p.x[i], i + p.col_offset, thr);
    fw_select_tail(p, cd, blockIdx.x, gridDim.x, sh_c, &sh_last, &sh_go, &sh_idx);
}

// u = Hinv v (warp per row)            D_opt_alg.py:78 / :165 / :174
__global__ void __launch_bounds__(256) fw_hv_kernel(const double* __restrict__ Hinv, int m, const double* __restrict__ v,
                                                    double* __restrict__ u, const double* ctrl,
                                                    const unsigned long long* col_flag, unsigned long long epoch) {
    // the dependent pass may become resident while the previous pass drains: it fetches rows of V (which never change)
    // before its own wait, and that wait returns only when this grid - hence everything before it - has completed
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    asm volatile("griddepcontrol.wait;" ::: "memory");
    if (ld_cg(&ctrl[C_STOP]) != 0.0) return;
    if (col_flag) {                          // peer memory: v arrives from the rank that owns the chosen column
        if (threadIdx.x == 0) peer_flag_wait(col_flag, epoch);
        __syncthreads();
    }
    const int lane = threadIdx.x & 31;
    const int row = blockIdx.x * 8 + (threadIdx.x >> 5);
    if (row >= m) return;
    const double* hr = Hinv + (size_t)row * m;
    double s = 0.0;
    for (int c = lane; c < m; c += 32) s += __ldcg(hr + c) * __ldcg(v + c);
    s = warp_sum(s);
    if (lane == 0) u[row] = s;
}

// The one pass over V of iteration k-1 (p_j = u^T v_j; w_j <- (w_j - cs p_j^2)/den; x_j <- x_j*den (+- t at the chosen
// column)), the rank-one update Hinv <- (Hinv - cs u u^T)/den on the CTAs beyond the column blocks, and -- in the tail --
// the selection and decision of iteration k on the freshly updated (w, x): one kernel per iteration besides u = Hinv v.
// A CTA owns 128 columns; its four 64-thread groups split the rows and meet in shared memory (fixed order).
// Column blocks are walked in alternating directions from one iteration to the next, so the part of V the previous
// pass read last -- still resident in the 126 MB L2 -- is read first.
constexpr int FWP_THREADS = 256;
constexpr int FWP_COLS = 128;
constexpr int FWP_UNROLL = 16;       // rows in flight per thread (16 x 16 B)
// rows per row group fetched before the dependency wait: the first FWP_UNROLL into registers, the rest as L2 prefetches
// (measured at 500 x 50000: 48 rows 19.2 k iterations per second, 80 rows 18.8 k, 125 rows 17.6 k)
constexpr int FWP_EARLY = 48;

template <bool VEC2>
__global__ void __launch_bounds__(FWP_THREADS) fw_pass_kernel(FwParams p) {
    extern __shared__ double us[];                         // u (m doubles)
    __shared__ double part[4][FWP_COLS];
    __shared__ FwCand sh_c[32];
    __shared__ bool sh_last;
    __shared__ int sh_go;
    __shared__ long long sh_idx;
    // ---- before the dependency wait: only V (constant for the whole solve) and the launch parameters are touched.
    // Launched programmatically behind u = Hinv v, this CTA can be resident while the previous pass drains and takes its
    // decision; the first rows of its columns go to registers and the next ones are pulled into L2 meanwhile.
    const int m = p.m;
    const int blk = (int)blockIdx.x - p.nr1;
    const int cb = p.reverse ? (p.nblk - 1 - blk) : blk;
    const int rg = threadIdx.x >> 6, ct = threadIdx.x & 63;
    const int rows_per = (m + 3) / 4;
    const int r0 = rg * rows_per, r1 = min(m, r0 + rows_per);
    const int64_t j = (int64_t)cb * p.width + ct * 2;
    const bool owns = blk >= 0 && (ct * 2 < p.width) && (j < p.n);
    const bool pre = VEC2 && p.early > 0 && owns && (j + 1 < p.n) && (r0 + FWP_UNROLL <= r1);
    double2 a0[FWP_UNROLL];
    if (pre) {
        const double* col = p.V + j;
#pragma unroll
        for (int q = 0; q < FWP_UNROLL; ++q)
            asm volatile("ld.global.nc.L1::no_allocate.v2.f64 {%0,%1}, [%2];"
                         : "=d"(a0[q].x), "=d"(a0[q].y) : "l"(col + (int64_t)(r0 + q) * p.ldv));
        if ((ct & 3) == 0) {                                 // one request per 64 bytes of a row
            const int rl = min(r1, r0 + p.early);
            for (int r = r0 + FWP_UNROLL; r < rl; ++r)
                asm volatile("prefetch.global.L2 [%0];" ::"l"(col + (int64_t)r * p.ldv));
        }
    }
    asm volatile("griddepcontrol.wait;" ::: "memory");
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    if (ld_cg(&p.ctrl[C_STOP]) != 0.0) return;               // uniform over the whole grid
    const double cs = ld_cg(&p.ctrl[C_CS]), den = ld_cg(&p.ctrl[C_DEN]);
    if ((int)blockIdx.x < p.nr1) {                           // Hinv <- (Hinv - cs u u^T)/den     D_opt_alg.py:79 / :166 / :175
        const int64_t total = (int64_t)m * m;
        const int64_t stride = (int64_t)p.nr1 * blockDim.x;
        for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += stride) {
            int r = (int)(e / m), c = (int)(e - (int64_t)r * m);
            double o = __ldcg(p.u + r) * __ldcg(p.u + c);
            p.Hinv[e] = (p.Hinv[e] - cs * o) / den;
        }
        return;
    }
    for (int r = threadIdx.x; r < m; r += blockDim.x) us[r] = __ldcg(p.u + r);
    __syncthreads();
    double s0 = 0.0, s1 = 0.0;
    if (owns) {
        const double* col = p.V + j;
        int r = r0;
        if (VEC2 && j + 1 < p.n) {
            if (pre) {                                       // the batch fetched before the wait: same rows, same order
#pragma unroll
                for (int q = 0; q < FWP_UNROLL; ++q) {
                    double uq = us[r + q];
                    s0 += uq * a0[q].x;
                    s1 += uq * a0[q].y;
                }
                r += FWP_UNROLL;
            }
            for (; r + FWP_UNROLL <= r1; r += FWP_UNROLL) {
                double2 a[FWP_UNROLL];
#pragma unroll
                for (int q = 0; q < FWP_UNROLL; ++q)
                    asm volatile("ld.global.nc.L1::no_allocate.v2.f64 {%0,%1}, [%2];"
                                 : "=d"(a[q].x), "=d"(a[q].y) : "l"(col + (int64_t)(r + q) * p.ldv));
#pragma unroll
                for (int q = 0; q < FWP_UNROLL; ++q) {
                    double uq = us[r + q];
                    s0 += uq * a[q].x;
                    s1 += uq * a[q].y;
                }
            }
            const int rem = r1 - r;                      // < 16 rows left: one more batch, predicated
            if (rem > 0) {
                double2 a[FWP_UNROLL];
#pragma unroll
                for (int q = 0; q < FWP_UNROLL; ++q)
                    if (q < rem)
                        asm volatile("ld.global.nc.L1::no_allocate.v2.f64 {%0,%1}, [%2];"
                                     : "=d"(a[q].x), "=d"(a[q].y) : "l"(col + (int64_t)(r + q) * p.ldv));
#pragma unroll
                for (int q = 0; q < FWP_UNROLL; ++q)
                    if (q < rem) {
                        double uq = us[r + q];
                        s0 += uq * a[q].x;
                        s1 += uq * a[q].y;
                    }
            }
        } else {
            const bool two = (j + 1 < p.n);
            for (; r < r1; ++r) {
                double uq = us[r];
                s0 += uq * __ldcs(col + (int64_t)r * p.ldv);
                if (two) s1 += uq * __ldcs(col + (int64_t)r * p.ldv + 1);
            }
        }
    }
    part[rg][2 * ct] = s0;
    part[rg][2 * ct + 1] = s1;
    __syncthreads();
    FwCand cd;
    fw_cand_init(cd);
    if (rg == 0 && owns) {
        const double thr = p.away ? 1.0e-8 : 0.0;
        const int64_t idx = (int64_t)ld_cg(&p.ctrl[C_IDX]);
        const double tsign = ld_cg(&p.ctrl[C_TSIGN]);
#pragma unroll
        for (int e = 0; e < 2; ++e) {
            if (j + e < p.n) {
                const double pj = ((part[0][2 * ct + e] + part[1][2 * ct + e]) + part[2][2 * ct + e]) + part[3][2 * ct + e];
                const double wn = (p.w[j + e] - cs * (pj * pj)) / den;
                double xn = p.x[j + e] * den;
                if (j + e + p.col_offset == idx) xn = xn + tsign;
                p.w[j + e] = wn;
                p.x[j + e] = xn;
                fw_cand_add(cd, wn, xn, j + e + p.col_offset, thr);
            }
        }
    }
    if (!p.decide) return;
    fw_select_tail(p, cd, blk, p.nblk, sh_c, &sh_last, &sh_go, &sh_idx);
}

// ------------------------------------------------------------------------------------------------------------------
// The same loop as ONE persistent launch per batch of iterations (one GPU; accbpg_fw_run takes it when V is 16-byte
// aligned with even n and ldv, n < 2^31, m <= 4096 and at least three ring stages fit in shared memory).  One CTA per SM
// owns the column blocks b = blockIdx.x, blockIdx.x + G, ... of W columns; one producer thread streams their rows into a
// shared-memory ring (one 3-D tensor copy per stage when 4 | m, else one 2-D copy per row group: a stage holds FWR_ROWS
// rows of each of the four row groups; single row copies issued per lane serialise in the TMA unit and reach 3 TB/s
// only).  Bytes in flight are bounded by shared memory (6 x 32 KB per SM) instead of registers.
// Measured with this ring feeding the pass of the launch chain at 500 x 50000 (DESIGN.md section 11): the ring streams the
// 200 MB of V in 29.6 us (6.8 TB/s, the copy roof), but an iteration takes 53 us because the decision tail (13.5 us after
// the last CTA has finished streaming) and the u = Hinv v launch (8.6 us between the decision and the next pass) are
// serial.  Here nothing is launched between iterations:
//   records   every CTA reads all G selection records itself (one store -> poll hop), merges them and takes the
//             decision of iteration k on its own copy of the log-det accumulator (CTA 0 writes the history entry and the
//             control block), then gathers the chosen column
//   u         rows cta + i G of Hinv times the column (warp per row), delivered as (value, token) words every CTA collects
//   pass      warps 0-7 consume the ring (row groups and summation order of fw_pass_kernel: four row groups, rows in
//             order, groups merged ((0+1)+2)+3, so w, x and the vertex sequence are bit-identical), lane 0 of warp 8
//             feeds it and, towards the end of the pass, already issues the first stages of the NEXT iteration (V never
//             changes), which land during the exchanges; warps 9-15 apply the rank-one update to the own rows of Hinv
//   record    of the updated columns, for the next decision
// The arithmetic is that of the launch chain, operation for operation.  Exchanges are stores followed by a release of a
// token word that the consumer polls; tokens are unique per launch and iteration, buffers alternate on the iteration's
// parity.
constexpr int FWR_ROWS = 8;                                  // rows per row group and stage (one tensor box)
constexpr int FWR_BOX_BYTES = FWR_ROWS * FWP_COLS * 8;       // bytes reserved per box (rows packed at width * 8 bytes)
constexpr int FWR_STAGE_BYTES = 4 * FWR_BOX_BYTES;           // 32 KB
constexpr int FWR_MAX_STAGES = 6;
constexpr int FWR_STATIC_SMEM = 12 * 1024;                   // part, records, barriers (upper bound used by the host)
constexpr int FWS_THREADS = 512;
constexpr int FWS_CONS = 256;                                // consuming threads (warps 0-7)
constexpr int FWQ_REC_DOUBLES = 16;                          // a selection record's slot: one 128-byte line

struct FwPersist {
    double* ux;                    // [2][m] (value, token) pairs: the entries of u, each written by the CTA that owns the row
    double* recs;                  // [2][G][FWQ_REC_DOUBLES] selection records
    unsigned long long* tok;       // [2][256] flag words, one per CTA, released after its record
    unsigned long long base;
    int G, k_start, k_count;
    int stages;                    // stages of the shared-memory ring
    int ring_3d;                   // the tensor map is 3-D (columns, rows of a group, row groups)
};

__device__ __forceinline__ void fwr_mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void fwr_mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void fwr_mbar_expect(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void fwr_mbar_wait(uint32_t bar, uint32_t parity) {      // bounded: a protocol error traps
    uint32_t ok = 0;
    for (int spin = 0; spin < (1 << 24); ++spin) {
        asm volatile("{\n .reg .pred p;\n mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n selp.u32 %0, 1, 0, p;\n}\n"
                     : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
        if (ok) return;
    }
    __trap();
}
__device__ __forceinline__ void fwr_tma_load_3d(uint32_t dst, const void* tmap, int c0, int c1, int c2, uint32_t bar) {
    asm volatile("cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];"
                 ::"r"(dst), "l"(tmap), "r"(c0), "r"(c1), "r"(c2), "r"(bar) : "memory");
}
__device__ __forceinline__ void fwr_tma_load_2d(uint32_t dst, const void* tmap, int c0, int c1, uint32_t bar) {
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
                 ::"r"(dst), "l"(tmap), "r"(c0), "r"(c1), "r"(bar) : "memory");
}

__device__ __forceinline__ void fwq_post(unsigned long long* p, unsigned long long token) {
    asm volatile("st.release.gpu.global.u64 [%0], %1;" ::"l"(p), "l"(token) : "memory");
}
__device__ __forceinline__ void fwq_st_pair(double* p, double v, unsigned long long tok) {
    asm volatile("st.volatile.global.v2.u64 [%0], {%1, %2};" ::"l"(p), "l"(__double_as_longlong(v)), "l"(tok) : "memory");
}
__device__ __forceinline__ double fwq_wait_pair(const double* p, unsigned long long token) {
    unsigned long long v, tk, t0 = 0;
    unsigned spin = 0;
    for (;;) {
        asm volatile("ld.volatile.global.v2.u64 {%0, %1}, [%2];" : "=l"(v), "=l"(tk) : "l"(p) : "memory");
        if (tk == token) return __longlong_as_double((long long)v);
        __nanosleep(64);
        if ((++spin & 0x3ffu) == 0) {
            unsigned long long now;
            asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(now));
            if (t0 == 0) t0 = now;
            else if (now - t0 > 4000000000ULL) __trap();
        }
    }
}

// the step rule of fw_decide on a copy of the log-det accumulator kept by every CTA (all CTAs take the same decision from
// the same records; only the writer touches the control block and the histories)
struct FwDec { double cs, den, tsign; long long idx; int go; };
__device__ __forceinline__ void fwq_decide(const FwParams& p, const FwCand& cd, int kk, double& hi_state, double& lo_state,
                                           bool writer, FwDec& d) {
    double* c = p.ctrl;
    const double md = (double)p.m;
    const double wmax = -cd.amax;
    const long long imax = cd.imax;
    long long jmin = cd.imin;
    double wj = cd.smin, xj = cd.xmin;
    if (p.away && !(cd.imin != FW_NOIDX && cd.smin < wmax) && cd.fmask < cd.imin) {
        jmin = cd.fmask; wj = cd.wmask; xj = cd.xmask;
    }
    if (jmin == FW_NOIDX) { jmin = 0; wj = wmax; xj = 1.0; }
    const double logdet = hi_state + lo_state;
    const double eps_pos = wmax / md - 1.0;
    const double eps_neg = 1.0 - wj / md;
    if (writer) {
        p.hist_F[kk] = -logdet;
        p.hist_SP[kk] = eps_pos;
        p.hist_SN[kk] = eps_neg;
        unsigned long long ns;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(ns));
        p.hist_T[kk] = (double)ns;
        c[C_WMAX] = wmax; c[C_IMAX] = (double)imax;
        c[C_WMIN] = wj; c[C_JMIN] = (double)jmin;
        c[C_NITER] = (double)(kk + 1);
    }
    d.go = 1;
    if (eps_pos <= p.eps && eps_neg <= p.eps) {
        if (writer) { c[C_STOP] = 1.0; c[C_KSTOP] = (double)kk; }
        d.go = 0;
        return;
    }
    double t, cs, den, inc, tsign;
    long long chosen;
    int mode;
    if (!p.away) {
        t = (wmax / md - 1.0) / (wmax - 1.0);
        double qq = 1.0 + t * (wmax - 1.0);
        cs = t / qq; den = 1.0 - t; chosen = imax; mode = 0; tsign = t;
        inc = (md - 1.0) * log(1.0 - t) + log(qq);
    } else if (eps_pos >= eps_neg) {
        t = (wmax / md - 1.0) / (wmax - 1.0);
        double qq = 1.0 - t + t * wmax;
        cs = t / qq; den = 1.0 - t; chosen = imax; mode = 0; tsign = t;
        inc = (md - 1.0) * log1p(-t) + log(qq);
    } else {
        t = fmin((1.0 - wj / md) / (wj - 1.0), xj / (1.0 - xj));
        double qq = 1.0 + t - t * wj;
        cs = -(t / qq); den = 1.0 + t; chosen = jmin; mode = 1; tsign = -t;
        inc = (md - 1.0) * log1p(t) + log(qq);
    }
    const double hi = hi_state;
    const double sv = hi + inc;
    const double bb = sv - hi;
    const double err = (hi - (sv - bb)) + (inc - bb);
    hi_state = sv;
    lo_state += err;
    if (writer) {
        c[C_LOGDET_HI] = sv;
        c[C_LOGDET_LO] = lo_state;
        c[C_MODE] = (double)mode; c[C_T] = t; c[C_CS] = cs; c[C_DEN] = den;
        c[C_IDX] = (double)chosen; c[C_TSIGN] = tsign;
    }
    d.cs = cs; d.den = den; d.tsign = tsign; d.idx = chosen;
}

__global__ void __launch_bounds__(FWS_THREADS, 1)
fw_persist_ring_kernel(FwParams p, FwPersist q, const __grid_constant__ CUtensorMap tmV) {
    extern __shared__ __align__(128) unsigned char fws_raw[];      // ring [S][32 KB], then u, v, second v (mpad each)
    __shared__ double part[2][4][FWP_COLS];
    __shared__ FwCand sh_c[32];
    __shared__ FwCand sh_merged;
    __shared__ FwDec sh_dec;
    __shared__ double sh_logdet[2];
    __shared__ __align__(8) unsigned long long bar_mem[2 * FWR_MAX_STAGES];
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const int m = p.m, S = q.stages, G = q.G, cta = blockIdx.x;
    const int mpad = (m + 1) / 2 * 2;
    const uint32_t ring = (uint32_t)__cvta_generic_to_shared(fws_raw);
    double* us = reinterpret_cast<double*>(fws_raw + (size_t)S * FWR_STAGE_BYTES);
    double* vs = us + mpad;                             // the chosen column
    double* vs2 = vs + mpad;                            // the other candidate (both are fetched while thread 0 decides)
    const uint32_t bars = (uint32_t)__cvta_generic_to_shared(bar_mem);
    if (ld_cg(&p.ctrl[C_STOP]) != 0.0) return;          // stopped in an earlier batch: uniform over the grid
    if (tid == 0) {
        sh_logdet[0] = ld_cg(&p.ctrl[C_LOGDET_HI]); sh_logdet[1] = ld_cg(&p.ctrl[C_LOGDET_LO]);
        for (int s = 0; s < S; ++s) {
            fwr_mbar_init(bars + 8 * s, 1);
            fwr_mbar_init(bars + 8 * (FWR_MAX_STAGES + s), FWS_CONS / 32);
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    // column blocks cta, cta + G, ... of W columns each: at any moment the CTAs read neighbouring segments of the same rows
    // (contiguous strips per CTA scatter the requests over DRAM pages: 43 us per pass against 30)
    const int W = p.width;
    const int nsub = (cta < p.nblk) ? (p.nblk - 1 - cta) / G + 1 : 0;
    const int rows_per = (m + 3) / 4;
    const int chunks = (rows_per + FWR_ROWS - 1) / FWR_ROWS;
    const int per_it = nsub * chunks;                    // stages per iteration
    const double thr = p.away ? 1.0e-8 : 0.0;
    const int rg = (tid & 255) >> 6, ct = tid & 63;
    const int r0 = rg * rows_per, r1 = min(m, r0 + rows_per);
    const int nown = cta < m ? (m - cta + G - 1) / G : 0;      // rows of Hinv / entries of u this CTA owns: cta + i G
    const uint32_t seg = (uint32_t)W * 8u;
    const bool producer = (tid == FWS_CONS);
    // ---- producer state (one thread): stages issued over the whole launch, kept as (slot, use count of the slot, position
    //      inside the iteration) so that no division sits on the issue path
    // Odd iterations walk the column blocks in the opposite order: what the previous pass read last - still in the
    // 126 MB L2 - is read first (a pass in the same order every time finds nothing of a 200 MB V left).
    int pc = 0, p_st = 0, p_use = 0, p_sb = 0, p_ch = 0, p_rev = q.k_start & 1;
    const uint32_t stage_tx = 4u * FWR_ROWS * seg;
    auto issue = [&]() {
        const int j0 = (cta + (p_rev ? nsub - 1 - p_sb : p_sb) * G) * W;
        if (p_use > 0) fwr_mbar_wait(bars + 8 * (FWR_MAX_STAGES + p_st), (uint32_t)((p_use + 1) & 1));
        fwr_mbar_expect(bars + 8 * p_st, stage_tx);
        if (q.ring_3d) {
            fwr_tma_load_3d(ring + p_st * FWR_STAGE_BYTES, &tmV, j0, p_ch * FWR_ROWS, 0, bars + 8 * p_st);
        } else {
#pragma unroll
            for (int g4 = 0; g4 < 4; ++g4)
                fwr_tma_load_2d(ring + p_st * FWR_STAGE_BYTES + g4 * (FWR_ROWS * seg), &tmV, j0, g4 * rows_per + p_ch * FWR_ROWS,
                                bars + 8 * p_st);
        }
        ++pc;
        if (++p_st == S) { p_st = 0; ++p_use; }
        if (++p_ch == chunks) { p_ch = 0; if (++p_sb == nsub) { p_sb = 0; p_rev ^= 1; } }
    };
    if (producer && per_it > 0) {                        // the first stages of the first pass
        const int lim = per_it < S ? per_it : S;
        while (pc < lim) issue();
    }
    int cc_done = 0, c_st = 0, c_ph = 0;                 // stages consumed so far; the consumers' slot and its phase parity
    // ---- the record of the first decision: candidates of the own columns from (w, x) as they are
    FwCand cd;
    fw_cand_init(cd);
    for (int sb = 0; sb < nsub; ++sb) {
        const int64_t b0 = (int64_t)(cta + sb * G) * W;
        const int64_t b1 = b0 + W < p.n ? b0 + W : p.n;
        for (int64_t j = b0 + tid; j < b1; j += FWS_THREADS) fw_cand_add(cd, p.w[j], p.x[j], j, thr);
    }
    // Exchanges.  Records: plain words, then ONE flag word per CTA (compact array, sixteen flags per line) released after
    // them; a waiting CTA polls the G flags with one warp and a 100 ns back-off, then reads the records once.  Polling the
    // records themselves - (value, token) words, a line per CTA - costs a hop less but disturbs the CTAs that are still
    // streaming: their pass ran at 27 GB/s per SM instead of 43 with every thread polling, and still did with one polling
    // warp and a 300 ns back-off.  u: (value, token) words; everybody waits for u together, nothing streams meanwhile.
    unsigned long long* frec = q.tok;                    // [2][256]
    auto wait_flags = [&](const unsigned long long* f, unsigned long long token) {      // warp 0; all G <= 256 flags == token
        unsigned long long t0 = 0;
        unsigned spin = 0, done = 0;
        for (;;) {
            unsigned long long v[8];
#pragma unroll
            for (int e = 0; e < 8; ++e) {                // all of a lane's flags in flight at once
                v[e] = token;
                if (!(done & (1u << e)) && lane + 32 * e < G)
                    asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(v[e]) : "l"(f + lane + 32 * e) : "memory");
            }
#pragma unroll
            for (int e = 0; e < 8; ++e) if (v[e] == token) done |= 1u << e;
            if (__all_sync(0xffffffffu, done == 0xffu)) break;
            __nanosleep(100);
            if ((++spin & 0x3ffu) == 0) {
                unsigned long long now;
                asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(now));
                if (t0 == 0) t0 = now;
                else if (now - t0 > 4000000000ULL) __trap();
            }
        }
        asm volatile("fence.acq_rel.gpu;" ::: "memory");      // acquire: the records behind the flags
    };
    auto deliver_record = [&](int it) {                 // record for the decision of batch iteration `it`
        fw_cand_block(cd, sh_c);
        if (tid == 0) {                                  // warp 0 holds the merged record in every lane
            double* dst = q.recs + ((size_t)(it & 1) * G + cta) * FWQ_REC_DOUBLES;
            __stcg(dst + 0, cd.amax); __stcg(dst + 1, __longlong_as_double(cd.imax));
            __stcg(dst + 2, cd.smin); __stcg(dst + 3, __longlong_as_double(cd.imin)); __stcg(dst + 4, cd.xmin);
            __stcg(dst + 5, __longlong_as_double(cd.fmask)); __stcg(dst + 6, cd.wmask); __stcg(dst + 7, cd.xmask);
            fwq_post(frec + (size_t)(it & 1) * 256 + cta, q.base + 4ULL * (unsigned long long)it);
        }
    };
    deliver_record(0);
    for (int it = 0; it < q.k_count; ++it) {
        const int par = it & 1;
        const unsigned long long tokD = q.base + 4ULL * it, tokB = tokD + 2;
        // ---- every CTA gathers the G records itself and merges them (any order: the combines are total orders on
        //      (value, index)), then takes the decision of iteration k
        if (wid == 0) wait_flags(frec + (size_t)par * 256, tokD);
        __syncthreads();
        fw_cand_init(cd);
        for (int b = tid; b < G; b += FWS_THREADS) {
            const double* src = q.recs + ((size_t)par * G + b) * FWQ_REC_DOUBLES;
            FwCand o;
            o.amax = __ldcg(src + 0); o.imax = __double_as_longlong(__ldcg(src + 1));
            o.smin = __ldcg(src + 2); o.imin = __double_as_longlong(__ldcg(src + 3)); o.xmin = __ldcg(src + 4);
            o.fmask = __double_as_longlong(__ldcg(src + 5)); o.wmask = __ldcg(src + 6); o.xmask = __ldcg(src + 7);
            fw_cand_merge(cd, o);
        }
        fw_cand_block(cd, sh_c);                          // merged record in every lane of warp 0
        if (wid == 0 && lane == 0) sh_merged = cd;
        __syncthreads();
        // Thread 0 takes the decision (a few hundred dependent FP64 instructions) while the other warps fetch BOTH columns
        // the step rule can choose (argmax w, or the away vertex).  (Forming the own rows of u for both candidates under
        // the decision as well was measured slower: 17.7 k against 19.9 k iterations per second.)
        {
            const FwCand mc = sh_merged;
            long long jm = mc.imin;
            if (p.away && !(mc.imin != FW_NOIDX && mc.smin < -mc.amax) && mc.fmask < mc.imin) jm = mc.fmask;
            if (jm == FW_NOIDX) jm = 0;
            const long long im = mc.imax;
            if (tid == 0) {
                FwDec d;
                d.cs = d.den = d.tsign = 0.0; d.idx = 0; d.go = 0;
                fwq_decide(p, mc, q.k_start + it, sh_logdet[0], sh_logdet[1], cta == 0, d);
                sh_dec = d;
            } else if (tid >= 32) {
                for (int r = tid - 32; r < 2 * m; r += FWS_THREADS - 32) {
                    const int rr = r < m ? r : r - m;
                    const long long col = r < m ? im : jm;
                    const double val = (col >= 0 && col < p.n) ? __ldg(p.V + (int64_t)rr * p.ldv + col) : 0.0;
                    if (r < m) vs[rr] = val; else vs2[rr] = val;
                }
            }
        }
        __syncthreads();
        if (!sh_dec.go) {                                // the optimality test fired at this iteration: uniform over the grid
            if (producer) {                              // let the copies in flight land before the CTA gives up its shared memory
                int st = c_st, ph = c_ph;
                for (int c = cc_done; c < pc; ++c) {
                    fwr_mbar_wait(bars + 8 * st, (uint32_t)ph);
                    if (++st == S) { st = 0; ph ^= 1; }
                }
            }
            return;
        }
        const double cs = sh_dec.cs, den = sh_dec.den, tsign = sh_dec.tsign;
        const int64_t idx = sh_dec.idx;
        const double* vc = (idx == sh_merged.imax) ? vs : vs2;      // (when both candidates coincide the columns are equal)
        // ---- u_r = Hinv[r,:] v for the own rows (warp per row, summation order of fw_hv_kernel), delivered to every CTA
        for (int i = wid; i < nown; i += FWS_THREADS / 32) {
            const int r = cta + i * G;
            const double* hr = p.Hinv + (size_t)r * m;
            double sacc = 0.0;
            for (int cb = 0; cb < m; cb += 256) {         // eight loads in flight per lane
                double hv[8];
#pragma unroll
                for (int e = 0; e < 8; ++e) {
                    const int c = cb + lane + 32 * e;
                    hv[e] = c < m ? __ldcg(hr + c) : 0.0;
                }
#pragma unroll
                for (int e = 0; e < 8; ++e) {
                    const int c = cb + lane + 32 * e;
                    if (c < m) sacc += hv[e] * vc[c];
                }
            }
            sacc = warp_sum(sacc);
            if (lane == 0) fwq_st_pair(q.ux + ((size_t)par * m + r) * 2, sacc, tokB);
        }
        // (value, token) words: one hop; everybody waits here together, so the polling does not disturb a pass
        for (int r = tid; r < m; r += FWS_THREADS) us[r] = fwq_wait_pair(q.ux + ((size_t)par * m + r) * 2, tokB);
        __syncthreads();
        fw_cand_init(cd);
        if (tid < FWS_CONS) {
            // ---- the pass over the own column blocks
            int st = c_st, ph = c_ph;
            const int rev = (q.k_start + it) & 1;
            for (int sq = 0; sq < nsub; ++sq) {
                const int sb = rev ? nsub - 1 - sq : sq;
                const int64_t j = (int64_t)(cta + sb * G) * W + ct * 2;
                const bool owns = (ct * 2 < W) && (j < p.n);
                double s0 = 0.0, s1 = 0.0;
                for (int ch = 0; ch < chunks; ++ch) {
                    fwr_mbar_wait(bars + 8 * st, (uint32_t)ph);
                    if (owns) {
                        const uint32_t base = ring + st * FWR_STAGE_BYTES + rg * (FWR_ROWS * seg) + ct * 16;
                        const int rb = r0 + ch * FWR_ROWS;
#pragma unroll
                        for (int e = 0; e < FWR_ROWS; ++e) {
                            if (rb + e < r1) {
                                double ax, ay;
                                asm volatile("ld.shared.v2.f64 {%0,%1}, [%2];" : "=d"(ax), "=d"(ay) : "r"(base + e * seg));
                                const double uq = us[rb + e];
                                s0 += uq * ax;
                                s1 += uq * ay;
                            }
                        }
                    }
                    __syncwarp();
                    if (lane == 0) fwr_mbar_arrive(bars + 8 * (FWR_MAX_STAGES + st));
                    if (++st == S) { st = 0; ph ^= 1; }
                }
                const int buf = sq & 1;
                part[buf][rg][2 * ct] = s0;
                part[buf][rg][2 * ct + 1] = s1;
                asm volatile("bar.sync 1, %0;" ::"n"(FWS_CONS) : "memory");
                if (rg == 0 && owns) {
#pragma unroll
                    for (int e = 0; e < 2; ++e) {
                        if (j + e < p.n) {
                            const double pj = ((part[buf][0][2 * ct + e] + part[buf][1][2 * ct + e]) + part[buf][2][2 * ct + e]) +
                                              part[buf][3][2 * ct + e];
                            const double wn = (p.w[j + e] - cs * (pj * pj)) / den;
                            double xn = p.x[j + e] * den;
                            if (j + e == idx) xn = xn + tsign;
                            p.w[j + e] = wn;
                            p.x[j + e] = xn;
                            fw_cand_add(cd, wn, xn, j + e, thr);
                        }
                    }
                }
            }
        } else if (producer) {
            // ---- the rest of this pass, then the first stages of the next one (they land during the exchanges)
            const int end_it = cc_done + per_it;
            const int lim = (it + 1 < q.k_count) ? end_it + (per_it < S ? per_it : S) : end_it;
            while (pc < lim) issue();
        } else if (wid > FWS_CONS / 32) {
            // ---- Hinv <- (Hinv - cs u u^T)/den on the own rows (warps 9-15)      D_opt_alg.py:79 / :166 / :175
            const int ht = tid - (FWS_CONS + 32), hn = FWS_THREADS - FWS_CONS - 32;
            for (int e0 = ht; e0 < nown * m; e0 += hn * 4) {
                double hv[4];
#pragma unroll
                for (int u4 = 0; u4 < 4; ++u4) {
                    const int e = e0 + u4 * hn;
                    if (e < nown * m) { const int i = e / m, c = e - i * m; hv[u4] = __ldcg(p.Hinv + (size_t)(cta + i * G) * m + c); }
                }
#pragma unroll
                for (int u4 = 0; u4 < 4; ++u4) {
                    const int e = e0 + u4 * hn;
                    if (e < nown * m) {
                        const int i = e / m, c = e - i * m, r = cta + i * G;
                        const double o = us[r] * us[c];
                        p.Hinv[(size_t)r * m + c] = (hv[u4] - cs * o) / den;
                    }
                }
            }
        }
        cc_done += per_it;
        {   // every thread advances its copy of the consumers' ring position by per_it stages
            const int adv = c_st + per_it;
            c_ph ^= (adv / S) & 1;
            c_st = adv % S;
        }
        __syncthreads();
        deliver_record(it + 1);
    }
}

// Hinv = Linv^T Linv  (setup only; Linv lower triangular, zero padded, leading dimension mp)
__global__ void __launch_bounds__(256) fw_hinv_kernel(const double* __restrict__ Linv, int m, int mp,
                                                      double* __restrict__ Hinv) {
    __shared__ double Ar[32][33], Ac[32][33];
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;       // 32 x 8
    const int r0 = blockIdx.y * 32, c0 = blockIdx.x * 32;
    if (c0 > r0) return;                                          // lower blocks only, mirrored below
    double acc[4] = {0.0, 0.0, 0.0, 0.0};
    for (int k0 = r0; k0 < mp; k0 += 32) {                        // Linv[k][r] = 0 for k < r
        __syncthreads();
        for (int e = ty; e < 32; e += 8) {
            Ar[e][tx] = Linv[(size_t)(k0 + e) * mp + r0 + tx];
            Ac[e][tx] = Linv[(size_t)(k0 + e) * mp + c0 + tx];
        }
        __syncthreads();
#pragma unroll 8
        for (int kk = 0; kk < 32; ++kk) {
            double b = Ac[kk][tx];
#pragma unroll
            for (int q = 0; q < 4; ++q) acc[q] = fma(Ar[kk][ty + 8 * q], b, acc[q]);
        }
    }
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        int r = r0 + ty + 8 * q, c = c0 + tx;
        if (r < m && c < m) {
            Hinv[(size_t)r * m + c] = acc[q];
            Hinv[(size_t)c * m + r] = acc[q];
        }
    }
}

__global__ void fw_ctrl_init_from_slot_kernel(double* ctrl, const double* neg_logdet_slot) {
    for (int i = threadIdx.x; i < ACCBPG_FW_CTRL_DOUBLES; i += blockDim.x) ctrl[i] = 0.0;
    __syncthreads();
    if (threadIdx.x == 0) ctrl[C_LOGDET_HI] = -neg_logdet_slot[0];
}
__global__ void fw_zero_lo_kernel(double* ctrl) { ctrl[C_LOGDET_LO] = 0.0; }
__global__ void __launch_bounds__(256) negate_kernel(int64_t n, double* x) {
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) x[i] = -x[i];
}

}  // namespace accbpg

using namespace accbpg;

extern "C" {

size_t accbpg_fw_workspace_bytes(int m, int64_t n_local) {
    // dopt workspace (gram / factor / Linv / gradient partials) + v and u vectors
    size_t base = accbpg_dopt_workspace_bytes(m, n_local);
    const size_t nparts = (size_t)((n_local + 127) / 128) + 4096;        // selection candidates, one per selecting CTA
    // + the exchange tables of the persistent loop, each on a 128-byte boundary (accbpg_fw_run): u as (value, token)
    //   pairs (2 x m), records (2 x 256 CTAs x 128 B), flag words (2 x 256)
    return base + 2 * (((size_t)m + 31) / 32 * 32 * 8) + nparts * 64 + 128 + (size_t)4 * m * 8 + 128 + 2 * 256 * 128 +
           2 * 256 * 8;
}

// D_opt_alg.py:39-45 / :123-129:  M = V diag(x0) V^T, Hinv = M^{-1}, w_j = v_j^T Hinv v_j, log det M
int accbpg_fw_setup(void* ctx, void* stream, const double* V, int m, int64_t n, int64_t ldv, const double* x0,
                    void* ws, double* Hinv, double* w, double* ctrl) {
    Ctx* c = (Ctx*)ctx;
    cudaStream_t s = (cudaStream_t)stream;
    if (!c || !V || !x0 || !ws || !Hinv || !w || !ctrl) return arg_err("fw_setup: NULL pointer");
    ACCBPG_ON_DEVICE(c);
    double* slot = c->d_slots + 247;
    // func_grad(flag=2): slot <- -log det M, w <- gradient = -(v_j^T Hinv v_j); Linv stays in the workspace
    int rc = accbpg_dopt_func_grad(ctx, stream, V, m, n, ldv, x0, 2, ws, slot, w);
    if (rc) return rc;
    int g = grid_for(c, n, 256, 2, 8);
    negate_kernel<<<g, 256, 0, s>>>(n, w);
    ACCBPG_LAUNCHED("negate_kernel");
    fw_ctrl_init_from_slot_kernel<<<1, 32, 0, s>>>(ctrl, slot);
    ACCBPG_LAUNCHED("fw_ctrl_init");
    // Linv sits at a fixed offset of the dopt workspace: recover it through the same plan
    int mp = 0;
    size_t off = dopt_linv_offset(m, n, c->sm_count, &mp);
    const double* Linv = (const double*)((const char*)ws + off);
    dim3 grid((m + 31) / 32, (m + 31) / 32);
    fw_hinv_kernel<<<grid, 256, 0, s>>>(Linv, m, mp, Hinv);
    ACCBPG_LAUNCHED("fw_hinv_kernel");
    return ACCBPG_OK;
}

struct FwLaunch {
    FwParams p;
    int sel_grid, hv_grid, nblk, r1_ctas;
    size_t pass_smem;
    bool pass_vec;
    double* persist_mem;       // exchange tables of the persistent loop (inside the workspace)
};

static int fw_prepare(Ctx* c, const double* V, int m, int64_t n, int64_t ldv, int away, double eps, void* ws, double* Hinv,
                      double* x, double* w, double* ctrl, double* hist_F, double* hist_SP, double* hist_SN,
                      double* hist_T, FwLaunch* L) {
    if (m < 1 || n < 1 || ldv < n) return arg_err("fw: shape");
    size_t base = accbpg_dopt_workspace_bytes(m, n);
    double* v = (double*)((char*)ws + base);
    double* u = v + ((size_t)m + 31) / 32 * 32;
    FwCand* parts = (FwCand*)(u + ((size_t)m + 31) / 32 * 32);
    {
        const size_t nparts = (size_t)((n + 127) / 128) + 4096;
        uintptr_t a = reinterpret_cast<uintptr_t>(parts + nparts);
        L->persist_mem = reinterpret_cast<double*>((a + 127) / 128 * 128);
    }
    // block width: the smallest number of whole waves of (3 CTAs per SM) that covers n with <= 128 columns per CTA.
    // (Measured at 500 x 50000, round 2: sizing the waves by the kernel's real occupancy - 2 CTAs per SM at 110 registers, or
    // 3 with __launch_bounds__(256, 3) - gives 18.3 k / 18.6 k iterations per second against 19.2 k with this rule: the
    // iteration is bound by its serial chain - decision, column gather, u = Hinv v, tail - not by wave quantisation.)
    L->r1_ctas = c->sm_count / 4 < 1 ? 1 : c->sm_count / 4;
    int64_t per_wave = (int64_t)c->sm_count * 3;
    int64_t waves = (n + per_wave * FWP_COLS - 1) / (per_wave * FWP_COLS);
    int64_t width = (n + waves * per_wave - 1) / (waves * per_wave);
    width = (width + 1) / 2 * 2;
    if (width < 16) width = 16;
    if (width > FWP_COLS) width = FWP_COLS;
    const int64_t nblk64 = (n + width - 1) / width;
    if (nblk64 > 2000000000LL) return arg_err("fw: n too large");
    L->nblk = (int)nblk64;
    L->p.width = (int)width;
    L->sel_grid = grid_for(c, n, FW_THREADS, 4, 2);
    L->hv_grid = (m + 7) / 8;
    L->pass_smem = (size_t)m * sizeof(double);
    if (L->pass_smem > 160 * 1024) return arg_err("fw: m too large for the shared-memory copy of u");
    L->pass_vec = ((reinterpret_cast<uintptr_t>(V) & 15u) == 0) && (ldv % 2 == 0);
    if (L->pass_smem > 32 * 1024) {
        if (L->pass_vec) ACCBPG_CUDA(cudaFuncSetAttribute(fw_pass_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)L->pass_smem));
        else ACCBPG_CUDA(cudaFuncSetAttribute(fw_pass_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)L->pass_smem));
    }
    FwParams& p = L->p;
    p.V = V; p.m = m; p.n = n; p.ldv = ldv; p.x = x; p.w = w; p.Hinv = Hinv; p.u = u; p.v = v; p.ctrl = ctrl;
    p.hist_F = hist_F; p.hist_SP = hist_SP; p.hist_SN = hist_SN; p.hist_T = hist_T;
    p.parts = parts; p.counter = c->d_counter; p.away = away; p.eps = eps; p.nblk = L->nblk; p.nr1 = L->r1_ctas;
    p.k = 0; p.decide = 0; p.reverse = 0; p.cand_out = nullptr; p.col_offset = 0; p.sharded = 0; p.early = FWP_EARLY;
    p.peer.world = 0; p.peer.rank = 0;
    return ACCBPG_OK;
}

// one pass launch on the configuration the caller prepared (stream, launch attributes)
static cudaError_t fw_launch_pass(const FwLaunch& L, cudaLaunchConfig_t cfg, const FwParams& p) {
    cfg.gridDim = dim3(L.nblk + L.r1_ctas); cfg.blockDim = dim3(FWP_THREADS); cfg.dynamicSmemBytes = L.pass_smem;
    return cudaLaunchKernelEx(&cfg, L.pass_vec ? fw_pass_kernel<true> : fw_pass_kernel<false>, p);
}

// run iterations k_start .. k_start+k_count-1 (no-ops after the stop flag is raised), as one persistent launch when the
// ring of fw_persist_ring_kernel can run on this instance, else as the launch chain
//   select+decide(k_start);  then per iteration  u = Hinv v;  pass (+ rank-one update of Hinv, + decision of k+1)
// chained with programmatic dependent launch.
int accbpg_fw_run(void* ctx, void* stream, const double* V, int m, int64_t n, int64_t ldv, int away, double eps,
                  int k_start, int k_count, void* ws, double* Hinv, double* x, double* w, double* ctrl,
                  double* hist_F, double* hist_SP, double* hist_SN, double* hist_T) {
    Ctx* c = (Ctx*)ctx;
    cudaStream_t s = (cudaStream_t)stream;
    if (!c || !V || !ws || !Hinv || !x || !w || !ctrl || !hist_F || !hist_SP || !hist_SN || !hist_T)
        return arg_err("fw_run: NULL pointer");
    ACCBPG_ON_DEVICE(c);
    if (k_count < 0) return arg_err("fw_run: shape");
    if (k_count == 0) return ACCBPG_OK;
    FwLaunch L;
    int rc = fw_prepare(c, V, m, n, ldv, away, eps, ws, Hinv, x, w, ctrl, hist_F, hist_SP, hist_SN, hist_T, &L);
    if (rc) return rc;
    FwParams& p = L.p;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cudaLaunchConfig_t cfg = {};
    cfg.stream = s;
    cfg.attrs = attr;
    if (away && k_start > 0) {
        // D_opt_FW_away records log det of the *updated, rounded* Hinv by a fresh LU every iteration (D_opt_alg.py:136);
        // the determinant-lemma accumulator follows the exact update instead, so it is re-anchored on the actual Hinv
        // at every batch boundary (value-only Cholesky: -log det(Hinv) = log det(V X V^T))
        rc = accbpg_dopt_factor(ctx, stream, m, Hinv, nullptr, 0, ws, ctrl + C_LOGDET_HI);
        if (rc) return rc;
        fw_zero_lo_kernel<<<1, 1, 0, s>>>(ctrl);
        ACCBPG_LAUNCHED("fw_zero_lo_kernel");
    }
    // ---- one persistent launch for the whole batch when V is 16-byte aligned with even n and ldv, n < 2^31, m <= 4096,
    //      at least three ring stages fit in shared memory next to u and the two candidate columns, and the tensor map
    //      of V encodes
    if (L.pass_vec && n % 2 == 0 && n < (1LL << 31) && m <= 4096) {
        const int mpad = (m + 1) / 2 * 2;
        int max_optin = 0;
        cudaDeviceGetAttribute(&max_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, c->device);
        const long long room = (long long)max_optin - FWR_STATIC_SMEM - 3LL * mpad * 8;
        int stages = room > 0 ? (int)(room / FWR_STAGE_BYTES) : 0;
        if (stages > FWR_MAX_STAGES) stages = FWR_MAX_STAGES;
        // V in boxes of p.width columns x FWR_ROWS rows; p.width is even, so boxes packed in a stage stay 128-byte aligned
        CUtensorMap tmV;
        int ring_3d = 0;
        bool tmap = false;
        if (stages >= 3) {
            // one box over (columns, rows of a group, row groups) per stage when 4 | m, else one box per row group
            if (m % 4 == 0 &&
                encode_tmap_f64_3d(&tmV, V, (uint64_t)n, (uint64_t)(m / 4), 4, (uint64_t)ldv, (uint32_t)p.width, FWR_ROWS, 4)) {
                ring_3d = 1;
                tmap = true;
            } else {
                tmap = encode_tmap_f64_2d(&tmV, V, (uint64_t)n, (uint64_t)m, (uint64_t)ldv, (uint32_t)p.width, FWR_ROWS);
            }
        }
        if (tmap) {
            static bool attr_done[kMaxDevices] = {};
            if (c->device >= 0 && c->device < kMaxDevices && !attr_done[c->device]) {
                ACCBPG_CUDA(cudaFuncSetAttribute(fw_persist_ring_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                                 max_optin - FWR_STATIC_SMEM));
                attr_done[c->device] = true;
            }
            FwPersist q;
            q.ux = L.persist_mem;
            q.recs = reinterpret_cast<double*>((reinterpret_cast<uintptr_t>(q.ux + (size_t)4 * m) + 127) / 128 * 128);
            q.tok = reinterpret_cast<unsigned long long*>(q.recs + (size_t)2 * 256 * FWQ_REC_DOUBLES);
            static unsigned long long calls = 0;
            q.base = (++calls) << 24;
            q.G = c->sm_count < 256 ? c->sm_count : 256;
            q.k_start = k_start; q.k_count = k_count; q.stages = stages; q.ring_3d = ring_3d;
            p.k = k_start; p.decide = 1; p.reverse = 0;
            const size_t smem = (size_t)stages * FWR_STAGE_BYTES + (size_t)3 * mpad * 8;
            ProfScope ps(P_FW_BATCH, s);
            fw_persist_ring_kernel<<<q.G, FWS_THREADS, smem, s>>>(p, q, tmV);
            ACCBPG_LAUNCHED("fw_persist_ring_kernel");
            return ACCBPG_OK;
        }
    }
    // the first decision of the batch
    p.k = k_start; p.decide = 1; p.reverse = 0;
    cfg.gridDim = dim3(L.sel_grid); cfg.blockDim = dim3(FW_THREADS); cfg.dynamicSmemBytes = 0; cfg.numAttrs = 0;
    ACCBPG_CUDA(cudaLaunchKernelEx(&cfg, fw_select_kernel, p));
    ACCBPG_LAUNCHED("fw_select_kernel");
    for (int k = k_start; k < k_start + k_count; ++k) {
        ProfScope ps_iter(P_FW_ITER, s);
        cfg.gridDim = dim3(L.hv_grid); cfg.blockDim = dim3(256); cfg.dynamicSmemBytes = 0; cfg.numAttrs = 1;
        ACCBPG_CUDA(cudaLaunchKernelEx(&cfg, fw_hv_kernel, (const double*)Hinv, m, (const double*)p.v, p.u, (const double*)ctrl,
                                       (const unsigned long long*)nullptr, 0ULL));
        ACCBPG_LAUNCHED("fw_hv_kernel");
        p.k = k + 1;                                        // the tail decides the next iteration ...
        p.decide = (k + 1 < k_start + k_count) ? 1 : 0;     // ... except after the last pass of the batch
        p.reverse = k & 1;
        {
            ProfScope ps(P_FW_PASS, s);
            ACCBPG_CUDA(fw_launch_pass(L, cfg, p));
        }
        ACCBPG_LAUNCHED("fw_pass_kernel");
    }
    return ACCBPG_OK;
}

// ---- column-sharded building blocks (one rank's slab of V and slices of x, w; Hinv, ctrl and the histories replicated).
// Per iteration the caller runs:  accbpg_fw_decide(k, records of all ranks) -> sum v over the ranks ->
// accbpg_fw_step(k) [u = Hinv v; local pass + rank-one update; local record of the updated slice] -> all-gather records.
size_t accbpg_fw_record_bytes(void) { return sizeof(FwCand); }

int accbpg_fw_select_local(void* ctx, void* stream, int64_t n_local, int64_t col_offset, int away, const double* x,
                           const double* w, void* ws, int m, void* d_record_out) {
    Ctx* c = (Ctx*)ctx;
    cudaStream_t s = (cudaStream_t)stream;
    if (!c || !x || !w || !ws || !d_record_out) return arg_err("fw_select_local: NULL pointer");
    ACCBPG_ON_DEVICE(c);
    FwLaunch L;
    int rc = fw_prepare(c, x /* any aligned pointer: V is not read */, m, n_local, n_local, away, 0.0, ws, nullptr,
                        (double*)x, (double*)w, nullptr, nullptr, nullptr, nullptr, nullptr, &L);
    if (rc) return rc;
    L.p.decide = 2; L.p.cand_out = (FwCand*)d_record_out; L.p.col_offset = col_offset;
    fw_select_kernel<<<L.sel_grid, FW_THREADS, 0, s>>>(L.p);
    ACCBPG_LAUNCHED("fw_select_kernel");
    return ACCBPG_OK;
}

int accbpg_fw_decide(void* ctx, void* stream, const double* V, int m, int64_t n_local, int64_t ldv, int64_t col_offset,
                     int away, double eps, int k, const void* d_records, int world, void* ws, double* ctrl,
                     double* hist_F, double* hist_SP, double* hist_SN, double* hist_T, double* d_vcol) {
    Ctx* c = (Ctx*)ctx;
    cudaStream_t s = (cudaStream_t)stream;
    if (!c || !V || !d_records || !ws || !ctrl || !hist_F || !hist_SP || !hist_SN || !hist_T || !d_vcol)
        return arg_err("fw_decide: NULL pointer");
    ACCBPG_ON_DEVICE(c);
    if (world < 1) return arg_err("fw_decide: world");
    FwLaunch L;
    int rc = fw_prepare(c, V, m, n_local, ldv, away, eps, ws, nullptr, nullptr, nullptr, ctrl, hist_F, hist_SP, hist_SN,
                        hist_T, &L);
    if (rc) return rc;
    L.p.k = k; L.p.decide = 1; L.p.col_offset = col_offset; L.p.sharded = 1; L.p.v = d_vcol;
    fw_decide_kernel<<<1, FW_THREADS, 0, s>>>(L.p, (const FwCand*)d_records, world);
    ACCBPG_LAUNCHED("fw_decide_kernel");
    return ACCBPG_OK;
}

int accbpg_fw_step(void* ctx, void* stream, const double* V, int m, int64_t n_local, int64_t ldv, int64_t col_offset,
                   int away, int k, void* ws, double* Hinv, const double* d_vcol, double* x, double* w, double* ctrl,
                   void* d_record_out) {
    Ctx* c = (Ctx*)ctx;
    cudaStream_t s = (cudaStream_t)stream;
    if (!c || !V || !ws || !Hinv || !d_vcol || !x || !w || !ctrl || !d_record_out) return arg_err("fw_step: NULL pointer");
    ACCBPG_ON_DEVICE(c);
    FwLaunch L;
    int rc = fw_prepare(c, V, m, n_local, ldv, away, 0.0, ws, Hinv, x, w, ctrl, nullptr, nullptr, nullptr, nullptr, &L);
    if (rc) return rc;
    FwParams& p = L.p;
    fw_hv_kernel<<<L.hv_grid, 256, 0, s>>>(Hinv, m, d_vcol, p.u, ctrl, nullptr, 0ULL);
    ACCBPG_LAUNCHED("fw_hv_kernel");
    p.k = k + 1; p.decide = 2; p.reverse = k & 1; p.cand_out = (FwCand*)d_record_out; p.col_offset = col_offset;
    {
        cudaLaunchConfig_t cfg = {};
        cfg.stream = s;
        ProfScope ps(P_FW_PASS, s);
        ACCBPG_CUDA(fw_launch_pass(L, cfg, p));
    }
    ACCBPG_LAUNCHED("fw_pass_kernel");
    return ACCBPG_OK;
}

// The column-sharded loop with both exchanges over NVLink peer memory instead of NCCL: iterations k_start ..
// k_start+k_count-1 in one call, three launches each (programmatic dependent launch):
//   decide(k): wait for the `world` records of iteration k, merge in rank order, decide; the owner of the chosen column
//              stores it into every rank's column slot and releases the column flag
//   u = Hinv v: waits for the column flag
//   pass(k):   local pass + rank-one update; its tail stores this rank's record of iteration k+1 into every rank's
//              record slots and releases this rank's flag word there
// Records and columns are double-buffered on the iteration's parity; a rank can be one iteration ahead of a peer, never two.
int accbpg_fw_run_peer(void* ctx, void* stream, const double* V, int m, int64_t n_local, int64_t ldv, int64_t col_offset,
                       int away, double eps, int k_start, int k_count, int rank, int world, void* const* peer_rec,
                       void* const* peer_col, void* const* peer_flags, void* ws, double* Hinv, double* x, double* w,
                       double* ctrl, double* hist_F, double* hist_SP, double* hist_SN, double* hist_T) {
    Ctx* c = (Ctx*)ctx;
    cudaStream_t s = (cudaStream_t)stream;
    if (!c || !V || !ws || !Hinv || !x || !w || !ctrl || !hist_F || !hist_SP || !hist_SN || !hist_T || !peer_rec ||
        !peer_col || !peer_flags)
        return arg_err("fw_run_peer: NULL pointer");
    ACCBPG_ON_DEVICE(c);
    if (world < 1 || world > FW_MAX_PEERS || rank < 0 || rank >= world || k_count < 0 || k_start < 0)
        return arg_err("fw_run_peer: rank / world / range");
    if (k_count == 0) return ACCBPG_OK;
    FwLaunch L;
    int rc = fw_prepare(c, V, m, n_local, ldv, away, eps, ws, Hinv, x, w, ctrl, hist_F, hist_SP, hist_SN, hist_T, &L);
    if (rc) return rc;
    FwParams& p = L.p;
    for (int r = 0; r < world; ++r) {
        p.peer.rec[r] = (FwCand*)peer_rec[r]; p.peer.col[r] = (double*)peer_col[r];
        p.peer.flags[r] = (unsigned long long*)peer_flags[r];
        if (!p.peer.rec[r] || !p.peer.col[r] || !p.peer.flags[r]) return arg_err("fw_run_peer: NULL peer pointer");
    }
    p.peer.rank = rank; p.peer.world = world;
    p.col_offset = col_offset; p.sharded = 1;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cudaLaunchConfig_t cfg = {};
    cfg.stream = s;
    cfg.attrs = attr;
    if (away && k_start > 0) {           // re-anchor log det on the actual (replicated) Hinv, as accbpg_fw_run does
        rc = accbpg_dopt_factor(ctx, stream, m, Hinv, nullptr, 0, ws, ctrl + C_LOGDET_HI);
        if (rc) return rc;
        fw_zero_lo_kernel<<<1, 1, 0, s>>>(ctrl);
        ACCBPG_LAUNCHED("fw_zero_lo_kernel");
    }
    if (k_start == 0) {                  // the record of iteration 0; later ones come from the tail of the previous pass
        p.k = 0; p.decide = 2; p.reverse = 0;
        fw_select_kernel<<<L.sel_grid, FW_THREADS, 0, s>>>(p);
        ACCBPG_LAUNCHED("fw_select_kernel");
    }
    const unsigned long long* col_flag = p.peer.flags[rank] + world;
    for (int k = k_start; k < k_start + k_count; ++k) {
        const unsigned long long epoch = (unsigned long long)k + 1ULL;
        p.k = k; p.decide = 1;
        cfg.gridDim = dim3(1); cfg.blockDim = dim3(FW_THREADS); cfg.dynamicSmemBytes = 0; cfg.numAttrs = 1;
        ACCBPG_CUDA(cudaLaunchKernelEx(&cfg, fw_decide_peer_kernel, p));
        ACCBPG_LAUNCHED("fw_decide_peer_kernel");
        const double* vcol = p.peer.col[rank] + (size_t)(epoch & 1ULL) * m;
        cfg.gridDim = dim3(L.hv_grid); cfg.blockDim = dim3(256);
        ACCBPG_CUDA(cudaLaunchKernelEx(&cfg, fw_hv_kernel, (const double*)Hinv, m, vcol, p.u, (const double*)ctrl, col_flag, epoch));
        ACCBPG_LAUNCHED("fw_hv_kernel");
        p.k = k + 1; p.decide = 2; p.reverse = k & 1;
        {
            ProfScope ps(P_FW_PASS, s);
            ACCBPG_CUDA(fw_launch_pass(L, cfg, p));
        }
        ACCBPG_LAUNCHED("fw_pass_kernel");
    }
    return ACCBPG_OK;
}

// setup from an already summed Gram matrix M = V diag(x0) V^T (column-sharded: the caller all-reduces it):
// Hinv = M^{-1}, w_j = v_j^T Hinv v_j for the local columns, ctrl <- {log det M, not stopped}
int accbpg_fw_setup_from_gram(void* ctx, void* stream, const double* V, int m, int64_t n_local, int64_t ldv,
                              const double* M, void* ws, double* Hinv, double* w, double* ctrl) {
    Ctx* c = (Ctx*)ctx;
    cudaStream_t s = (cudaStream_t)stream;
    if (!c || !V || !M || !ws || !Hinv || !w || !ctrl) return arg_err("fw_setup_from_gram: NULL pointer");
    ACCBPG_ON_DEVICE(c);
    double* slot = c->d_slots + 247;
    int rc = accbpg_dopt_factor(ctx, stream, m, M, nullptr, 1, ws, slot);
    if (rc) return rc;
    rc = accbpg_dopt_grad(ctx, stream, V, m, n_local, ldv, ws, w);
    if (rc) return rc;
    int g = grid_for(c, n_local, 256, 2, 8);
    negate_kernel<<<g, 256, 0, s>>>(n_local, w);
    ACCBPG_LAUNCHED("negate_kernel");
    fw_ctrl_init_from_slot_kernel<<<1, 32, 0, s>>>(ctrl, slot);
    ACCBPG_LAUNCHED("fw_ctrl_init");
    int mp = 0;
    size_t off = dopt_linv_offset(m, n_local, c->sm_count, &mp);
    const double* Linv = (const double*)((const char*)ws + off);
    dim3 grid((m + 31) / 32, (m + 31) / 32);
    fw_hinv_kernel<<<grid, 256, 0, s>>>(Linv, m, mp, Hinv);
    ACCBPG_LAUNCHED("fw_hinv_kernel");
    return ACCBPG_OK;
}

}  // extern "C"
