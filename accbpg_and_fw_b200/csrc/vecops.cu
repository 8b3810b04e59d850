// Context management, iterate arithmetic, Burg / Shannon Bregman kernels and the simplex LMO.
// HBM-bound elementwise + reduction kernels; every reduction is a fixed tree (per-thread grid-stride
// partial -> warp shuffle -> block -> ordered sum of block partials by the last block to finish).
// Compiled with -fmad=false: expressions are rounded exactly as NumPy rounds them (no contraction).
#include "common.cuh"

namespace accbpg {
thread_local char g_err[512] = "";
unsigned long long g_launches = 0;

constexpr int kThreads = 256;
#define kInf (__longlong_as_double(0x7ff0000000000000LL))

// ---------------------------------------------------------------- generic multi-output sum reduction
// F::operator()(int64_t i, double* acc, uint32_t& st) accumulates element i into acc[0..NOUT)
template <int NOUT, class F>
__global__ void __launch_bounds__(kThreads) reduce_sum_kernel(int64_t n, F f, double* partials,
                                                              unsigned int* counter, double* out,
                                                              uint32_t* status) {
    __shared__ double sh[32];
    __shared__ bool is_last;
    double acc[NOUT];
#pragma unroll
    for (int o = 0; o < NOUT; ++o) acc[o] = 0.0;
    uint32_t st = 0;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) f(i, acc, st);
#pragma unroll
    for (int o = 0; o < NOUT; ++o) {
        double s = block_sum(acc[o], sh);
        if (threadIdx.x == 0) partials[o * kPartialStride + blockIdx.x] = s;
    }
    if (st) atomicOr(status, st);
    if (last_block_ticket(counter, &is_last)) {
#pragma unroll
        for (int o = 0; o < NOUT; ++o) {
            double s = 0.0;
            for (int b = threadIdx.x; b < (int)gridDim.x; b += blockDim.x)
                s += ld_cg(&partials[o * kPartialStride + b]);
            s = block_sum(s, sh);
            if (threadIdx.x == 0) out[o] = s;
        }
    }
}

template <int NOUT, class F>
static int launch_reduce(Ctx* c, cudaStream_t s, int64_t n, F f, double* d_out, const char* name) {
    int grid = grid_for(c, n, kThreads, 4, 4);
    reduce_sum_kernel<NOUT, F><<<grid, kThreads, 0, s>>>(n, f, c->d_partials, c->d_counter, d_out, c->d_status);
    ACCBPG_LAUNCHED(name);
    return ACCBPG_OK;
}

template <class F>
__global__ void __launch_bounds__(kThreads) map_kernel(int64_t n, F f, uint32_t* status) {
    uint32_t st = 0;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) f(i, st);
    if (st) atomicOr(status, st);
}

template <class F>
static int launch_map(Ctx* c, cudaStream_t s, int64_t n, F f, const char* name) {
    int grid = grid_for(c, n, kThreads, 2, 8);
    map_kernel<F><<<grid, kThreads, 0, s>>>(n, f, c->d_status);
    ACCBPG_LAUNCHED(name);
    return ACCBPG_OK;
}

// ---------------------------------------------------------------- functors: iterate arithmetic
struct AxpbyF {
    double a, b; const double *x, *y; double* out;
    __device__ void operator()(int64_t i, uint32_t&) const {
        out[i] = __dadd_rn(__dmul_rn(a, x[i]), __dmul_rn(b, y[i]));
    }
};
struct StepTowardF {   // x + a*(s - x)
    double a; const double *x, *s; double* out;
    __device__ void operator()(int64_t i, uint32_t&) const {
        double xi = x[i];
        out[i] = __dadd_rn(xi, __dmul_rn(a, __dsub_rn(s[i], xi)));
    }
};
struct DivideF {
    double denom; const double* x; double* out;
    __device__ void operator()(int64_t i, uint32_t&) const { out[i] = x[i] / denom; }
};
struct DotF {
    const double *x, *y;
    __device__ void operator()(int64_t i, double* acc, uint32_t&) const { acc[0] += __dmul_rn(x[i], y[i]); }
};
struct DotDiffF {
    const double *g, *a, *b;
    __device__ void operator()(int64_t i, double* acc, uint32_t&) const {
        acc[0] += __dmul_rn(g[i], __dsub_rn(a[i], b[i]));
    }
};
struct SqDistF {
    const double *a, *b;
    __device__ void operator()(int64_t i, double* acc, uint32_t&) const {
        const double d = __dsub_rn(a[i], b[i]);
        acc[0] += __dmul_rn(d, d);
    }
};
struct SumF {
    const double* x;
    __device__ void operator()(int64_t i, double* acc, uint32_t&) const { acc[0] += x[i]; }
};

// ---------------------------------------------------------------- functors: Burg entropy
struct BurgValueF {     // -sum log x
    const double* x;
    __device__ void operator()(int64_t i, double* acc, uint32_t& st) const {
        double xi = x[i];
        if (!(xi > 0.0)) st |= ACCBPG_ST_ARG_NOT_POS;
        acc[0] += -log(xi);      // sum of negated terms rounds exactly like the negated sum
    }
};
struct BurgGradF {
    const double* x; double* out;
    __device__ void operator()(int64_t i, uint32_t& st) const {
        double xi = x[i];
        if (!(xi > 0.0)) st |= ACCBPG_ST_ARG_NOT_POS;
        out[i] = -1.0 / xi;
    }
};
struct BurgDivF {       // sum (x/y - log(x/y) - 1)
    const double *x, *y;
    __device__ void operator()(int64_t i, double* acc, uint32_t& st) const {
        double xi = x[i], yi = y[i];
        if (!(xi > 0.0) || !(yi > 0.0)) st |= ACCBPG_ST_ARG_NOT_POS;
        double r = xi / yi;
        acc[0] += (r - log(r)) - 1.0;
    }
};
// shifted gradient s = g - L*(-1/y) (or g when y == nullptr)
__device__ __forceinline__ double burg_shift(const double* y, const double* g, double L, int64_t i, uint32_t& st) {
    double gi = g[i];
    if (y != nullptr) {
        double yi = y[i];
        if (!(yi > 0.0)) st |= ACCBPG_ST_ARG_NOT_POS;
        gi = gi - L * (-1.0 / yi);
    }
    return gi;
}
struct BurgProxF {
    int kind; double lamda, L, four_lamL, two_lamL; const double *y, *g; double* out;
    __device__ void operator()(int64_t i, uint32_t& st) const {
        double s = burg_shift(y, g, L, i, st);
        double r;
        if (kind == ACCBPG_BURG_PLAIN) {
            if (!(s > 0.0)) st |= ACCBPG_ST_PROX_NOT_POS;
            r = L / s;
        } else if (kind == ACCBPG_BURG_L1) {
            if (!(s > -lamda)) st |= ACCBPG_ST_PROX_NOT_POS;
            r = L / (lamda + s);
        } else {
            double gg = s / L;
            r = (sqrt(gg * gg + four_lamL) - gg) / two_lamL;
        }
        out[i] = r;
    }
};
struct BurgSimplexFinishDevF {
    const double* gg; const double* c; double* out;
    __device__ void operator()(int64_t i, uint32_t&) const { out[i] = 1.0 / (gg[i] + ld_cg(c)); }
};

// ---------------------------------------------------------------- functors: Shannon entropy
struct ShannonValueF {
    const double* x; double delta;
    __device__ void operator()(int64_t i, double* acc, uint32_t& st) const {
        double xi = x[i];
        if (!(xi >= 0.0)) st |= ACCBPG_ST_ARG_NEGATIVE;
        double xx = fmax(xi, delta);
        acc[0] += xx * log(xx);
    }
};
struct ShannonGradF {
    const double* x; double delta; double* out;
    __device__ void operator()(int64_t i, uint32_t& st) const {
        double xi = x[i];
        if (!(xi >= 0.0)) st |= ACCBPG_ST_ARG_NEGATIVE;
        out[i] = 1.0 + log(fmax(xi, delta));
    }
};
struct ShannonDivF {    // acc0 = sum x log((x+d)/(y+d)); acc1 = sum y; acc2 = sum x
    const double *x, *y; double delta;
    __device__ void operator()(int64_t i, double* acc, uint32_t& st) const {
        double xi = x[i], yi = y[i];
        if (!(xi >= 0.0) || !(yi >= 0.0)) st |= ACCBPG_ST_ARG_NEGATIVE;
        acc[0] += xi * log((xi + delta) / (yi + delta));
        acc[1] += yi;
        acc[2] += xi;
    }
};
__device__ __forceinline__ double shannon_point(const double* y, const double* g, double lamda, double L,
                                                int need_pos, int64_t i, uint32_t& st) {
    double gi = g[i];
    if (lamda != 0.0) gi = lamda + gi;          // ShannonEntropyL1: prox on (lamda + g)
    if (y == nullptr) return exp(-gi / L - 1.0);
    double yi = y[i];
    if (need_pos) { if (!(yi > 0.0)) st |= ACCBPG_ST_Y_NOT_POS; }
    else          { if (!(yi >= 0.0)) st |= ACCBPG_ST_ARG_NEGATIVE; }
    return yi * exp(-gi / L);
}
struct ShannonProxF {
    double lamda, L; const double *y, *g; double* out;
    __device__ void operator()(int64_t i, uint32_t& st) const { out[i] = shannon_point(y, g, lamda, L, 0, i, st); }
};
struct ShannonProxSumF {   // writes the un-normalised point and accumulates its sum
    double lamda, L; const double *y, *g; double* out;
    __device__ void operator()(int64_t i, double* acc, uint32_t& st) const {
        double v = shannon_point(y, g, lamda, L, 1, i, st);
        out[i] = v;
        acc[0] += v;
    }
};
struct DivideBySlotF {
    const double* x; const double* denom; double* out;
    __device__ void operator()(int64_t i, uint32_t&) const { out[i] = x[i] / ld_cg(denom); }
};

// ---------------------------------------------------------------- LMO functors
struct FillVertexF {
    double fill, radius; int64_t idx; double* out;
    __device__ void operator()(int64_t i, uint32_t&) const { out[i] = (i == idx) ? radius : fill; }
};
struct FillVertexSlotF {   // vertex index read from a device slot
    double fill, radius; const double* idx_slot; double* out;
    __device__ void operator()(int64_t i, uint32_t&) const {
        int64_t idx = (int64_t)ld_cg(idx_slot);
        out[i] = (i == idx) ? radius : fill;
    }
};
struct LmoLinfF {
    double radius; const double *g, *center; double* out;
    __device__ void operator()(int64_t i, uint32_t&) const {
        double gi = g[i];
        double sg = (gi > 0.0) ? 1.0 : ((gi < 0.0) ? -1.0 : gi);   // np.sign (nan stays nan)
        double ci = center ? center[i] : 0.0;
        out[i] = ci - radius * sg;
    }
};
struct LmoL2F {
    double radius, gnorm; const double *g, *center; double* out;
    __device__ void operator()(int64_t i, uint32_t&) const {
        double ci = center ? center[i] : 0.0;
        out[i] = ci - radius * g[i] / gnorm;      // (radius*g)/gnorm, left to right as in NumPy
    }
};
struct LmoBoxF {
    const double *g, *lo, *hi; double* out;
    __device__ void operator()(int64_t i, uint32_t&) const { out[i] = (g[i] < 0.0) ? hi[i] : lo[i]; }
};

// ---------------------------------------------------------------- min / max / arg-extremum
__global__ void __launch_bounds__(kThreads) minmax_kernel(int64_t n, const double* x, double* partials,
                                                          unsigned int* counter, double* out) {
    __shared__ double sh[32];
    __shared__ bool is_last;
    double lo = kInf, hi = -kInf;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        double v = x[i];
        lo = fmin(lo, v);
        hi = fmax(hi, v);
    }
    lo = block_min(lo, sh);
    hi = block_max(hi, sh);
    if (threadIdx.x == 0) {
        partials[blockIdx.x] = lo;
        partials[kPartialStride + blockIdx.x] = hi;
    }
    if (last_block_ticket(counter, &is_last)) {
        lo = kInf; hi = -kInf;
        for (int b = threadIdx.x; b < (int)gridDim.x; b += blockDim.x) {
            lo = fmin(lo, ld_cg(&partials[b]));
            hi = fmax(hi, ld_cg(&partials[kPartialStride + b]));
        }
        lo = block_min(lo, sh);
        hi = block_max(hi, sh);
        if (threadIdx.x == 0) { out[0] = lo; out[1] = hi; }
    }
}

// (value, first index) extremum.  sign = +1 argmin, -1 argmax (compares sign*x).
__device__ __forceinline__ void arg_combine(double& v, long long& i, double v2, long long i2) {
    if (v2 < v || (v2 == v && i2 < i)) { v = v2; i = i2; }
}
__device__ __forceinline__ void block_argmin(double& v, long long& i, double* shv, long long* shi) {
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = blockDim.x >> 5;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        double v2 = __shfl_xor_sync(0xffffffffu, v, o);
        long long i2 = __shfl_xor_sync(0xffffffffu, i, o);
        arg_combine(v, i, v2, i2);
    }
    __syncthreads();
    if (lane == 0) { shv[wid] = v; shi[wid] = i; }
    __syncthreads();
    v = (lane < nw) ? shv[lane] : kInf;
    i = (lane < nw) ? shi[lane] : 0x7fffffffffffffffLL;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        double v2 = __shfl_xor_sync(0xffffffffu, v, o);
        long long i2 = __shfl_xor_sync(0xffffffffu, i, o);
        arg_combine(v, i, v2, i2);
    }
}
__global__ void __launch_bounds__(kThreads) argext_kernel(int64_t n, const double* x, double sign,
                                                          double* partials, long long* ipartials,
                                                          unsigned int* counter, double* out) {
    __shared__ double shv[32];
    __shared__ long long shi[32];
    __shared__ bool is_last;
    double v = kInf;
    long long idx = 0x7fffffffffffffffLL;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    // i only grows, so a tie is taken only while idx still holds the empty marker: the first index wins inside a thread,
    // and a thread whose elements are all +inf (after the sign) reports the first of them, as np.argmin does
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride)
        arg_combine(v, idx, sign * x[i], i);
    block_argmin(v, idx, shv, shi);
    if (threadIdx.x == 0) { partials[blockIdx.x] = v; ipartials[blockIdx.x] = idx; }
    if (last_block_ticket(counter, &is_last)) {
        v = kInf; idx = 0x7fffffffffffffffLL;
        for (int b = threadIdx.x; b < (int)gridDim.x; b += blockDim.x)
            arg_combine(v, idx, ld_cg(&partials[b]), __ldcg(&ipartials[b]));
        block_argmin(v, idx, shv, shi);
        if (threadIdx.x == 0) { out[0] = sign * v; out[1] = (double)idx; }
    }
}

// ---------------------------------------------------------------- Burg-simplex root-find
// The recurrence of functions.py:341-356 in one persistent kernel with the iterate held in REGISTERS; the grid-wide sums
// of a step go through a slot table (burgx_round) instead of grid.sync + a second pass over L2.  Sums are added in block
// order, so the multiplier c and the step counts do not depend on which block finishes first, and a Newton step costs one
// store -> poll hop (two above 128 blocks) instead of a grid barrier plus an L2 round trip.
// Launched as an ordinary kernel with at most as many blocks as are co-resident on an idle GPU: blocks that are not
// resident yet are waited for by the others (nothing they wait for depends on this kernel), cooperative launches of
// different streams would serialise against each other.
constexpr int kBurgThreads = 512;
constexpr int kBurgSlot = 4;                           // doubles per slot: a, token, b, token
constexpr int kBurgMaxG = kMaxBlocks / 4;              // 296 blocks at most
struct BurgX {
    double* tab;                                       // the slot table (layout at burgx_round)
    int onehop;                                        // every block gathers the block partials itself
    unsigned long long base;                           // token of round r is base + r (unique per call on this table)
};

// a value and its round token travel together in one aligned 16-byte word (single transaction: the reader sees both or
// neither), so a delivery needs no fence and a poll is one load
__device__ __forceinline__ void st_pair(double* p, double v, unsigned long long tok) {
    asm volatile("st.volatile.global.v2.u64 [%0], {%1, %2};" ::"l"(p), "l"(__double_as_longlong(v)), "l"(tok) : "memory");
}
__device__ __forceinline__ void ld_pair(const double* p, unsigned long long& v, unsigned long long& tok) {
    asm volatile("ld.volatile.global.v2.u64 {%0, %1}, [%2];" : "=l"(v), "=l"(tok) : "l"(p) : "memory");
}

// wait until the 16-byte word at p carries `token`; returns its value
__device__ __forceinline__ double wait_pair(const double* p, unsigned long long token) {
    unsigned long long v, tk, t0 = 0;
    unsigned spin = 0;
    for (;;) {
        ld_pair(p, v, tk);
        if (tk == token) return __longlong_as_double((long long)v);
        __nanosleep(32);
        if ((++spin & 0x3ffu) == 0) {
            unsigned long long now;
            asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(now));
            if (t0 == 0) t0 = now;
            else if (now - t0 > 4000000000ULL) __trap();
        }
    }
}

// gather `count` slots (a, b pairs) starting at `slots` in increasing index: the 32 lanes of one warp take slots
// lane, lane + 32, ... (four in flight each), add them up in that order, then a fixed shuffle tree
template <bool IS_MIN>
__device__ __forceinline__ void gather_slots(const double* slots, int count, unsigned long long token, double& ra,
                                             double& rb) {
    const int lane = threadIdx.x & 31;
    double sa = IS_MIN ? kInf : 0.0, sb = 0.0;
    for (int q0 = lane; q0 < count; q0 += 32 * 4) {
        double va[4], vb[4];
        unsigned done = 0, want = 0;
#pragma unroll
        for (int u = 0; u < 4; ++u) if (q0 + 32 * u < count) want |= 1u << u;
        unsigned long long t0 = 0;
        unsigned spin = 0;
        while (done != want) {
            unsigned long long wa[4], ta[4], wb[4], tb[4];
#pragma unroll
            for (int u = 0; u < 4; ++u)
                if ((want & ~done) & (1u << u)) {
                    const double* sl = slots + (size_t)(q0 + 32 * u) * kBurgSlot;
                    ld_pair(sl, wa[u], ta[u]);
                    ld_pair(sl + 2, wb[u], tb[u]);
                }
#pragma unroll
            for (int u = 0; u < 4; ++u)
                if (((want & ~done) & (1u << u)) && ta[u] == token && tb[u] == token) {
                    va[u] = __longlong_as_double((long long)wa[u]);
                    vb[u] = __longlong_as_double((long long)wb[u]);
                    done |= 1u << u;
                }
            if (done != want && (++spin & 0x3ffu) == 0) {
                unsigned long long now;
                asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(now));
                if (t0 == 0) t0 = now;
                else if (now - t0 > 4000000000ULL) __trap();
            }
        }
#pragma unroll
        for (int u = 0; u < 4; ++u)
            if (want & (1u << u)) {
                if (IS_MIN) sa = fmin(sa, va[u]);
                else { sa += va[u]; sb += vb[u]; }
            }
    }
    if (IS_MIN) { ra = warp_min(sa); rb = 0.0; }
    else { ra = warp_sum(sa); rb = warp_sum(sb); }
}

// One exchange round; (a, b) are this thread's partial sums (IS_MIN: a is a partial minimum, b unused).  One block adds
// its warps' sums in shared memory.  Otherwise every block stores its partials into its slot, and then
//   onehop: every block gathers all block partials itself (G polls per block and round);
//   leader: block 0 gathers them and stores the total into the result slot, which every other block polls,
// so that above 128 blocks no cache line is polled by more than one block except the result slot.  Both forms add the
// block partials in the same order (same lanes, same shuffle tree), so they give the same bits.  Every store carries
// its value and the round's token in one 16-byte word: no fences.  Table (kBurgSlot doubles per slot): [2][kBurgMaxG]
// block partials, then [2] result slots, both indexed by the round's parity.
constexpr int kBurgOffR = 2 * kBurgMaxG;
constexpr int kBurgTableSlots = kBurgOffR + 2;
template <bool IS_MIN>
__device__ __forceinline__ void burgx_round(const BurgX& X, int round, double a, double b, double* sh, int& flip, double& ra,
                                            double& rb) {
    const int G = gridDim.x, tid = threadIdx.x, lane = tid & 31, wid = tid >> 5, nw = blockDim.x >> 5;
    double* s = sh + flip * 64;
    flip ^= 1;
    if (IS_MIN) {
        a = warp_min(a);
        if (lane == 0) s[wid] = a;
    } else {
        a = warp_sum(a);
        b = warp_sum(b);
        if (lane == 0) { s[wid] = a; s[32 + wid] = b; }
    }
    __syncthreads();
    if (G == 1) {                                      // one block holds the whole vector (n <= 4096): no exchange at all
        if (IS_MIN) { ra = warp_min((lane < nw) ? s[lane] : kInf); rb = 0.0; }
        else { ra = warp_sum((lane < nw) ? s[lane] : 0.0); rb = warp_sum((lane < nw) ? s[32 + lane] : 0.0); }
        return;                                        // (the buffers alternate, so the next round needs no second barrier)
    }
    if (wid == 0) {
        double ba, bb = 0.0;
        if (IS_MIN) ba = warp_min((lane < nw) ? s[lane] : kInf);
        else { ba = warp_sum((lane < nw) ? s[lane] : 0.0); bb = warp_sum((lane < nw) ? s[32 + lane] : 0.0); }
        const unsigned long long token = X.base + (unsigned long long)round;
        const int par = round & 1;
        const double* parts = X.tab + (size_t)par * kBurgMaxG * kBurgSlot;
        double* res = X.tab + ((size_t)kBurgOffR + par) * kBurgSlot;
        if (lane == 0) {
            double* dst = X.tab + ((size_t)par * kBurgMaxG + blockIdx.x) * kBurgSlot;
            st_pair(dst, ba, token);
            st_pair(dst + 2, bb, token);
        }
        double ta, tb;
        if (X.onehop) {
            gather_slots<IS_MIN>(parts, G, token, ta, tb);
        } else if (blockIdx.x == 0) {                  // the leader adds the block partials and posts the total
            gather_slots<IS_MIN>(parts, G, token, ta, tb);
            if (lane == 0) { st_pair(res, ta, token); st_pair(res + 2, tb, token); }
        } else if (lane == 0) {                        // only lane 0's total is used below
            ta = wait_pair(res, token);
            tb = wait_pair(res + 2, token);
        }
        double* o = sh + flip * 64;                    // the other buffer: nobody reads it before the barrier below
        if (lane == 0) { o[0] = ta; o[1] = tb; }
    }
    __syncthreads();
    ra = sh[flip * 64];
    rb = sh[flip * 64 + 1];
    flip ^= 1;
}

// EPT > 0: each thread keeps EPT elements of gg in registers (n <= EPT * G * 512); EPT == 0: gg lives in `out` and is
// re-read every round (any n)
template <int EPT>
__global__ void __launch_bounds__(kBurgThreads) burg_simplex_x_kernel(int64_t n, const double* y, const double* g, double L,
                                                                      double eps, double* out, double* info,
                                                                      uint32_t* status, BurgX X, const double* gg_in) {
    __shared__ double sh[128];
    const int tid = threadIdx.x;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    const int64_t first = (int64_t)blockIdx.x * blockDim.x + tid;
    uint32_t st = 0;
    double gg[EPT > 0 ? EPT : 1];
    double lo = kInf;
    // gg_in != NULL: root-find only, on a ready vector gg (the gathered slices of a column-sharded run; padding entries are
    // +inf and drop out of the minimum and of both sums); nothing but `info` is written then
    const double* ggsrc = gg_in ? gg_in : out;
    if (EPT > 0) {
#pragma unroll
        for (int e = 0; e < EPT; ++e) {
            const int64_t i = first + e * stride;
            gg[e] = kInf;                               // padding drops out of the minimum and of both sums
            if (i < n) { gg[e] = gg_in ? gg_in[i] : burg_shift(y, g, L, i, st) / L; lo = fmin(lo, gg[e]); }
        }
    } else if (gg_in) {
        for (int64_t i = first; i < n; i += stride) lo = fmin(lo, gg_in[i]);
    } else {
        for (int64_t i = first; i < n; i += stride) {
            const double v = burg_shift(y, g, L, i, st) / L;
            out[i] = v;
            lo = fmin(lo, v);
        }
    }
    int flip = 0, round = 0;
    double s1, s2;
    burgx_round<true>(X, round++, lo, 0.0, sh, flip, s1, s2);
    const double cmin = -s1;
    double c = cmin + 1.0;
    int nbis = 0, nnewton = 0;
    auto sums = [&](double cc, double& a, double& b) {
        a = 0.0; b = 0.0;
        if (EPT > 0) {
#pragma unroll
            for (int e = 0; e < EPT; ++e) {
                const double t = gg[e] + cc;
                a += 1.0 / t;
                b += -1.0 / (t * t);
            }
        } else {
            for (int64_t i = first; i < n; i += stride) {
                const double t = ggsrc[i] + cc;
                a += 1.0 / t;
                b += -1.0 / (t * t);
            }
        }
    };
    // bisection: halve toward cmin until sum 1/(gg+c) - 1 >= 0   (functions.py:344-346)
    for (;;) {
        double a, b;
        sums(c, a, b);
        burgx_round<false>(X, round++, a, b, sh, flip, s1, s2);
        if (s1 - 1.0 < 0.0 && nbis < 2000) { c = (cmin + c) / 2.0; ++nbis; }
        else break;
    }
    double fc = s1 - 1.0;
    // Newton  (functions.py:348-354); s2 already holds fpc at the current c
    while (fabs(fc) > eps) {
        const double fpc = s2;
        const double cn = c - fc / fpc;
        if (c - cn == 0.0) break;
        c = cn;
        double a, b;
        sums(c, a, b);
        burgx_round<false>(X, round++, a, b, sh, flip, s1, s2);
        fc = s1 - 1.0;
        if (++nnewton >= 200) { st |= ACCBPG_ST_NEWTON_MAXIT; break; }
    }
    if (gg_in) {
        // root-find only
    } else if (EPT > 0) {
#pragma unroll
        for (int e = 0; e < EPT; ++e) {
            const int64_t i = first + e * stride;
            if (i < n) out[i] = 1.0 / (gg[e] + c);
        }
    } else {
        for (int64_t i = first; i < n; i += stride) out[i] = 1.0 / (out[i] + c);
    }
    if (st) atomicOr(status, st);
    if (info != nullptr && blockIdx.x == 0 && tid == 0) {
        info[0] = (double)nbis; info[1] = (double)nnewton; info[2] = c;
    }
}

__global__ void __launch_bounds__(kThreads) burg_prepare_kernel(int64_t n, const double* y, const double* g,
                                                                double L, double* gg, double* partials,
                                                                unsigned int* counter, double* out,
                                                                uint32_t* status) {
    __shared__ double sh[32];
    __shared__ bool is_last;
    uint32_t st = 0;
    double lo = kInf;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        double v = burg_shift(y, g, L, i, st) / L;
        gg[i] = v;
        lo = fmin(lo, v);
    }
    lo = block_min(lo, sh);
    if (threadIdx.x == 0) partials[blockIdx.x] = lo;
    if (st) atomicOr(status, st);
    if (last_block_ticket(counter, &is_last)) {
        lo = kInf;
        for (int b = threadIdx.x; b < (int)gridDim.x; b += blockDim.x) lo = fmin(lo, ld_cg(&partials[b]));
        lo = block_min(lo, sh);
        if (threadIdx.x == 0) out[0] = lo;
    }
}

// ---- exchanges over NVLink peer memory (column-sharded runs; buffers mapped into every rank) ----
constexpr int kMaxPeerRanks = 16;
constexpr int kPeerScalars = 16;
struct PeerVec {
    double* buf[kMaxPeerRanks];                    // every rank's receive buffer, double-buffered on the epoch's parity
    unsigned long long* flags[kMaxPeerRanks];      // every rank's flag words, one per sender
    int rank, world;
    unsigned long long epoch;
};

// gg = (g [+ L/y]) / L for this rank's slice, padded with +inf up to `width`, stored locally (for the finishing map) and
// into segment `rank` of every rank's gathered vector; the last CTA releases this rank's flag word on every rank
__global__ void __launch_bounds__(kThreads) burg_prepare_push_kernel(int64_t n, int64_t width, const double* y,
                                                                     const double* g, double L, double* gg, PeerVec pv,
                                                                     unsigned int* counter, uint32_t* status) {
    __shared__ bool is_last;
    uint32_t st = 0;
    const size_t seg = ((size_t)(pv.epoch & 1ULL) * pv.world + pv.rank) * (size_t)width;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < width; i += stride) {
        double v = kInf;
        if (i < n) { v = burg_shift(y, g, L, i, st) / L; gg[i] = v; }
        for (int r = 0; r < pv.world; ++r) {
            int q = pv.rank + r;
            if (q >= pv.world) q -= pv.world;
            pv.buf[q][seg + i] = v;
        }
    }
    if (st) atomicOr(status, st);
    __threadfence_system();
    if (last_block_ticket(counter, &is_last)) {
        __threadfence_system();
        if ((int)threadIdx.x < pv.world) st_release_sys(pv.flags[threadIdx.x] + pv.rank, pv.epoch);
    }
}

// stream-ordered wait: returns once every one of the `count` flag words has reached `epoch`
__global__ void peer_wait_kernel(const unsigned long long* flags, int count, unsigned long long epoch) {
    if ((int)threadIdx.x < count) peer_flag_wait(flags + threadIdx.x, epoch);
}

// The last slot of a table row carries the sender's status word: every rank ORs all of them into its own, so a
// precondition violated on one rank's slice raises the same exception on every rank at the same fetch.
__global__ void __launch_bounds__(64) peer_sum_scalars_kernel(const double* in, double* out, int count, PeerVec pv,
                                                              uint32_t* status) {
    const int t = threadIdx.x;
    const size_t row = (size_t)(pv.epoch & 1ULL) * pv.world;
    if (t < pv.world) {
        double* dst = pv.buf[t] + (row + pv.rank) * kPeerScalars;
        for (int k = 0; k < count; ++k) dst[k] = in[k];
        dst[kPeerScalars - 1] = (double)__ldcg(status);
        __threadfence_system();
        st_release_sys(pv.flags[t] + pv.rank, pv.epoch);
    }
    __syncthreads();
    if (t < pv.world) peer_flag_wait(pv.flags[pv.rank] + t, pv.epoch);
    __syncthreads();
    const double* tab = pv.buf[pv.rank] + row * kPeerScalars;
    if (t < count) {
        double s = 0.0;
        for (int r = 0; r < pv.world; ++r) s += __ldcg(tab + (size_t)r * kPeerScalars + t);
        out[t] = s;
    } else if (t == kPeerScalars - 1) {
        uint32_t all = 0;
        for (int r = 0; r < pv.world; ++r) all |= (uint32_t)__ldcg(tab + (size_t)r * kPeerScalars + kPeerScalars - 1);
        if (all) atomicOr(status, all);
    }
}

// status word <-> a float64 slot (the NCCL / gloo fallback of the same exchange carries it through an all-reduce(max))
__global__ void status_export_kernel(const uint32_t* status, double* slot) { slot[0] = (double)__ldcg(status); }
__global__ void status_import_kernel(uint32_t* status, const double* slot) {
    const uint32_t v = (uint32_t)__ldcg(slot);
    if (v) atomicOr(status, v);
}

// lowest (value, global index) pair over the ranks: the same single-CTA exchange with a different combine.  Ties in the
// value go to the lowest index, so the selected vertex does not depend on the number of ranks (functions_lmo.py:153-158).
__global__ void __launch_bounds__(64) peer_argmin_pair_kernel(double* pair, PeerVec pv) {
    const int t = threadIdx.x;
    const size_t row = (size_t)(pv.epoch & 1ULL) * pv.world;
    if (t < pv.world) {
        double* dst = pv.buf[t] + (row + pv.rank) * kPeerScalars;
        dst[0] = pair[0]; dst[1] = pair[1];
        __threadfence_system();
        st_release_sys(pv.flags[t] + pv.rank, pv.epoch);
    }
    __syncthreads();
    if (t < pv.world) peer_flag_wait(pv.flags[pv.rank] + t, pv.epoch);
    __syncthreads();
    if (t == 0) {
        const double* tab = pv.buf[pv.rank] + row * kPeerScalars;
        double bv = __ldcg(tab), bi = __ldcg(tab + 1);
        for (int r = 1; r < pv.world; ++r) {
            const double v = __ldcg(tab + (size_t)r * kPeerScalars), i = __ldcg(tab + (size_t)r * kPeerScalars + 1);
            if (v < bv || (v == bv && i < bi)) { bv = v; bi = i; }
        }
        pair[0] = bv; pair[1] = bi;
    }
}

// all-reduce(sum) of an n-vector over peer memory: push this rank's vector into slot `rank` of every rank's buffer ...
__global__ void __launch_bounds__(kThreads) peer_vec_push_kernel(const double* x, int64_t n, int64_t cap, PeerVec pv,
                                                                 unsigned int* counter) {
    __shared__ bool is_last;
    const size_t seg = ((size_t)(pv.epoch & 1ULL) * pv.world + pv.rank) * (size_t)cap;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        const double v = x[i];
        for (int r = 0; r < pv.world; ++r) {
            int q = pv.rank + r;
            if (q >= pv.world) q -= pv.world;
            pv.buf[q][seg + i] = v;
        }
    }
    __threadfence_system();
    if (last_block_ticket(counter, &is_last)) {
        __threadfence_system();
        if ((int)threadIdx.x < pv.world) st_release_sys(pv.flags[threadIdx.x] + pv.rank, pv.epoch);
    }
}
// ... and, once all `world` vectors have arrived, add them up in rank order (every rank forms the same sums)
__global__ void __launch_bounds__(kThreads) peer_vec_sum_kernel(double* x, int64_t n, int64_t cap, PeerVec pv) {
    if ((int)threadIdx.x < pv.world) peer_flag_wait(pv.flags[pv.rank] + threadIdx.x, pv.epoch);
    __syncthreads();
    const double* src = pv.buf[pv.rank] + (size_t)(pv.epoch & 1ULL) * pv.world * (size_t)cap;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        double s = 0.0;
        for (int r = 0; r < pv.world; ++r) s += __ldcg(src + (size_t)r * cap + i);
        x[i] = s;
    }
}

}  // namespace accbpg

using namespace accbpg;

// ======================================================================== C ABI
extern "C" {

int accbpg_abi_version(void) { return ACCBPG_ABI_VERSION; }
const char* accbpg_last_error(void) { return g_err; }
uint64_t accbpg_launch_count(void) { return g_launches; }

int accbpg_ctx_create(void** out) {
    if (!out) return arg_err("ctx out pointer is NULL");
    Ctx* c = new Ctx();
    ACCBPG_CUDA(cudaGetDevice(&c->device));
    ACCBPG_CUDA(cudaDeviceGetAttribute(&c->sm_count, cudaDevAttrMultiProcessorCount, c->device));
    ACCBPG_CUDA(cudaMalloc(&c->d_slots, kSlots * sizeof(double)));
    ACCBPG_CUDA(cudaMalloc(&c->d_status, 256));
    ACCBPG_CUDA(cudaMalloc(&c->d_partials, (size_t)kPartialRows * kPartialStride * sizeof(double)));
    ACCBPG_CUDA(cudaMalloc(&c->d_ipartials, (size_t)kPartialStride * sizeof(long long)));
    ACCBPG_CUDA(cudaMalloc(&c->d_counter, 256));
    ACCBPG_CUDA(cudaMalloc(&c->d_burg_slots, (size_t)kBurgTableSlots * kBurgSlot * sizeof(double)));
    ACCBPG_CUDA(cudaMemset(c->d_burg_slots, 0, (size_t)kBurgTableSlots * kBurgSlot * sizeof(double)));
    ACCBPG_CUDA(cudaMemset(c->d_slots, 0, kSlots * sizeof(double)));
    ACCBPG_CUDA(cudaMemset(c->d_status, 0, 256));
    ACCBPG_CUDA(cudaMemset(c->d_counter, 0, 256));
    ACCBPG_CUDA(cudaMallocHost(&c->h_slots, kSlots * sizeof(double)));
    ACCBPG_CUDA(cudaMallocHost(&c->h_status, 64));
    ACCBPG_CUDA(cudaMallocHost(&c->h_ring, (size_t)kReadRing * (kSlots + 1) * sizeof(double)));
    for (int i = 0; i < kReadRing; ++i) ACCBPG_CUDA(cudaEventCreateWithFlags(&c->ring_ev[i], cudaEventDisableTiming));
    c->ring_next = 0;
    ACCBPG_CUDA(cudaStreamCreateWithFlags(&c->side, cudaStreamNonBlocking));
    ACCBPG_CUDA(cudaEventCreateWithFlags(&c->ev_fork, cudaEventDisableTiming));
    ACCBPG_CUDA(cudaEventCreateWithFlags(&c->ev_join, cudaEventDisableTiming));
    ACCBPG_CUDA(cudaStreamCreateWithFlags(&c->side2, cudaStreamNonBlocking));
    ACCBPG_CUDA(cudaEventCreateWithFlags(&c->ev_early_done, cudaEventDisableTiming));
    c->burg_calls = 0;
    ACCBPG_CUDA(cudaDeviceSynchronize());
    *out = c;
    return ACCBPG_OK;
}

int accbpg_ctx_destroy(void* ctx) {
    Ctx* c = (Ctx*)ctx;
    if (!c) return ACCBPG_OK;
    ACCBPG_ON_DEVICE(c);
    cudaFree(c->d_slots); cudaFree(c->d_status); cudaFree(c->d_partials);
    cudaFree(c->d_ipartials); cudaFree(c->d_counter); cudaFree(c->d_burg_slots);
    cudaFreeHost(c->h_slots); cudaFreeHost(c->h_status);
    cudaStreamDestroy(c->side); cudaEventDestroy(c->ev_fork); cudaEventDestroy(c->ev_join);
    cudaStreamDestroy(c->side2); cudaEventDestroy(c->ev_early_done);
    delete c;
    return ACCBPG_OK;
}

double* accbpg_ctx_slots(void* ctx) { return ctx ? ((Ctx*)ctx)->d_slots : nullptr; }
int accbpg_ctx_sm_count(void* ctx) { return ctx ? ((Ctx*)ctx)->sm_count : 0; }

int accbpg_ctx_read(void* ctx, void* stream, const double* d_src, int count, double* h_out, uint32_t* h_status) {
    Ctx* c = (Ctx*)ctx;
    cudaStream_t s = (cudaStream_t)stream;
    if (!c) return arg_err("ctx is NULL");
    ACCBPG_ON_DEVICE(c);
    if (count < 0 || count > kSlots) return arg_err("ctx_read: count must be in [0, 256]");
    if (count > 0 && (!d_src || !h_out)) return arg_err("ctx_read: NULL pointer");
    if (count > 0)
        ACCBPG_CUDA(cudaMemcpyAsync(c->h_slots, d_src, count * sizeof(double), cudaMemcpyDeviceToHost, s));
    ACCBPG_CUDA(cudaMemcpyAsync(c->h_status, c->d_status, sizeof(uint32_t), cudaMemcpyDeviceToHost, s));
    ACCBPG_CUDA(cudaMemsetAsync(c->d_status, 0, sizeof(uint32_t), s));
    ACCBPG_CUDA(cudaStreamSynchronize(s));
    for (int i = 0; i < count; ++i) h_out[i] = c->h_slots[i];
    if (h_status) *h_status = *c->h_status;
    return ACCBPG_OK;
}

int accbpg_ctx_read_async(void* ctx, void* stream, const double* d_src, int count, int* ticket) {
    Ctx* c = (Ctx*)ctx;
    cudaStream_t s = (cudaStream_t)stream;
    if (!c || !ticket) return arg_err("ctx_read_async: NULL pointer");
    ACCBPG_ON_DEVICE(c);
    if (count < 0 || count > kSlots) return arg_err("ctx_read_async: count must be in [0, 256]");
    if (count > 0 && !d_src) return arg_err("ctx_read_async: NULL pointer");
    const int t = c->ring_next;
    c->ring_next = (t + 1) % kReadRing;
    double* row = c->h_ring + (size_t)t * (kSlots + 1);
    if (count > 0) ACCBPG_CUDA(cudaMemcpyAsync(row, d_src, count * sizeof(double), cudaMemcpyDeviceToHost, s));
    ACCBPG_CUDA(cudaMemcpyAsync(row + kSlots, c->d_status, sizeof(uint32_t), cudaMemcpyDeviceToHost, s));
    ACCBPG_CUDA(cudaMemsetAsync(c->d_status, 0, sizeof(uint32_t), s));
    ACCBPG_CUDA(cudaEventRecord(c->ring_ev[t], s));
    *ticket = t;
    return ACCBPG_OK;
}
int accbpg_ctx_read_wait(void* ctx, int ticket, int count, double* h_out, uint32_t* h_status) {
    Ctx* c = (Ctx*)ctx;
    if (!c) return arg_err("ctx is NULL");
    ACCBPG_ON_DEVICE(c);
    if (ticket < 0 || ticket >= kReadRing) return arg_err("ctx_read_wait: bad ticket");
    if (count < 0 || count > kSlots || (count > 0 && !h_out)) return arg_err("ctx_read_wait: count / NULL pointer");
    ACCBPG_CUDA(cudaEventSynchronize(c->ring_ev[ticket]));
    const double* row = c->h_ring + (size_t)ticket * (kSlots + 1);
    for (int i = 0; i < count; ++i) h_out[i] = row[i];
    if (h_status) *h_status = *reinterpret_cast<const uint32_t*>(row + kSlots);
    return ACCBPG_OK;
}

#define CTX_STREAM                       \
    Ctx* c = (Ctx*)ctx;                  \
    cudaStream_t s = (cudaStream_t)stream; \
    if (!c) return arg_err("ctx is NULL"); \
    ACCBPG_ON_DEVICE(c);                 \
    if (n < 0) return arg_err("n < 0");

int accbpg_vec_axpby(void* ctx, void* stream, int64_t n, double a, const double* x, double b, const double* y,
                     double* out) {
    CTX_STREAM
    if (n == 0) return ACCBPG_OK;
    return launch_map(c, s, n, AxpbyF{a, b, x, y, out}, "vec_axpby");
}
int accbpg_vec_step_toward(void* ctx, void* stream, int64_t n, const double* x, const double* sv, double a,
                           double* out) {
    CTX_STREAM
    if (n == 0) return ACCBPG_OK;
    return launch_map(c, s, n, StepTowardF{a, x, sv, out}, "vec_step_toward");
}
int accbpg_vec_divide(void* ctx, void* stream, int64_t n, const double* x, double denom, double* out) {
    CTX_STREAM
    if (n == 0) return ACCBPG_OK;
    return launch_map(c, s, n, DivideF{denom, x, out}, "vec_divide");
}
int accbpg_vec_dot(void* ctx, void* stream, int64_t n, const double* x, const double* y, double* d_out) {
    CTX_STREAM
    return launch_reduce<1>(c, s, n, DotF{x, y}, d_out, "vec_dot");
}
int accbpg_vec_dot_diff(void* ctx, void* stream, int64_t n, const double* g, const double* a, const double* b,
                        double* d_out) {
    CTX_STREAM
    return launch_reduce<1>(c, s, n, DotDiffF{g, a, b}, d_out, "vec_dot_diff");
}
// out[i][j] = u[i] * v[j]   (p x q, row-major)
__global__ void __launch_bounds__(256) outer_kernel(const double* __restrict__ u, int64_t p, const double* __restrict__ v,
                                                    int64_t q, double* __restrict__ out) {
    const int64_t total = p * q, stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += stride) {
        const int64_t i = e / q, j = e - i * q;
        out[e] = u[i] * v[j];
    }
}
int accbpg_mat_outer(void* ctx, void* stream, int64_t p, const double* u, int64_t q, const double* v, double* out) {
    Ctx* c = (Ctx*)ctx;
    cudaStream_t s = (cudaStream_t)stream;
    if (!c || !u || !v || !out) return arg_err("mat_outer: NULL pointer");
    ACCBPG_ON_DEVICE(c);
    if (p < 1 || q < 1) return arg_err("mat_outer: shape");
    int grid = grid_for(c, p * q, 256, 2, 8);
    outer_kernel<<<grid, 256, 0, s>>>(u, p, v, q, out);
    ACCBPG_LAUNCHED("outer_kernel");
    return ACCBPG_OK;
}
int accbpg_vec_sqdist(void* ctx, void* stream, int64_t n, const double* a, const double* b, double* d_out) {
    CTX_STREAM
    return launch_reduce<1>(c, s, n, SqDistF{a, b}, d_out, "vec_sqdist");
}
int accbpg_vec_sum(void* ctx, void* stream, int64_t n, const double* x, double* d_out) {
    CTX_STREAM
    return launch_reduce<1>(c, s, n, SumF{x}, d_out, "vec_sum");
}
int accbpg_vec_minmax(void* ctx, void* stream, int64_t n, const double* x, double* d_out) {
    CTX_STREAM
    int grid = grid_for(c, n, kThreads, 4, 4);
    minmax_kernel<<<grid, kThreads, 0, s>>>(n, x, c->d_partials, c->d_counter, d_out);
    ACCBPG_LAUNCHED("vec_minmax");
    return ACCBPG_OK;
}
int accbpg_vec_argext(void* ctx, void* stream, int64_t n, const double* x, int want_max, double* d_out) {
    CTX_STREAM
    int grid = grid_for(c, n, kThreads, 4, 4);
    argext_kernel<<<grid, kThreads, 0, s>>>(n, x, want_max ? -1.0 : 1.0, c->d_partials, c->d_ipartials,
                                            c->d_counter, d_out);
    ACCBPG_LAUNCHED("vec_argext");
    return ACCBPG_OK;
}

// ---- Burg
int accbpg_burg_value(void* ctx, void* stream, int64_t n, const double* x, double* d_out) {
    CTX_STREAM
    return launch_reduce<1>(c, s, n, BurgValueF{x}, d_out, "burg_value");
}
int accbpg_burg_gradient(void* ctx, void* stream, int64_t n, const double* x, double* out) {
    CTX_STREAM
    if (n == 0) return ACCBPG_OK;
    return launch_map(c, s, n, BurgGradF{x, out}, "burg_gradient");
}
int accbpg_burg_divergence(void* ctx, void* stream, int64_t n, const double* x, const double* y, double* d_out) {
    CTX_STREAM
    return launch_reduce<1>(c, s, n, BurgDivF{x, y}, d_out, "burg_divergence");
}
int accbpg_burg_prox(void* ctx, void* stream, int64_t n, int kind, double lamda, const double* y,
                     const double* g, double L, double* out) {
    CTX_STREAM
    if (kind < 0 || kind > 2) return arg_err("burg kind");
    if (!(L > 0.0)) return arg_err("L must be positive");
    if (n == 0) return ACCBPG_OK;
    double lamL = lamda / L;
    return launch_map(c, s, n, BurgProxF{kind, lamda, L, 4 * lamL, 2 * lamL, y, g, out}, "burg_prox");
}
static int burgx_launch(Ctx* c, cudaStream_t s, int64_t n, const double* y, const double* g, double L, double eps,
                        double* out, double* info, const double* gg_in = nullptr) {
    int64_t want = (n + kBurgThreads - 1) / kBurgThreads;
    static int per_sm_x = 0;                           // co-resident blocks per SM of burg_simplex_x_kernel (all variants)
    if (per_sm_x == 0) {
        int a = 0, b = 0;
        ACCBPG_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&a, burg_simplex_x_kernel<8>, kBurgThreads, 0));
        ACCBPG_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&b, burg_simplex_x_kernel<0>, kBurgThreads, 0));
        per_sm_x = a < b ? a : b;
        if (per_sm_x < 1) return arg_err("burg_simplex_x_kernel cannot be made resident");
        if (per_sm_x > 2) per_sm_x = 2;
    }
    int cap = c->sm_count * per_sm_x;
    if (cap > kBurgMaxG) cap = kBurgMaxG;
    int grid = (int)(want < cap ? want : cap);
    if (grid < 1) grid = 1;
    if (n <= 8 * kBurgThreads) grid = 1;               // small vectors: one block, no exchange (shared memory only)
    const int64_t per = (n + (int64_t)grid * kBurgThreads - 1) / ((int64_t)grid * kBurgThreads);
    BurgX X;
    X.tab = c->d_burg_slots;
    X.base = (++c->burg_calls) << 12;                  // at most 2201 rounds per call
    // one hop costs G polls per block and round (G^2 in all): measured 2 us faster per call at 98 blocks, slower at 196
    X.onehop = grid <= 128;
    ProfScope ps(P_BURG_SIMPLEX, s);
    if (per <= 1) burg_simplex_x_kernel<1><<<grid, kBurgThreads, 0, s>>>(n, y, g, L, eps, out, info, c->d_status, X, gg_in);
    else if (per <= 2) burg_simplex_x_kernel<2><<<grid, kBurgThreads, 0, s>>>(n, y, g, L, eps, out, info, c->d_status, X, gg_in);
    else if (per <= 3) burg_simplex_x_kernel<3><<<grid, kBurgThreads, 0, s>>>(n, y, g, L, eps, out, info, c->d_status, X, gg_in);
    else if (per <= 4) burg_simplex_x_kernel<4><<<grid, kBurgThreads, 0, s>>>(n, y, g, L, eps, out, info, c->d_status, X, gg_in);
    else if (per <= 6) burg_simplex_x_kernel<6><<<grid, kBurgThreads, 0, s>>>(n, y, g, L, eps, out, info, c->d_status, X, gg_in);
    else if (per <= 8) burg_simplex_x_kernel<8><<<grid, kBurgThreads, 0, s>>>(n, y, g, L, eps, out, info, c->d_status, X, gg_in);
    else burg_simplex_x_kernel<0><<<grid, kBurgThreads, 0, s>>>(n, y, g, L, eps, out, info, c->d_status, X, gg_in);
    ACCBPG_LAUNCHED("burg_simplex_x_kernel");
    return ACCBPG_OK;
}

int accbpg_burg_simplex_prox(void* ctx, void* stream, int64_t n, const double* y, const double* g, double L,
                             double eps, double* out, double* info) {
    CTX_STREAM
    if (!(L > 0.0)) return arg_err("L must be positive");
    if (n < 1) return arg_err("n must be >= 1");
    return burgx_launch(c, s, n, y, g, L, eps, out, info);
}
int accbpg_burg_simplex_root(void* ctx, void* stream, int64_t n, const double* gg, double eps, double* d_info) {
    CTX_STREAM
    if (!gg || !d_info) return arg_err("burg_simplex_root: NULL pointer");
    if (n < 1) return arg_err("n must be >= 1");
    return burgx_launch(c, s, n, nullptr, nullptr, 1.0, eps, nullptr, d_info, gg);
}

// Column-sharded prox over NVLink peer memory, in two calls.  push: the prepare kernel stores this rank's (padded) slice
// of gg straight into every rank's gathered vector and releases a flag word there.  root: a one-warp kernel waits for
// the `world` flags (so the root-find's blocks never spin on a peer while they occupy the GPU), then the
// root-find runs on the gathered vector.
static int peer_vec_fill(PeerVec& pv, int rank, int world, void* const* bufs, void* const* flags, uint64_t epoch,
                         const char* what) {
    if (!bufs || !flags) return arg_err(what);
    if (world < 1 || world > kMaxPeerRanks || rank < 0 || rank >= world || epoch < 1) return arg_err(what);
    for (int r = 0; r < world; ++r) {
        pv.buf[r] = (double*)bufs[r]; pv.flags[r] = (unsigned long long*)flags[r];
        if (!pv.buf[r] || !pv.flags[r]) return arg_err(what);
    }
    pv.rank = rank; pv.world = world; pv.epoch = epoch;
    return ACCBPG_OK;
}
int accbpg_burg_simplex_push_peer(void* ctx, void* stream, int64_t n_local, int64_t width, const double* y,
                                  const double* g, double L, int rank, int world, void* const* peer_gg,
                                  void* const* peer_flags, uint64_t epoch, double* d_gg_local) {
    Ctx* c = (Ctx*)ctx;
    cudaStream_t s = (cudaStream_t)stream;
    if (!c) return arg_err("ctx is NULL");
    ACCBPG_ON_DEVICE(c);
    if (!g || !d_gg_local) return arg_err("burg_simplex_push_peer: NULL pointer");
    if (!(L > 0.0)) return arg_err("L must be positive");
    if (n_local < 0 || width < n_local || width < 1) return arg_err("burg_simplex_push_peer: width");
    PeerVec pv;
    int rc = peer_vec_fill(pv, rank, world, peer_gg, peer_flags, epoch, "burg_simplex_push_peer: peer tables / rank / epoch");
    if (rc) return rc;
    int pgrid = grid_for(c, width, kThreads, 4, 4);
    ProfScope ps(P_GG_PUSH, s);
    burg_prepare_push_kernel<<<pgrid, kThreads, 0, s>>>(n_local, width, y, g, L, d_gg_local, pv, c->d_counter + 18,
                                                        c->d_status);
    ACCBPG_LAUNCHED("burg_prepare_push_kernel");
    return ACCBPG_OK;
}
int accbpg_burg_simplex_root_peer(void* ctx, void* stream, int64_t width, double eps, int rank, int world,
                                  void* const* peer_gg, void* const* peer_flags, uint64_t epoch, double* d_info) {
    Ctx* c = (Ctx*)ctx;
    cudaStream_t s = (cudaStream_t)stream;
    if (!c) return arg_err("ctx is NULL");
    ACCBPG_ON_DEVICE(c);
    if (!d_info || width < 1) return arg_err("burg_simplex_root_peer: NULL pointer / width");
    PeerVec pv;
    int rc = peer_vec_fill(pv, rank, world, peer_gg, peer_flags, epoch, "burg_simplex_root_peer: peer tables / rank / epoch");
    if (rc) return rc;
    {
        ProfScope psw(P_GG_WAIT, s);
        peer_wait_kernel<<<1, 32, 0, s>>>(pv.flags[rank], world, epoch);
        ACCBPG_LAUNCHED("peer_wait_kernel");
    }
    const int64_t n = width * world;
    const double* gg = pv.buf[rank] + (size_t)(epoch & 1ULL) * (size_t)n;
    return burgx_launch(c, s, n, nullptr, nullptr, 1.0, eps, nullptr, d_info, gg);
}

// Sum `count` (<= 15) per-rank partial scalars over the ranks through peer memory, in rank order: one CTA stores its
// values (and its status word) into slot `rank` of every rank's table, releases its flag word there, waits for the
// `world` flags of its own table and adds the rows up (every rank forms the same sums).  d_out may equal d_in.
int accbpg_peer_sum_scalars(void* ctx, void* stream, const double* d_in, double* d_out, int count, int rank, int world,
                            void* const* peer_tab, void* const* peer_flags, uint64_t epoch) {
    Ctx* c = (Ctx*)ctx;
    cudaStream_t s = (cudaStream_t)stream;
    if (!c) return arg_err("ctx is NULL");
    ACCBPG_ON_DEVICE(c);
    if (!d_in || !d_out || !peer_tab || !peer_flags) return arg_err("peer_sum_scalars: NULL pointer");
    if (count < 1 || count > kPeerScalars - 1 || world < 1 || world > kMaxPeerRanks || rank < 0 || rank >= world || epoch < 1)
        return arg_err("peer_sum_scalars: count / rank / world / epoch");
    PeerVec pv;
    for (int r = 0; r < world; ++r) {
        pv.buf[r] = (double*)peer_tab[r]; pv.flags[r] = (unsigned long long*)peer_flags[r];
        if (!pv.buf[r] || !pv.flags[r]) return arg_err("peer_sum_scalars: NULL peer pointer");
    }
    pv.rank = rank; pv.world = world; pv.epoch = epoch;
    ProfScope ps(P_SCAL_SUM, s);
    peer_sum_scalars_kernel<<<1, 64, 0, s>>>(d_in, d_out, count, pv, c->d_status);
    ACCBPG_LAUNCHED("peer_sum_scalars_kernel");
    return ACCBPG_OK;
}

int accbpg_ctx_status_export(void* ctx, void* stream, double* d_slot) {
    Ctx* c = (Ctx*)ctx;
    cudaStream_t s = (cudaStream_t)stream;
    if (!c || !d_slot) return arg_err("ctx_status_export: NULL pointer");
    ACCBPG_ON_DEVICE(c);
    status_export_kernel<<<1, 1, 0, s>>>(c->d_status, d_slot);
    ACCBPG_LAUNCHED("status_export_kernel");
    return ACCBPG_OK;
}
int accbpg_ctx_status_import(void* ctx, void* stream, const double* d_slot) {
    Ctx* c = (Ctx*)ctx;
    cudaStream_t s = (cudaStream_t)stream;
    if (!c || !d_slot) return arg_err("ctx_status_import: NULL pointer");
    ACCBPG_ON_DEVICE(c);
    status_import_kernel<<<1, 1, 0, s>>>(c->d_status, d_slot);
    ACCBPG_LAUNCHED("status_import_kernel");
    return ACCBPG_OK;
}

// lowest (value, global index) over the ranks, in place on the two doubles at d_pair (tables as accbpg_peer_sum_scalars)
int accbpg_peer_argmin_pair(void* ctx, void* stream, double* d_pair, int rank, int world, void* const* peer_tab,
                            void* const* peer_flags, uint64_t epoch) {
    Ctx* c = (Ctx*)ctx;
    cudaStream_t s = (cudaStream_t)stream;
    if (!c) return arg_err("ctx is NULL");
    ACCBPG_ON_DEVICE(c);
    if (!d_pair) return arg_err("peer_argmin_pair: NULL pointer");
    PeerVec pv;
    int rc = peer_vec_fill(pv, rank, world, peer_tab, peer_flags, epoch, "peer_argmin_pair: peer tables / rank / epoch");
    if (rc) return rc;
    peer_argmin_pair_kernel<<<1, 64, 0, s>>>(d_pair, pv);
    ACCBPG_LAUNCHED("peer_argmin_pair_kernel");
    return ACCBPG_OK;
}

// all-reduce(sum), in place, of the n doubles at d_x over peer memory; every rank's buffer holds 2*world slots of `cap`
// doubles (cap >= n)
int accbpg_peer_sum_vector(void* ctx, void* stream, double* d_x, int64_t n, int64_t cap, int rank, int world,
                           void* const* peer_buf, void* const* peer_flags, uint64_t epoch) {
    Ctx* c = (Ctx*)ctx;
    cudaStream_t s = (cudaStream_t)stream;
    if (!c) return arg_err("ctx is NULL");
    ACCBPG_ON_DEVICE(c);
    if (!d_x || n < 1 || cap < n) return arg_err("peer_sum_vector: NULL pointer / n / cap");
    PeerVec pv;
    int rc = peer_vec_fill(pv, rank, world, peer_buf, peer_flags, epoch, "peer_sum_vector: peer tables / rank / epoch");
    if (rc) return rc;
    int grid = grid_for(c, n, kThreads, 4, 4);
    peer_vec_push_kernel<<<grid, kThreads, 0, s>>>(d_x, n, cap, pv, c->d_counter + 19);
    ACCBPG_LAUNCHED("peer_vec_push_kernel");
    peer_vec_sum_kernel<<<grid, kThreads, 0, s>>>(d_x, n, cap, pv);
    ACCBPG_LAUNCHED("peer_vec_sum_kernel");
    return ACCBPG_OK;
}
int accbpg_burg_simplex_finish_dev(void* ctx, void* stream, int64_t n, const double* gg, const double* d_c, double* out) {
    CTX_STREAM
    if (n == 0) return ACCBPG_OK;
    if (!gg || !d_c || !out) return arg_err("burg_simplex_finish_dev: NULL pointer");
    return launch_map(c, s, n, BurgSimplexFinishDevF{gg, d_c, out}, "burg_simplex_finish_dev");
}
int accbpg_burg_simplex_prepare(void* ctx, void* stream, int64_t n, const double* y, const double* g, double L,
                                double* gg, double* d_out) {
    CTX_STREAM
    if (!(L > 0.0)) return arg_err("L must be positive");
    int grid = grid_for(c, n, kThreads, 4, 4);
    burg_prepare_kernel<<<grid, kThreads, 0, s>>>(n, y, g, L, gg, c->d_partials, c->d_counter, d_out, c->d_status);
    ACCBPG_LAUNCHED("burg_simplex_prepare");
    return ACCBPG_OK;
}

// ---- Shannon
int accbpg_shannon_value(void* ctx, void* stream, int64_t n, const double* x, double delta, double* d_out) {
    CTX_STREAM
    return launch_reduce<1>(c, s, n, ShannonValueF{x, delta}, d_out, "shannon_value");
}
int accbpg_shannon_gradient(void* ctx, void* stream, int64_t n, const double* x, double delta, double* out) {
    CTX_STREAM
    if (n == 0) return ACCBPG_OK;
    return launch_map(c, s, n, ShannonGradF{x, delta, out}, "shannon_gradient");
}
__global__ void shannon_div_finish_kernel(const double* t, double* o) {   // sum(x log ..) + (sum y - sum x)
    o[0] = t[0] + (t[1] - t[2]);
}
int accbpg_shannon_divergence(void* ctx, void* stream, int64_t n, const double* x, const double* y, double delta,
                              double* d_out) {
    CTX_STREAM
    // three sums land in scratch slots 250..252, then are combined into d_out
    double* tmp = c->d_slots + 250;
    int rc = launch_reduce<3>(c, s, n, ShannonDivF{x, y, delta}, tmp, "shannon_divergence");
    if (rc) return rc;
    shannon_div_finish_kernel<<<1, 1, 0, s>>>(tmp, d_out);
    ACCBPG_LAUNCHED("shannon_div_finish");
    return ACCBPG_OK;
}
int accbpg_shannon_prox(void* ctx, void* stream, int64_t n, double lamda, const double* y, const double* g,
                        double L, int normalize, double* out, double* d_sum_out) {
    CTX_STREAM
    if (!(L > 0.0)) return arg_err("L must be positive");
    if (n == 0) return ACCBPG_OK;
    if (!normalize) return launch_map(c, s, n, ShannonProxF{lamda, L, y, g, out}, "shannon_prox");
    double* sum_slot = d_sum_out ? d_sum_out : (c->d_slots + 253);
    int rc = launch_reduce<1>(c, s, n, ShannonProxSumF{lamda, L, y, g, out}, sum_slot, "shannon_prox_sum");
    if (rc || normalize == 2) return rc;
    return launch_map(c, s, n, DivideBySlotF{out, sum_slot, out}, "shannon_normalize");
}

// ---- LMO
int accbpg_lmo_simplex(void* ctx, void* stream, int64_t n, const double* g, double radius, double* sv,
                       double* d_out) {
    CTX_STREAM
    if (n < 1) return arg_err("n must be >= 1");
    double* slot = d_out ? d_out : (c->d_slots + 254);
    int rc = accbpg_vec_argext(ctx, stream, n, g, 0, slot);
    if (rc) return rc;
    return launch_map(c, s, n, FillVertexSlotF{1e-15, radius, slot + 1, sv}, "lmo_simplex_fill");
}
int accbpg_lmo_fill_vertex(void* ctx, void* stream, int64_t n, double fill, int64_t idx, double radius,
                           double* sv) {
    CTX_STREAM
    if (n == 0) return ACCBPG_OK;
    return launch_map(c, s, n, FillVertexF{fill, radius, idx, sv}, "lmo_fill_vertex");
}
int accbpg_lmo_linf(void* ctx, void* stream, int64_t n, const double* g, double radius, const double* center,
                    double* sv) {
    CTX_STREAM
    if (n == 0) return ACCBPG_OK;
    return launch_map(c, s, n, LmoLinfF{radius, g, center, sv}, "lmo_linf");
}
int accbpg_lmo_l2(void* ctx, void* stream, int64_t n, const double* g, double radius, double gnorm,
                  const double* center, double* sv) {
    CTX_STREAM
    if (n == 0) return ACCBPG_OK;
    return launch_map(c, s, n, LmoL2F{radius, gnorm, g, center, sv}, "lmo_l2");
}
int accbpg_lmo_box(void* ctx, void* stream, int64_t n, const double* g, const double* lo, const double* hi,
                   double* sv) {
    CTX_STREAM
    if (n == 0) return ACCBPG_OK;
    return launch_map(c, s, n, LmoBoxF{g, lo, hi, sv}, "lmo_box");
}

}  // extern "C"
