// Shared device/host helpers for libaccbpg_b200.so (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include "../../include/accbpg_b200.h"

#ifndef __CUDA_ARCH__
#define ACCBPG_HOST_ONLY 1
#endif

namespace accbpg {

constexpr int kSlots = 256;          // result slots per context
constexpr int kMaxBlocks = 1184;     // 148 SMs x 8: upper bound on reduction grid sizes
constexpr int kPartialStride = kMaxBlocks;
constexpr int kPartialRows = 4;      // up to 4 simultaneous reduction outputs per kernel

struct Ctx {
    int device;
    int sm_count;
    double* d_slots;        // kSlots doubles
    uint32_t* d_status;     // status word
    double* d_partials;     // kPartialRows * kPartialStride doubles (double-buffered by the simplex kernel)
    long long* d_ipartials; // kPartialStride int64 (arg-reductions)
    unsigned int* d_counter;// "last block done" ticket
    double* h_slots;        // pinned mirror (kSlots doubles)
    uint32_t* h_status;     // pinned
    unsigned long long burg_calls;   // Burg-simplex root-finds launched: token base of the next one (one per call)
    double* d_burg_slots;   // their slot table (2 x 296 block-partial slots + 2 result slots, 4 doubles each)
    cudaStream_t side;      // side stream: a second latency-bound chain (Cholesky) runs next to the main one
    cudaEvent_t ev_fork, ev_join;
    cudaStream_t side2;     // early launches of the triangular GEMM, next to the tail of the Cholesky chain
    cudaEvent_t ev_early_done;
    // deferred reads (accbpg_ctx_read_async / _wait): a ring of pinned buffers, one event each
    double* h_ring;         // kReadRing * (kSlots + 1) doubles; the last double of a row carries the status word
    cudaEvent_t ring_ev[8];
    int ring_next;
};
constexpr int kReadRing = 8;

extern thread_local char g_err[512];
extern unsigned long long g_launches;

inline int set_err(const char* what, cudaError_t e) {
    snprintf(g_err, sizeof(g_err), "%s: %s", what, cudaGetErrorString(e));
    return ACCBPG_E_CUDA;
}
inline int arg_err(const char* what) {
    snprintf(g_err, sizeof(g_err), "bad argument: %s", what);
    return ACCBPG_E_ARG;
}

#define ACCBPG_CUDA(call)                                         \
    do {                                                          \
        cudaError_t e__ = (call);                                 \
        if (e__ != cudaSuccess) return accbpg::set_err(#call, e__); \
    } while (0)

#define ACCBPG_LAUNCHED(name)                                     \
    do {                                                          \
        ++accbpg::g_launches;                                     \
        cudaError_t e__ = cudaGetLastError();                     \
        if (e__ != cudaSuccess) return accbpg::set_err(name, e__); \
    } while (0)

// Every entry point runs on the device its context was created on, whatever device is current in the calling thread
// (the previous one is restored on return): `device=` of the Python operators works without torch.cuda.set_device.
struct DeviceGuard {
    int prev_; bool switched_;
    explicit DeviceGuard(int dev) : prev_(-1), switched_(false) {
        if (cudaGetDevice(&prev_) == cudaSuccess && prev_ != dev) switched_ = (cudaSetDevice(dev) == cudaSuccess);
    }
    ~DeviceGuard() { if (switched_) cudaSetDevice(prev_); }
};
#define ACCBPG_ON_DEVICE(c) accbpg::DeviceGuard dev_guard__((c)->device)
constexpr int kMaxDevices = 64;      // per-device once-flags (function attributes are per device)

// optional cudaEvent bracketing of selected launches (prof.cu); a no-op unless accbpg_prof_enable(1)
enum ProfId { P_SYRK = 0, P_SYRK_REDUCE, P_CHOL, P_TRINV, P_TRMM, P_GRAD_FIN, P_BURG_SIMPLEX, P_MATVEC, P_RMATVEC,
              P_FW_PASS, P_FW_ITER, P_GRAM_PUSH, P_GRAM_SUM, P_GG_PUSH, P_GG_WAIT, P_SCAL_SUM, P_FW_BATCH, P_COUNT };
struct ProfScope {
    ProfScope(int id, cudaStream_t s);
    ~ProfScope();
    int id_; cudaStream_t s_; bool active_;
};

// defined in dopt.cu: byte offset of Linv (mp x mp, zero padded) inside the dopt workspace
size_t dopt_linv_offset(int m, int64_t n, int sm_count, int* mp_out);
// defined in dopt.cu: 2-D FP64 tensor map (no swizzle) over a row-major matrix; `out` points to a CUtensorMap
bool encode_tmap_f64_2d(void* out, const double* base, uint64_t cols, uint64_t rows, uint64_t ld, uint32_t box_cols,
                        uint32_t box_rows);
bool encode_tmap_f64_3d(void* out, const double* base, uint64_t cols, uint64_t rows, uint64_t groups, uint64_t ld,
                        uint32_t box_cols, uint32_t box_rows, uint32_t box_groups);

inline int grid_for(const Ctx* c, int64_t n, int threads, int items_per_thread, int blocks_per_sm) {
    int64_t per_block = (int64_t)threads * items_per_thread;
    int64_t want = (n + per_block - 1) / per_block;
    int64_t cap = (int64_t)c->sm_count * blocks_per_sm;
    if (cap > kMaxBlocks) cap = kMaxBlocks;
    if (want > cap) want = cap;
    if (want < 1) want = 1;
    return (int)want;
}

#ifdef __CUDACC__
// ------------------------------------------------------------------ device helpers
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ double warp_min(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmin(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}
__device__ __forceinline__ double warp_max(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}

// Block-wide sum with a fixed tree; every thread gets the result.  blockDim.x multiple of 32, <= 1024.
__device__ __forceinline__ double block_sum(double v, double* sh /* >= 32 doubles */) {
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = blockDim.x >> 5;
    v = warp_sum(v);
    __syncthreads();                 // protect sh against a previous use
    if (lane == 0) sh[wid] = v;
    __syncthreads();
    double r = (lane < nw) ? sh[lane] : 0.0;
    r = warp_sum(r);
    return r;
}
__device__ __forceinline__ double block_min(double v, double* sh) {
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = blockDim.x >> 5;
    v = warp_min(v);
    __syncthreads();
    if (lane == 0) sh[wid] = v;
    __syncthreads();
    double r = (lane < nw) ? sh[lane] : __longlong_as_double(0x7ff0000000000000LL);
    r = warp_min(r);
    return r;
}
__device__ __forceinline__ double block_max(double v, double* sh) {
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = blockDim.x >> 5;
    v = warp_max(v);
    __syncthreads();
    if (lane == 0) sh[wid] = v;
    __syncthreads();
    double r = (lane < nw) ? sh[lane] : __longlong_as_double(0xfff0000000000000LL);
    r = warp_max(r);
    return r;
}

// "last block done" ticket: returns true in exactly one block (the last to arrive), after all other
// blocks' global writes issued before the call are visible to it.
__device__ __forceinline__ bool last_block_ticket(unsigned int* counter, bool* sh_flag) {
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) {
        unsigned int t = atomicAdd(counter, 1u);
        bool last = (t == gridDim.x * gridDim.y - 1);
        *sh_flag = last;
        if (last) *counter = 0u;     // re-arm for the next kernel on the stream
    }
    __syncthreads();
    bool last = *sh_flag;
    if (last) __threadfence();
    return last;
}

__device__ __forceinline__ double ld_cg(const double* p) { return __ldcg(p); }

// ---- scalar control of the one-launch accelerated solves (linreg_small.cu, small.cu).  Written with explicit
//      round-to-nearest operations: the two files are compiled with and without FMA contraction, and these values must
//      round like the host's Python arithmetic in both.
__device__ __forceinline__ unsigned long long ls_clock() {
    unsigned long long ns;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(ns));
    return ns;
}

// x**y.  The host's pow is correctly rounded at these exponents and CUDA's may be 2 ulp off; theta**gamma decides the
// gain line search and the G / Gain histories that the golden runs compare exactly (gamma = 2), so the exponents 1 and
// 2 take the exact forms.
__device__ __forceinline__ double la_pow(double x, double y) {
    return y == 1.0 ? x : y == 2.0 ? __dmul_rn(x, x) : pow(x, y);
}

// solve_theta: Newton solve of (1-t)/t^gamma = gainratio/theta^gamma from theta   (drivers.py, algorithms.py:75-91)
__device__ inline double la_solve_theta(double theta, double gamma, double gainratio) {
    const double ckg = __ddiv_rn(la_pow(theta, gamma), gainratio);
    double cta = theta;
    const double tol = __dmul_rn(1e-6, theta);
    for (;;) {
        const double phi = __dsub_rn(la_pow(cta, gamma), __dmul_rn(ckg, __dsub_rn(1.0, cta)));
        if (!(fabs(phi) > tol)) return cta;
        cta = __dsub_rn(cta, __ddiv_rn(phi, __dadd_rn(__dmul_rn(gamma, la_pow(cta, __dsub_rn(gamma, 1.0))), ckg)));
    }
}

// ---- flag words in NVLink peer memory (symmetric buffers mapped into every rank) ----
// A sender stores its payload into the receiver's buffer, fences at system scope and releases a monotonically increasing
// epoch into its flag word on the receiver; the receiver acquires the word before touching the payload.
__device__ __forceinline__ void st_release_sys(unsigned long long* p, unsigned long long v) {
    asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ unsigned long long ld_acquire_sys(const unsigned long long* p) {
    unsigned long long v;
    asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
// bounded by wall time: a peer that has not arrived after two minutes (protocol error, dead rank) traps this kernel
// instead of hanging the GPU; ordinary host-side skew between ranks (seconds) is waited out
__device__ __forceinline__ void peer_flag_wait(const unsigned long long* f, unsigned long long epoch) {
    unsigned long long t0 = 0;
    unsigned int spin = 0;
    while (ld_acquire_sys(f) < epoch) {
        __nanosleep(40);
        if ((++spin & 0xffffu) == 0) {
            unsigned long long now;
            asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(now));
            if (t0 == 0) t0 = now;
            else if (now - t0 > 120000000000ULL) __trap();
        }
    }
}
#endif  // __CUDACC__

}  // namespace accbpg
