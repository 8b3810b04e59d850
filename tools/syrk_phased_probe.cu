// Column-phased SYRK probe: can the Gram matrix M = H diag(x) H^T be delivered one 128-wide tile column at a time, in
// order, at (almost) the speed of the one-wave SYRK?  If so, the Cholesky chain could run its first block columns
// underneath the SYRK (DESIGN section 13).
//
// The probe kernel walks the lower 128x128 tiles in column order (column 0: tiles (0,0),(1,0),..; then column 1, ...)
// cut into units of 512 columns of H.  A static plan hands every CTA of a persistent grid one contiguous range of units
// of about equal cost (diagonal unit: 0.5625), so a CTA covers one or a few tiles; the TMA / mbarrier ring of
// syrk_tma_kernel keeps running across tile boundaries.  At the end of each run of one tile a CTA stores its partial
// tile; the last CTA to finish a tile (ticket per tile) sums the partials in CTA order, writes M for the tile and counts
// the tile into its column; the CTA that completes a tile column stamps %globaltimer.  Printed: the one-wave SYRK and
// SYRK + split reduction at plans for 148 / 140 / 132 SMs, the phased kernel on grids of 148 / 140 / 132 CTAs, and the
// time at which each tile column of M became final.  Two schedules (below): contiguous unit ranges per CTA, and the
// grid sweeping the unit list in order.
//
//   nvcc -gencode arch=compute_100a,code=sm_100a -O3 -std=c++17 -o tools/build/syrk_phased_probe tools/syrk_phased_probe.cu \
//        accbpg_and_fw_b200/csrc/build/{chol,prof,vecops,small,sparse,linreg,fw}.o
//   tools/build/syrk_phased_probe [m n]
#include "../accbpg_and_fw_b200/csrc/dopt.cu"
#include <algorithm>
#include <cmath>
#include <vector>
using namespace accbpg;

constexpr int PH_UNIT = 32;     // k-slabs per unit (512 columns)

// schedules: CONTIG - CTA b owns the contiguous unit range [ubeg[b], ubeg[b+1]) (a run per tile it touches);
//            IN_ORDER - CTA b owns units b, b + grid, b + 2 grid, ... (the grid sweeps the list in column order; every
//            unit is a partial of its own)
struct PhParams {
    double* P;                  // partial tiles, BM*BN each, slots of tile t at slot0[t] .. slot0[t] + nruns[t]
    double* M;
    int m, nt, U, KT;
    const int* ubeg;            // [grid + 1] unit range of every CTA
    const int* slot0;           // [T]
    const int* first_cta;       // [T] lowest CTA that covers tile t
    const int* nruns;           // [T] CTAs that cover tile t
    unsigned int* ticket;       // [T]
    unsigned int* colcnt;       // [nt]
    unsigned long long* stamps; // [grid] CTA start, [grid] CTA end, [nt] tile column final, [T] tile's last partial in
};

__device__ __forceinline__ unsigned long long gtimer() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}

// tile t of the column-major list of lower tiles: column c holds tile rows c .. nt-1
__host__ __device__ inline void ph_tile(int t, int nt, int& bi, int& bj) {
    int c = 0;
    while (t >= nt - c) { t -= nt - c; ++c; }
    bj = c; bi = c + t;
}

__device__ __forceinline__ void mbar_arrive_relaxed_n(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.arrive.relaxed.cta.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}

template <bool IN_ORDER>
__global__ void __launch_bounds__(GEMM_THREADS, 1)
syrk_phased_kernel(PhParams p, const __grid_constant__ CUtensorMap tmH, const __grid_constant__ CUtensorMap tmX) {
    extern __shared__ unsigned char smem_raw[];
    __shared__ int sh_last;
    const uint32_t smem0 = ((uint32_t)__cvta_generic_to_shared(smem_raw) + 1023u) & ~1023u;
    const uint32_t bars = smem0 + TMA_STAGES * TMA_STAGE_BYTES;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int g = lane >> 2, t = lane & 3;
    const int b = blockIdx.x, G = gridDim.x;
    if (tid == 0) p.stamps[b] = gtimer();
    // run r of this CTA: tile run_tile(r), slabs [ks, ke)
    const int TU = p.nt * (p.nt + 1) / 2 * p.U;
    const int u0 = IN_ORDER ? b : p.ubeg[b], u1 = IN_ORDER ? TU : p.ubeg[b + 1];
    if (u0 >= u1) return;
    const int nrun = IN_ORDER ? (TU - b + G - 1) / G : (u1 - 1) / p.U - u0 / p.U + 1;
    auto run_tile = [&](int r) { return IN_ORDER ? (b + r * G) / p.U : u0 / p.U + r; };
    auto run_range = [&](int r, int& ks, int& ke) {
        if (IN_ORDER) {
            const int j = (b + r * G) % p.U;
            ks = j * PH_UNIT; ke = min(ks + PH_UNIT, p.KT);
        } else {
            const int tt = run_tile(r);
            const int a = max(u0, tt * p.U) - tt * p.U, e = min(u1, (tt + 1) * p.U) - tt * p.U;
            ks = a * PH_UNIT; ke = min(e * PH_UNIT, p.KT);
        }
    };

    if (tid == 0) {
        for (int s = 0; s < TMA_STAGES; ++s) {
            mbar_init(bars + 8 * s, 1);
            mbar_init(bars + 8 * (TMA_STAGES + s), GEMM_THREADS / 32);   // every warp releases every stage
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();

    // producer cursor (thread 0 only): next slab to issue, across tile boundaries
    int pr = 0, pk = 0, pke = 0, issued = 0;
    run_range(pr, pk, pke);
    auto issue_next = [&]() {
        if (pr >= nrun) return;
        const int st = issued % TMA_STAGES;
        const uint32_t base = smem0 + st * TMA_STAGE_BYTES, full = bars + 8 * st;
        int bi, bj;
        ph_tile(run_tile(pr), p.nt, bi, bj);
        const bool dg = bi == bj;
        if (issued >= TMA_STAGES) mbar_wait(bars + 8 * (TMA_STAGES + st), ((issued / TMA_STAGES) + 1) & 1);
        mbar_arrive_expect_tx(full, (dg ? 1u : 2u) * BM * BK * 8 + BK * 8);
        tma_load_2d(base, &tmH, pk * BK, bi * BM, full);
        if (!dg) tma_load_2d(base + BM * BK * 8, &tmH, pk * BK, bj * BN, full);
        tma_load_1d(base + 2 * BM * BK * 8, &tmX, pk * BK, full);
        ++issued;
        if (++pk >= pke && ++pr < nrun) run_range(pr, pk, pke);
    };
    if (tid == 0)
        for (int s = 0; s < TMA_PREFETCH; ++s) issue_next();

    const int pg = 2 * (g & 3) + (g >> 2);
    int gs = 0;
    for (int r = 0; r < nrun; ++r) {
        const int tt = run_tile(r);
        int bi, bj, ks, ke;
        ph_tile(tt, p.nt, bi, bj);
        run_range(r, ks, ke);
        const bool diag = bi == bj;
        int wm = warp >> 2, wn = warp & 3;
        if (diag) { wm = kDiagWm[warp]; wn = kDiagWn[warp]; }
        const bool active = wm >= 0;
        const bool diag_warp = diag && active && (wm == wn);
        const int ra = (active ? wm : 0) * 32 + pg, rb = (active ? wn : 0) * 32 + pg;
        const uint32_t offA = ra * 128 + ((((t >> 1) ^ pg)) << 4) + (t & 1) * 8;
        const uint32_t offB = rb * 128 + ((((t >> 1) ^ pg)) << 4) + (t & 1) * 8 + (diag ? 0 : BM * BK * 8);
        double acc[MI][NI][2];
#pragma unroll
        for (int i = 0; i < MI; ++i)
#pragma unroll
            for (int j = 0; j < NI; ++j) acc[i][j][0] = acc[i][j][1] = 0.0;

        // the six idle warps of a diagonal tile do not poll: warp 0 (always active) releases the stage for them
        if (!active) gs += ke - ks;
        for (int k = ks; active && k < ke; ++k, ++gs) {
            if (tid == 0) issue_next();
            const int st = gs % TMA_STAGES;
            const uint32_t base = smem0 + st * TMA_STAGE_BYTES;
            mbar_wait(bars + 8 * st, (gs / TMA_STAGES) & 1);
            {
                const uint32_t xs = base + 2 * BM * BK * 8 + t * 8;
                if (diag_warp) {
#pragma unroll
                    for (int kk = 0; kk < BK / 4; ++kk) {
                        const double xv = lds_f64(xs + kk * 32);
                        double a[MI], bq[NI];
#pragma unroll
                        for (int i = 0; i < MI; ++i) a[i] = lds_f64(base + ((offA ^ (kk << 5)) + i * 8 * 128));
#pragma unroll
                        for (int j = 0; j < NI; ++j) bq[j] = lds_f64(base + ((offB ^ (kk << 5)) + j * 8 * 128)) * xv;
#pragma unroll
                        for (int i = 0; i < MI; ++i)
#pragma unroll
                            for (int j = 0; j < NI; ++j)
                                if (i >= j) dmma884(acc[i][j][0], acc[i][j][1], a[i], bq[j]);
                    }
                } else {
#pragma unroll
                    for (int kk = 0; kk < BK / 4; ++kk) {
                        const double xv = lds_f64(xs + kk * 32);
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
            }
            __syncwarp();
            if (lane == 0) mbar_arrive_relaxed_n(bars + 8 * (TMA_STAGES + st), (diag && warp == 0) ? 7u : 1u);
        }

        // end of this CTA's run on tile tt: partial out, ticket, the last CTA sums the partials in CTA order
        const int slot = IN_ORDER ? tt * p.U + (b + r * G) % p.U : p.slot0[tt] + b - p.first_cta[tt];
        double* P = p.P + (size_t)slot * BM * BN;
        if (active) {
#pragma unroll
            for (int i = 0; i < MI; ++i) {
                const int r = wm * 32 + 8 * i + pg;
#pragma unroll
                for (int j = 0; j < NI; ++j)
#pragma unroll
                    for (int e = 0; e < 2; ++e) {
                        const int nn = 2 * t + e;
                        P[r * BN + wn * 32 + 8 * j + 2 * (nn & 3) + (nn >> 2)] = acc[i][j][e];
                    }
            }
        }
        __threadfence();
        __syncthreads();
        if (tid == 0) sh_last = atomicAdd(&p.ticket[tt], 1u) == (unsigned)(p.nruns[tt] - 1);
        __syncthreads();
        if (sh_last) {
            if (tid == 0) p.stamps[2 * G + p.nt + tt] = gtimer();
            __threadfence();
            const double* P0 = p.P + (size_t)p.slot0[tt] * BM * BN;
            const int nr = p.nruns[tt];
            for (int e = tid; e < BM * BN; e += GEMM_THREADS) {
                const int r = e / BN, c = e % BN, row = bi * BM + r, col = bj * BN + c;
                if (row >= p.m || col >= p.m || (diag && c > r)) continue;
                double s = 0.0;
                for (int q = 0; q < nr; ++q) s += __ldcg(P0 + (size_t)q * BM * BN + e);
                p.M[(size_t)row * p.m + col] = s;
                p.M[(size_t)col * p.m + row] = s;
            }
            __threadfence();
            __syncthreads();
            if (tid == 0 && atomicAdd(&p.colcnt[bj], 1u) == (unsigned)(p.nt - bj - 1)) p.stamps[2 * G + bj] = gtimer();
        }
    }
    if (tid == 0) p.stamps[G + b] = gtimer();
}

#define CK(x) do { cudaError_t e_ = (x); if (e_ != cudaSuccess) { fprintf(stderr, "%s:%d %s\n", __FILE__, __LINE__, cudaGetErrorString(e_)); return 1; } } while (0)

int main(int argc, char** argv) {
    const int m = argc > 1 ? atoi(argv[1]) : 500;
    const int64_t n = argc > 2 ? atoll(argv[2]) : 50000;
    if (m > 512 || n % 2) { fprintf(stderr, "m <= 512 and even n only\n"); return 1; }
    int sms = 0;
    CK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, 0));
    std::vector<double> hH((size_t)m * n), hx(n);
    uint64_t st = 12345;
    auto rnd = [&]() { st = st * 6364136223846793005ULL + 1442695040888963407ULL; return (double)(st >> 11) * 0x1.0p-53; };
    for (auto& v : hH) v = rnd() - 0.5;
    for (auto& v : hx) v = rnd() / n;
    double *H, *x, *Mref, *Mph;
    CK(cudaMalloc(&H, hH.size() * 8)); CK(cudaMalloc(&x, n * 8));
    CK(cudaMalloc(&Mref, (size_t)m * m * 8)); CK(cudaMalloc(&Mph, (size_t)m * m * 8));
    CK(cudaMemcpy(H, hH.data(), hH.size() * 8, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(x, hx.data(), n * 8, cudaMemcpyHostToDevice));
    Ctx c{};
    c.device = 0; c.sm_count = sms;
    CK(cudaMalloc(&c.d_status, 256)); CK(cudaMemset(c.d_status, 0, 256));
    void* ws;
    CK(cudaMalloc(&ws, make_plan(m, n, sms).total));
    cudaStream_t s;
    CK(cudaStreamCreate(&s));
    cudaEvent_t e0, e1;
    CK(cudaEventCreate(&e0)); CK(cudaEventCreate(&e1));
    const int reps = 50;
    auto time_it = [&](auto&& f) {
        for (int i = 0; i < 3; ++i) f();
        cudaEventRecord(e0, s);
        for (int i = 0; i < reps; ++i) f();
        cudaEventRecord(e1, s);
        cudaEventSynchronize(e1);
        float ms = 0; cudaEventElapsedTime(&ms, e0, e1);
        return 1e3 * ms / reps;
    };
    printf("m %d n %lld, %d SMs; mean over %d launches, H = %.0f MB (> L2)\n", m, (long long)n, sms, reps, m * n * 8e-6);
    for (int v : {sms, sms - 8, sms - 16}) {
        c.sm_count = v;
        DoptPlan pl = make_plan(m, n, v);
        double us_s = time_it([&]() { syrk_partials(&c, s, H, m, n, n, x, ws); });
        double us_g = time_it([&]() { accbpg_dopt_gram(&c, s, H, m, n, n, x, ws, Mref); });
        printf("one-wave SYRK, plan for %3d SMs: grid %3d  syrk %6.1f us  syrk+reduce %6.1f us\n", v,
               pl.n_off * pl.s_off + pl.nt * pl.s_diag, us_s, us_g);
    }
    c.sm_count = sms;
    accbpg_dopt_gram(&c, s, H, m, n, n, x, ws, Mref);
    CK(cudaStreamSynchronize(s));
    std::vector<double> ref((size_t)m * m), got((size_t)m * m);
    CK(cudaMemcpy(ref.data(), Mref, ref.size() * 8, cudaMemcpyDeviceToHost));

    // phased plan
    const int nt = (m + BM - 1) / BM, T = nt * (nt + 1) / 2, KT = (int)((n + BK - 1) / BK), U = (KT + PH_UNIT - 1) / PH_UNIT;
    CK(cudaFuncSetAttribute(syrk_phased_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, TMA_SMEM));
    CK(cudaFuncSetAttribute(syrk_phased_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, TMA_SMEM));
    for (int in_order : {0, 1})
    for (int G : {sms, sms - 8, sms - 16}) {
        std::vector<double> cost((size_t)T * U);
        double total = 0;
        for (int tt = 0; tt < T; ++tt) {
            int bi, bj;
            ph_tile(tt, nt, bi, bj);
            for (int j = 0; j < U; ++j) {
                const int sl = std::min(PH_UNIT, KT - j * PH_UNIT);
                cost[(size_t)tt * U + j] = (bi == bj ? 0.5625 : 1.0) * sl + (j == 0 ? 2.0 : 0.0);
                total += cost[(size_t)tt * U + j];
            }
        }
        std::vector<int> ubeg(G + 1, T * U);
        ubeg[0] = 0;
        {
            double acc = 0; int b = 1;
            for (int u = 0; u < T * U && b < G; ++u) {
                acc += cost[u];
                if (acc >= total * b / G) ubeg[b++] = u + 1;
            }
        }
        std::vector<int> first(T, -1), nr(T, 0), slot0(T, 0);
        for (int b = 0; b < G; ++b)
            for (int tt = ubeg[b] / U; ubeg[b] < ubeg[b + 1] && tt <= (ubeg[b + 1] - 1) / U; ++tt) {
                if (first[tt] < 0) first[tt] = b;
                ++nr[tt];
            }
        if (in_order) std::fill(nr.begin(), nr.end(), U);
        int slots = 0;
        for (int tt = 0; tt < T; ++tt) { slot0[tt] = slots; slots += nr[tt]; }
        int *d_ubeg, *d_first, *d_nr, *d_slot0;
        unsigned int *ticket, *colcnt;
        unsigned long long* stamps;
        double* P;
        CK(cudaMalloc(&d_ubeg, (G + 1) * 4)); CK(cudaMalloc(&d_first, T * 4)); CK(cudaMalloc(&d_nr, T * 4));
        CK(cudaMalloc(&d_slot0, T * 4)); CK(cudaMalloc(&ticket, (T + nt) * 4)); colcnt = ticket + T;
        CK(cudaMalloc(&stamps, (2 * G + nt + T) * 8)); CK(cudaMalloc(&P, (size_t)slots * BM * BN * 8));
        CK(cudaMemcpy(d_ubeg, ubeg.data(), (G + 1) * 4, cudaMemcpyHostToDevice));
        CK(cudaMemcpy(d_first, first.data(), T * 4, cudaMemcpyHostToDevice));
        CK(cudaMemcpy(d_nr, nr.data(), T * 4, cudaMemcpyHostToDevice));
        CK(cudaMemcpy(d_slot0, slot0.data(), T * 4, cudaMemcpyHostToDevice));
        PhParams p{P, Mph, m, nt, U, KT, d_ubeg, d_slot0, d_first, d_nr, ticket, colcnt, stamps};
        CUtensorMap tmH, tmX;
        cuuint64_t dimH[2] = {(cuuint64_t)n, (cuuint64_t)m}, strH[1] = {(cuuint64_t)n * 8}, dimX[1] = {(cuuint64_t)n};
        cuuint32_t boxH[2] = {BK, BM}, boxX[1] = {BK}, one[2] = {1, 1};
        if (encode_tiled_fn()(&tmH, CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 2, H, dimH, strH, boxH, one, CU_TENSOR_MAP_INTERLEAVE_NONE,
                              CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) ||
            encode_tiled_fn()(&tmX, CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 1, x, dimX, strH, boxX, one, CU_TENSOR_MAP_INTERLEAVE_NONE,
                              CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE)) {
            fprintf(stderr, "tensor map encode failed\n");
            return 1;
        }
        auto launch = [&]() {
            cudaMemsetAsync(ticket, 0, (T + nt) * 4, s);
            if (in_order) syrk_phased_kernel<true><<<G, GEMM_THREADS, TMA_SMEM, s>>>(p, tmH, tmX);
            else          syrk_phased_kernel<false><<<G, GEMM_THREADS, TMA_SMEM, s>>>(p, tmH, tmX);
        };
        double us = time_it(launch);
        CK(cudaGetLastError());
        CK(cudaStreamSynchronize(s));
        CK(cudaMemcpy(got.data(), Mph, got.size() * 8, cudaMemcpyDeviceToHost));
        double emax = 0, amax = 0;
        for (size_t i = 0; i < got.size(); ++i) { emax = std::max(emax, std::fabs(got[i] - ref[i])); amax = std::max(amax, std::fabs(ref[i])); }
        std::vector<unsigned long long> hs(2 * G + nt + T);
        CK(cudaMemcpy(hs.data(), stamps, hs.size() * 8, cudaMemcpyDeviceToHost));
        unsigned long long t0 = ~0ULL, t1 = 0;
        for (int b = 0; b < G; ++b) { t0 = std::min(t0, hs[b]); t1 = std::max(t1, hs[G + b]); }
        int maxruns = *std::max_element(nr.begin(), nr.end());
        printf("phased SYRK %s grid %3d: %6.1f us (memset + kernel)  span %6.1f us  M rel err %.1e  partials %d (max %d per "
               "tile)\n    tile column: last partial in / final at", in_order ? "in-order" : "contig  ", G, us, (t1 - t0) * 1e-3,
               emax / amax, slots, maxruns);
        for (int cc = 0, tt = 0; cc < nt; ++cc) {
            unsigned long long last_in = 0;
            for (int q = 0; q < nt - cc; ++q, ++tt) last_in = std::max(last_in, hs[2 * G + nt + tt]);
            printf("  %5.1f / %5.1f", (last_in - t0) * 1e-3, (hs[2 * G + cc] - t0) * 1e-3);
        }
        printf(" us\n");
        cudaFree(d_ubeg); cudaFree(d_first); cudaFree(d_nr); cudaFree(d_slot0); cudaFree(ticket); cudaFree(stamps); cudaFree(P);
    }
    uint32_t status = 0;
    CK(cudaMemcpy(&status, c.d_status, 4, cudaMemcpyDeviceToHost));
    printf("status word %u\n", status);
    return 0;
}
