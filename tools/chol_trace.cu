// Phase-by-phase cycle trace of the Cholesky + inverse step kernel (CTA 0 of every launch).
//   nvcc -gencode arch=compute_100a,code=sm_100a -O3 -std=c++17 -DCHOL_TRACE -o tools/build/chol_trace tools/chol_trace.cu \
//        accbpg_and_fw_b200/csrc/build/prof.o accbpg_and_fw_b200/csrc/build/vecops.o
#include "../accbpg_and_fw_b200/csrc/chol.cu"
#include <vector>
#include <cstdlib>
using namespace accbpg;

int main(int argc, char** argv) {
    int m = argc > 1 ? atoi(argv[1]) : 500;
    int mp = (m + 127) / 128 * 128;
    std::vector<double> A((size_t)m * m), M((size_t)m * m, 0.0);
    srand(1);
    for (auto& a : A) a = rand() / (double)RAND_MAX - 0.5;
    for (int i = 0; i < m; ++i)
        for (int j = 0; j <= i; ++j) {
            double s = (i == j) ? m * 0.1 : 0.0;
            for (int k = 0; k < m; ++k) s += A[(size_t)i * m + k] * A[(size_t)j * m + k];
            M[(size_t)i * m + j] = M[(size_t)j * m + i] = s;
        }
    double *dM, *dL, *dLinv, *dW, *dY, *dacc;
    cudaMalloc(&dM, (size_t)m * m * 8); cudaMalloc(&dL, (size_t)m * m * 8); cudaMalloc(&dW, (size_t)m * m * 8);
    cudaMalloc(&dLinv, (size_t)mp * mp * 8); cudaMalloc(&dY, (size_t)mp * mp * 8); cudaMalloc(&dacc, 64);
    cudaMemcpy(dM, M.data(), (size_t)m * m * 8, cudaMemcpyHostToDevice);
    Ctx c{};
    cudaMalloc(&c.d_status, 256); cudaMemset(c.d_status, 0, 256);
    int nblk = (m + 63) / 64;
    cudaMalloc(&g_chol_trace, nblk * 16 * 8);
    cudaStream_t s; cudaStreamCreate(&s);
    cudaEvent_t e0, e1; cudaEventCreate(&e0); cudaEventCreate(&e1);
    for (int want = 1; want >= 0; --want) {
        for (int rep = 0; rep < 3; ++rep) {
            cudaEventRecord(e0, s);
            int rc = chol_factor_inv(&c, s, m, mp, dM, nullptr, want, dLinv, dW, dY, dacc, dacc + 1);
            cudaEventRecord(e1, s);
            cudaStreamSynchronize(s);
            float ms; cudaEventElapsedTime(&ms, e0, e1);
            printf("m %d want_inv %d rc %d  total %.1f us  (%s)\n", m, want, rc, ms * 1e3, cudaGetErrorString(cudaGetLastError()));
        }
        std::vector<long long> tr(nblk * 16);
        cudaMemcpy(tr.data(), g_chol_trace, nblk * 16 * 8, cudaMemcpyDeviceToHost);
        printf(" J | stage  fac0  inv0  prod1  fac1  inv1  prod2+wait  publish  P1  P2  store | kernel us | gap us\n");
        for (int J = 0; J < nblk; ++J) {
            long long* t = &tr[J * 16];
            printf("%2d |", J);
            for (int i = 1; i <= 11; ++i) printf(" %6lld", (t[i] && t[i - 1]) ? t[i] - t[i - 1] : 0LL);
            printf(" | %7.2f | %6.2f\n", (t[15] - t[14]) * 1e-3, J ? (t[14] - tr[(J - 1) * 16 + 15]) * 1e-3 : 0.0);
        }
    }
    // ---- data-flow chain: phase stamps of the spine CTA
    {
        long long* dtr;
        cudaMalloc(&dtr, nblk * 16 * 8);
        cudaMemset(dtr, 0, nblk * 16 * 8);
        cudaMemcpyToSymbol(g_df_trace_dev, &dtr, sizeof(dtr));
        void* aux;
        size_t ab = chol_df_aux_bytes(m);
        cudaMalloc(&aux, ab); cudaMemset(aux, 0, ab);
        cudaMemset(dLinv, 0, (size_t)mp * mp * 8);
        c.sm_count = 148;
        for (int want = 1; want >= 0; --want) {
            for (int rep = 0; rep < 3; ++rep) {
                cudaEventRecord(e0, s);
                int rc = chol_factor_inv(&c, s, m, mp, dM, nullptr, want, dLinv, dW, dY, dacc, dacc + 1, aux);
                cudaEventRecord(e1, s);
                cudaStreamSynchronize(s);
                float ms; cudaEventElapsedTime(&ms, e0, e1);
                printf("DF m %d want_inv %d rc %d  total %.1f us  (%s)\n", m, want, rc, ms * 1e3, cudaGetErrorString(cudaGetLastError()));
            }
            std::vector<long long> tr(nblk * 16);
            cudaMemcpy(tr.data(), dtr, nblk * 16 * 8, cudaMemcpyDeviceToHost);
            printf(" J | tiles  P0  D00  fac0  inv0  sync+prod1  fac1  inv1+sync  prod2  stores | step cycles\n");
            for (int J = 0; J < nblk; ++J) {
                long long* t = &tr[J * 16];
                printf("%2d |", J);
                for (int i = 1; i <= 10; ++i) printf(" %6lld", (t[i] && t[i - 1]) ? t[i] - t[i - 1] : 0LL);
                printf(" | %7lld\n", t[10] - t[0]);
            }
        }
    }
    return 0;
}
