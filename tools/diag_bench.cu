// Tooling: times the 128x128 diagonal-block kernel (Cholesky + inverse) and the blocked chol_lower / trtri_lower.
#include <cstdio>
#include <cstdlib>
#include <vector>
#include <cmath>
#include <cuda_runtime.h>
#include "../t-svgp_b200/csrc/kernels.cuh"
#include "../t-svgp_b200/csrc/dense.cuh"
#include "../t-svgp_b200/csrc/gemm.cuh"
#include "../t-svgp_b200/csrc/common.cuh"
namespace tsvgp { thread_local long g_launches = 0; int g_debug_sync = 0; int g_pdl = 1; thread_local int g_pdl_suspended = 0; }
using namespace tsvgp;
#define CK(x) do { cudaError_t e = (x); if (e != cudaSuccess) { printf("CUDA error %s at %s:%d\n", cudaGetErrorString(e), __FILE__, __LINE__); exit(1);} } while (0)
int main(int argc, char** argv) {
    int n = argc > 1 ? atoi(argv[1]) : 2048;
    gemm_init(); diag_init(); dense_init();
    std::vector<double> A((size_t)n * n);
    for (int i = 0; i < n; ++i) for (int j = 0; j < n; ++j) A[(size_t)i * n + j] = exp(-0.5 * (i - j) * (i - j) / 9.0) + (i == j ? 0.5 : 0.0);
    double *dA, *dW, *dinv, *dLinv, *tmp; int* info;
    CK(cudaMalloc(&dA, sizeof(double) * n * n)); CK(cudaMalloc(&dW, sizeof(double) * n * n)); CK(cudaMalloc(&dLinv, sizeof(double) * n * n));
    CK(cudaMalloc(&tmp, sizeof(double) * n * n)); CK(cudaMalloc(&dinv, sizeof(double) * (n / 128) * 128 * 128)); CK(cudaMalloc(&info, 16)); CK(cudaMemset(info, 0, 16)); CK(cudaMemset(dinv, 0, sizeof(double) * (n / 128) * 128 * 128));
    CK(cudaMemcpy(dA, A.data(), sizeof(double) * n * n, cudaMemcpyHostToDevice));
    double* ws; const size_t ws_doubles = ((size_t)4 << 20) - 2048; CK(cudaMalloc(&ws, sizeof(double) * ws_doubles));   // split-K workspace (gemm_launch_auto), the library's size
    cudaEvent_t e0, e1; cudaEventCreate(&e0); cudaEventCreate(&e1); float ms;
    for (int rep = 0; rep < 3; ++rep) {
        CK(cudaMemcpy(dW, dA, sizeof(double) * n * n, cudaMemcpyDeviceToDevice));
        cudaEventRecord(e0); diag_potrf_inv_launch(dW, n, dinv, 0, info, 0); cudaEventRecord(e1); CK(cudaEventSynchronize(e1));
        cudaEventElapsedTime(&ms, e0, e1); printf("diag_potrf_inv (1 block): %.1f us\n", ms * 1e3);
    }
    {   // the block against a host Cholesky + inverse
        std::vector<double> Lb(128 * 128), Xb(128 * 128), Lh(128 * 128, 0.0);
        CK(cudaMemcpy2D(Lb.data(), 128 * 8, dW, (size_t)n * 8, 128 * 8, 128, cudaMemcpyDeviceToHost));
        CK(cudaMemcpy(Xb.data(), dinv, sizeof(double) * 128 * 128, cudaMemcpyDeviceToHost));
        for (int j = 0; j < 128; ++j) {
            double d = A[(size_t)j * n + j];
            for (int k = 0; k < j; ++k) d -= Lh[j * 128 + k] * Lh[j * 128 + k];
            Lh[j * 128 + j] = sqrt(d);
            for (int i = j + 1; i < 128; ++i) {
                double v = A[(size_t)i * n + j];
                for (int k = 0; k < j; ++k) v -= Lh[i * 128 + k] * Lh[j * 128 + k];
                Lh[i * 128 + j] = v / Lh[j * 128 + j];
            }
        }
        double eL = 0, eX = 0, eU = 0;
        for (int i = 0; i < 128; ++i)
            for (int j = 0; j < 128; ++j) {
                if (j <= i) eL = fmax(eL, fabs(Lb[i * 128 + j] - Lh[i * 128 + j]));   // the upper triangle of A is the caller's to zero
                double u = 0;
                for (int k = 0; k < 128; ++k) u += Xb[i * 128 + k] * Lh[k * 128 + j];
                eX = fmax(eX, fabs(u - (i == j ? 1.0 : 0.0)));
                if (j > i) eU = fmax(eU, fabs(Xb[i * 128 + j]));
            }
        printf("  max |L - L_host| %.2e   max |X L_host - I| %.2e   max |upper of X| %.2e\n", eL, eX, eU);
    }
    {   // failure reporting: a non-positive pivot at row 70 of block 3
        std::vector<double> Bad(128 * 128, 0.0);
        for (int i = 0; i < 128; ++i) Bad[i * 128 + i] = i == 70 ? -1.0 : 2.0;
        CK(cudaMemcpy2D(dW, (size_t)n * 8, Bad.data(), 128 * 8, 128 * 8, 128, cudaMemcpyHostToDevice));
        CK(cudaMemset(info, 0, 16));
        diag_potrf_inv_launch(dW, n, dinv, 3, info, 0);
        int h; CK(cudaMemcpy(&h, info, 4, cudaMemcpyDeviceToHost));
        printf("  failing pivot reported %d (expected %d)\n", h, 3 * 128 + 71);
        CK(cudaMemset(info, 0, 16));
    }
    for (int rep = 0; rep < 3; ++rep) {
        CK(cudaMemcpy(dW, dA, sizeof(double) * n * n, cudaMemcpyDeviceToDevice));
        double* w = rep == 0 ? nullptr : ws;   // first repetition without split-K, for comparison
        cudaEventRecord(e0); chol_lower(dW, n, n, dinv, info, 0, w, ws_doubles); cudaEventRecord(e1); CK(cudaEventSynchronize(e1));
        cudaEventElapsedTime(&ms, e0, e1); printf("chol_lower n=%d (%s): %.3f ms  (%.2f TFLOP/s of n^3/3)\n", n, w ? "auto split-K" : "no split", ms, (double)n * n * n / 3 / ms / 1e9);
        cudaEventRecord(e0); trtri_lower(dW, n, n, dinv, dLinv, tmp, 0, w, ws_doubles); cudaEventRecord(e1); CK(cudaEventSynchronize(e1));
        cudaEventElapsedTime(&ms, e0, e1); printf("trtri_lower n=%d (%s): %.3f ms\n", n, w ? "auto split-K" : "no split", ms);
    }
    {   // look-ahead over two streams (dense.cuh::CholAux) against the single-stream schedule, on explicit non-blocking streams
        cudaStream_t s1; CholAux aux;
        CK(cudaStreamCreateWithFlags(&s1, cudaStreamNonBlocking)); CK(cudaStreamCreateWithFlags(&aux.s2, cudaStreamNonBlocking));
        CK(cudaEventCreateWithFlags(&aux.e, cudaEventDisableTiming)); CK(cudaEventCreateWithFlags(&aux.f, cudaEventDisableTiming));
        for (int rep = 0; rep < 6; ++rep) {
            const bool la = rep >= 3;
            CK(cudaMemcpyAsync(dW, dA, sizeof(double) * n * n, cudaMemcpyDeviceToDevice, s1));
            cudaEventRecord(e0, s1); chol_lower(dW, n, n, dinv, info, s1, ws, ws_doubles, la ? &aux : nullptr); cudaEventRecord(e1, s1); CK(cudaEventSynchronize(e1));
            cudaEventElapsedTime(&ms, e0, e1); printf("chol_lower n=%d (%s): %.3f ms\n", n, la ? "look-ahead, 2 streams" : "single stream", ms);
        }
        CK(cudaStreamSynchronize(s1));
    }
    int h; CK(cudaMemcpy(&h, info, 4, cudaMemcpyDeviceToHost)); printf("info %d\n", h);
    std::vector<double> L((size_t)n * n), Li((size_t)n * n);
    CK(cudaMemcpy(L.data(), dW, sizeof(double) * n * n, cudaMemcpyDeviceToHost)); CK(cudaMemcpy(Li.data(), dLinv, sizeof(double) * n * n, cudaMemcpyDeviceToHost));
    double e1m = 0, e2m = 0;
    for (int t = 0; t < 2000; ++t) {
        int i = rand() % n, j = rand() % (i + 1); double s = 0, u = 0;
        for (int k = 0; k <= j; ++k) s += L[(size_t)i * n + k] * L[(size_t)j * n + k];
        for (int k = j; k <= i; ++k) u += Li[(size_t)i * n + k] * L[(size_t)k * n + j];
        e1m = fmax(e1m, fabs(s - A[(size_t)i * n + j])); e2m = fmax(e2m, fabs(u - (i == j ? 1.0 : 0.0)));
    }
    printf("max |LL^T - A| %.2e   max |Linv L - I| %.2e\n", e1m, e2m);
    return 0;
}
