// Tooling: one slab of the Gaussian step's constant-weight SYRK  C += alpha K K^T  (lower tiles) as the exact int8 Gram product
// (t-svgp_b200/csrc/int8_gram.cu) against the FP64 DMMA SYRK, and both against the exact integer product on the host for sampled
// entries.  Random K in [0, v] with exact 0 and v entries; per-kernel times with CUDA events.  The products are timed twice, each
// behind the residue kernel: (a) as the launcher runs them, (b) with pstride = 0, so that all 16 moduli read plane 0 (L2-resident
// operands; the tiles it writes are not checked).  (a) - (b) is what reading the 16 freshly written planes costs.
// Build: make -C tools i8_syrk_bench ; run: tools/i8_syrk_bench [Mp=2048] [ncols=16384]
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>
#include <cuda_runtime.h>
#include "../t-svgp_b200/csrc/gemm.cuh"
#include "../t-svgp_b200/csrc/int8_gram.cu"
namespace tsvgp { thread_local long g_launches = 0; int g_debug_sync = 0; int g_pdl = 1; thread_local int g_pdl_suspended = 0; }
using namespace tsvgp;
#define CK(x) do { cudaError_t e = (x); if (e != cudaSuccess) { printf("CUDA error %s at %s:%d\n", cudaGetErrorString(e), __FILE__, __LINE__); exit(1);} } while (0)

__global__ void fill(double* K, long n, long ld, int ncols, double v, unsigned seed) {
    const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const long r = i / ld, c = i % ld;
    unsigned x = seed ^ (unsigned)(i * 2654435761u); x ^= x >> 13; x *= 0x5bd1e995; x ^= x >> 15; x *= 0x27d4eb2d; x ^= x >> 16;
    double u = (x & 0xffffff) / 16777216.0;
    if ((x >> 24) == 0) u = 0.0;
    if ((x >> 24) == 1) u = 1.0;
    K[i] = c < ncols ? v * u * u : 0.0;   // skewed towards small values, like a covariance slab
    (void)r;
}

static float ev_ms(cudaEvent_t a, cudaEvent_t b) { float ms; cudaEventElapsedTime(&ms, a, b); return ms; }

int main(int argc, char** argv) {
    const int Mp = argc > 1 ? atoi(argv[1]) : 2048, ncols = argc > 2 ? atoi(argv[2]) : 16384;
    const long nc = ncols;
    const double v = 1.3, alpha = -5.0;
    cudaDeviceProp prop; CK(cudaGetDeviceProperties(&prop, 0));
    printf("device %s sms %d, Mp %d ncols %d\n", prop.name, prop.multiProcessorCount, Mp, ncols);
    CK(gemm_init() ? cudaErrorUnknown : cudaSuccess);
    double *K, *C8, *C64;
    int8_t* planes; uint8_t* tiles;
    CK(cudaMalloc(&K, sizeof(double) * Mp * nc));
    CK(cudaMalloc(&C8, sizeof(double) * Mp * Mp)); CK(cudaMalloc(&C64, sizeof(double) * Mp * Mp));
    CK(cudaMalloc(&planes, i8_plane_bytes(Mp, nc))); CK(cudaMalloc(&tiles, i8_tile_bytes(Mp)));
    fill<<<(unsigned)((Mp * nc + 255) / 256), 256>>>(K, (long)Mp * nc, nc, ncols, v, 7u);
    CK(cudaMemset(C8, 0, sizeof(double) * Mp * Mp)); CK(cudaMemset(C64, 0, sizeof(double) * Mp * Mp));
    CK((cudaError_t)i8_planes_init(planes, Mp, nc, 0));
    CK((cudaError_t)i8_syrk_launch(K, nc, Mp, ncols, v, alpha, planes, nc, tiles, C8, Mp, 0));
    GemmP p;
    p.A = K; p.lda = nc; p.a_kc = 1; p.B = K; p.ldb = nc; p.b_kc = 1;
    p.C = C64; p.ldc = Mp; p.m = p.n = Mp; p.k = ncols; p.beta = 1.0; p.lower_out = 1; p.alpha = alpha;
    CK((cudaError_t)gemm_launch(p, 0));
    CK(cudaDeviceSynchronize());

    // exact reference on sampled lower-tile entries
    std::vector<double> hK((size_t)Mp * nc), h8((size_t)Mp * Mp), h64((size_t)Mp * Mp);
    CK(cudaMemcpy(hK.data(), K, sizeof(double) * hK.size(), cudaMemcpyDeviceToHost));
    CK(cudaMemcpy(h8.data(), C8, sizeof(double) * h8.size(), cudaMemcpyDeviceToHost));
    CK(cudaMemcpy(h64.data(), C64, sizeof(double) * h64.size(), cudaMemcpyDeviceToHost));
    const double scale = 4503599627370496.0 / v;
    std::vector<uint64_t> A((size_t)Mp * nc);
    for (size_t i = 0; i < A.size(); ++i) A[i] = (uint64_t)std::rint(hK[i] * scale);
    long bad = 0, ns = 0;
    double max8 = 0, max64 = 0, maxref = 0, d64_ref = 0;
    srand(11);
    for (int s = 0; s < 4000; ++s) {
        int i = rand() % Mp, j = rand() % Mp;
        if (j / 128 > i / 128) std::swap(i, j);
        if (s < 8) { i = (s * 131) % Mp; j = i - (i % 128); }   // diagonal tiles included
        unsigned __int128 x = 0;
        for (long k = 0; k < ncols; ++k) x += (unsigned __int128)A[(size_t)i * nc + k] * A[(size_t)j * nc + k];
        const double want = (double)x * (alpha * v * v * 0x1p-104);
        const double got = h8[(size_t)i * Mp + j], f64 = h64[(size_t)i * Mp + j];
        if (memcmp(&want, &got, 8) && bad++ < 5) printf("  mismatch (%d,%d): int8 %.17g exact %.17g\n", i, j, got, want);
        ++ns;
        max8 = fmax(max8, fabs(got - want)); maxref = fmax(maxref, fabs(want));
        if ((j % 128) <= (i % 128) || i / 128 != j / 128) { max64 = fmax(max64, fabs(f64 - want)); d64_ref = fmax(d64_ref, fabs(f64)); }
    }
    printf("int8 Gram vs exact integer product rounded once: %ld of %ld sampled entries differ (max |diff| / max|C| = %.2e)\n", bad, ns,
           max8 / maxref);
    printf("FP64 DMMA SYRK vs the same exact product: max |diff| / max|C| = %.2e  (grid rounding + FP64 summation)\n", max64 / maxref);

    // timing: the three kernels separately, then the FP64 SYRK
    const int nt = Mp / 128, nrb = (nt + 1) & ~1, nkb = ncols / 128, nblk = blocks_per_modulus(nt);
    const size_t pstride = (size_t)(nc / 128) * nrb * KB_BYTES, tstride = (size_t)nt * (nt + 1) / 2 * KB_BYTES;
    int grid = 0;
    CK((cudaError_t)i8_gram_grid(nrb, grid));
    cudaEvent_t ev[7];
    for (auto& x : ev) cudaEventCreate(&x);
    const int reps = 10;
    float t[5] = {0, 0, 0, 0, 0};
    for (int r = 0; r < reps + 1; ++r) {
        cudaEventRecord(ev[0]);
        i8_residue_kernel<<<dim3(nkb, nt), 256>>>(K, nc, scale, planes, pstride, nrb);
        cudaEventRecord(ev[1]);
        i8_gram_kernel<<<grid, GEMM_THREADS, GEMM_SMEM>>>(planes, pstride, nrb, nkb, nblk, tiles, tstride);
        cudaEventRecord(ev[2]);
        i8_crt_kernel<<<(unsigned)(tstride / KB_BYTES) * 16, 256>>>(tiles, tstride, C8, Mp, alpha * v * v * 0x1p-104);
        cudaEventRecord(ev[3]);
        gemm_launch(p, 0);
        cudaEventRecord(ev[4]);
        i8_residue_kernel<<<dim3(nkb, nt), 256>>>(K, nc, scale, planes, pstride, nrb);
        cudaEventRecord(ev[5]);
        i8_gram_kernel<<<grid, GEMM_THREADS, GEMM_SMEM>>>(planes, 0, nrb, nkb, nblk, tiles, tstride);
        cudaEventRecord(ev[6]);
        CK(cudaEventSynchronize(ev[6]));
        if (r) {
            for (int k = 0; k < 4; ++k) t[k] += ev_ms(ev[k], ev[k + 1]) / reps;
            t[4] += ev_ms(ev[5], ev[6]) / reps;
        }
    }
    CK(cudaGetLastError());
    const double ops8 = 16.0 * nblk * 2.0 * 128 * 256 * ncols, flops64 = (double)nt * (nt + 1) / 2 * 2.0 * 128 * 128 * ncols;
    printf("i8_residue_kernel  %8.3f ms  (%.2f TB/s: slab read + planes written)\n", t[0], (8.0 * Mp * ncols + 16.0 * Mp * ncols) / t[0] * 1e-9);
    printf("i8_gram_kernel     %8.3f ms  %.1f TOP/s int8 (%d blocks of 128x256x%d, %d CTAs in pairs)  (a) as launched\n", t[1],
           ops8 / t[1] * 1e-9, 16 * nblk, ncols, grid);
    printf("i8_gram_kernel     %8.3f ms  %.1f TOP/s int8  (b) pstride = 0: every modulus reads plane 0\n", t[4], ops8 / t[4] * 1e-9);
    printf("i8_crt_kernel      %8.3f ms\n", t[2]);
    printf("int8 total         %8.3f ms\n", t[0] + t[1] + t[2]);
    printf("FP64 DMMA SYRK     %8.3f ms  %.1f TFLOP/s\n", t[3], flops64 / t[3] * 1e-9);
    return bad != 0;
}
