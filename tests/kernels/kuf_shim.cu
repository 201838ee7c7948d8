// Test shim for the covariance slab kernel (kuf_kernel in t-svgp_b200/csrc/kernels.cu): kuf_launch as an extern "C" entry
// point, so the tests can compare the slab and its dk/dr2 companion with NumPy on chosen inputs.
// Built by tests/test_gpu_matern_family.py:
//   nvcc -O3 -std=c++17 -gencode arch=compute_100a,code=sm_100a -Xcompiler -fPIC -shared -o libkufshim.so kuf_shim.cu
// Pointers are device pointers; the entry point returns the CUDA status (cudaSuccess = 0), or -1 for an unknown kind.
#include "../../t-svgp_b200/csrc/kernels.cu"
namespace tsvgp { thread_local long g_launches = 0; int g_debug_sync = 0; int g_pdl = 1; thread_local int g_pdl_suspended = 0; }

extern "C" int kuf_launch(int kind, double variance, const double* XsT, long ldx, const double* x2, long n0, long n_valid, int ncols,
                          const double* Zs, const double* z2, int M, int Mp, int D, const double* alpha, double* K, long ldk,
                          double* mu_part, long ldmu, int pad_identity, cudaStream_t s, double* Kp) {
    return tsvgp::kuf_launch(kind, variance, XsT, ldx, x2, n0, n_valid, ncols, Zs, z2, M, Mp, D, alpha, K, ldk, mu_part, ldmu,
                             pad_identity, s, Kp);
}
