// Test shim for the int8 Gram product (t-svgp_b200/csrc/int8_gram.cu): the launcher and its three stages as extern "C" entry
// points, so the tests can run each stage on its own and compare it with the exact references of tests/int8_gram_ref.py.
// Built by tests/test_gpu_int8_gram_kernels.py:
//   nvcc -O3 -std=c++17 -gencode arch=compute_100a,code=sm_100a -Xcompiler -fPIC -shared -o libi8shim.so int8_gram_shim.cu
// Pointers are device pointers; every entry point returns the CUDA status (cudaSuccess = 0).
#include "../../t-svgp_b200/csrc/int8_gram.cu"
namespace tsvgp { thread_local long g_launches = 0; int g_debug_sync = 0; int g_pdl = 1; thread_local int g_pdl_suspended = 0; }

extern "C" {

int i8_syrk_launch(const double* K, long ldk, int Mp, int ncols, double var, double alpha, int8_t* planes, long nc_alloc,
                   uint8_t* tiles, double* C, long ldc, cudaStream_t s) {
    return tsvgp::i8_syrk_launch(K, ldk, Mp, ncols, var, alpha, planes, nc_alloc, tiles, C, ldc, s);
}
int i8_planes_init(int8_t* planes, int Mp, long nc_alloc, cudaStream_t s) { return tsvgp::i8_planes_init(planes, Mp, nc_alloc, s); }
size_t i8_plane_bytes(int Mp, long nc) { return tsvgp::i8_plane_bytes(Mp, nc); }
size_t i8_tile_bytes(int Mp) { return tsvgp::i8_tile_bytes(Mp); }

// the three stages with the arguments i8_syrk_launch derives (nt = Mp / 128, nrb = plane row blocks, nkb = ncols / 128,
// nblk = lower 128 x 256 blocks of one modulus, pstride / tstride = bytes of one modulus's planes / tiles)
int i8_residue_launch(const double* K, long ldk, double scale, int8_t* planes, size_t pstride, int nrb, int nkb, int nt, cudaStream_t s) {
    tsvgp::i8::i8_residue_kernel<<<dim3(nkb, nt), 256, 0, s>>>(K, ldk, scale, planes, pstride, nrb);
    return (int)cudaGetLastError();
}
int i8_gram_launch(const int8_t* planes, size_t pstride, int nrb, int nkb, int nblk, uint8_t* tiles, size_t tstride, cudaStream_t s) {
    using namespace tsvgp::i8;
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    if (cudaError_t e = cudaFuncSetAttribute(i8_gram_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, GEMM_SMEM)) return (int)e;
    const int units = tsvgp::I8_NMOD * nblk;
    i8_gram_kernel<<<units < sms ? units : sms, GEMM_THREADS, GEMM_SMEM, s>>>(planes, pstride, nrb, nkb, nblk, tiles, tstride);
    return (int)cudaGetLastError();
}
int i8_crt_launch(const uint8_t* tiles, size_t tstride, double* C, long ldc, double scale, cudaStream_t s) {
    tsvgp::i8::i8_crt_kernel<<<(unsigned)(tstride / tsvgp::i8::KB_BYTES) * 16, 256, 0, s>>>(tiles, tstride, C, ldc, scale);
    return (int)cudaGetLastError();
}

}  // extern "C"
