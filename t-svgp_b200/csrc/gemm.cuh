// FP64 DMMA GEMM engine: one tiled mainloop (128x128 CTA tile, 8 warps of 64x32, BK=16, 5-stage cp.async pipeline)
// reused by the streaming statistics pass (weighted SYRK, triangular variance product) and by every dense M x M
// operation of the natural-gradient step (reference math: src/models/tsvgp.py:234-304, src/util.py:349-391).
//
//   C[m x n] = alpha * sum_k A(i,k) * [kscale(k)] * B(k,j) + beta * C          (row-major C, all dims multiples of 128)
//
// Operand storage:  a_kc = 1 : A stored [m][k] (k contiguous) ;  a_kc = 0 : A stored [k][m]
//                   b_kc = 1 : B stored [n][k]                ;  b_kc = 0 : B stored [k][n]
// Triangular structure lets a tile skip k-blocks that are identically zero (operands carry explicit zeros there):
//   a_tri = 1 : A(i,k) != 0 only for k <= i     a_tri = 2 : only for k >= i      (same for b_tri with j)
// lower_out = 1 : only tiles with tile_i >= tile_j are computed (symmetric results).
#pragma once
#include <cuda_runtime.h>

namespace tsvgp {

enum { EPI_STORE = 0, EPI_COLNORM = 1, EPI_STORE_COLNORM = 2 };   // 2: store C and also reduce its column norms

struct GemmP {
    const double* A = nullptr; long lda = 0; int a_kc = 1;
    const double* B = nullptr; long ldb = 0; int b_kc = 1;
    double* C = nullptr; long ldc = 0;
    int m = 0, n = 0, k = 0;
    double alpha = 1.0, beta = 0.0;
    int lower_out = 0;
    int a_tri = 0, b_tri = 0;
    const double* kscale = nullptr;   // optional [k] weights on the contraction index (the h_n of the weighted SYRK)
    // with kscale: optional fused mat-vec  bout[i] += sum_k A(i,k) gvec[k]  (b += Kuf g of the statistics pass), computed from the A
    // fragments the first tile column already holds in registers; the split-off k piece (C2) accumulates into bout2
    const double* gvec = nullptr; double* bout = nullptr; double* bout2 = nullptr;
    int epilogue = EPI_STORE;
    double* norm_out = nullptr; long ldn = 0;   // EPI_COLNORM: norm_out[tile_i * ldn + j] = sum_{i in tile} C(i,j)^2
    int ksplit = 1; double* part = nullptr; long part_stride = 0;   // split-K partial slabs [ksplit][m*ldc]; caller reduces
    long part_ld = 0, part_sC = 0;    // row / batch strides of the partial slabs when they are stored more compactly than C (0 = ldc / sC)
    int batch = 1; long sA = 0, sB = 0, sC = 0;
    // Two-piece k split for load balance (no atomics): CTAs with blockIdx.z == 0 contract k in [0, ksp) into C, CTAs with
    // blockIdx.z == 1 contract [ksp, k) into C2 (same layout, same beta).  The z = 0 pieces are dispatched first; with
    // ksp / k = (T / P) / ceil(T / P) for T output tiles on P SMs, greedy in-order dispatch fills every SM equally.
    int ksp = 0; double* C2 = nullptr;
    // Row-cyclic partition over ranks (distributed dense phase): only tile rows with ti % row_mod == row_rem are computed; the caller
    // zeroes C first and sums the ranks' pieces with one all-reduce (adding zeros is exact, so every rank gets identical bits)
    int row_mod = 1, row_rem = 0;
    int pdl = 0;   // launch with the programmatic-serialisation attribute (the kernels always run the PDL prologue)
    // warp -> sub-tile maps (one nibble per warp; 0 = the library default, see gemm.cu): general tiles / diagonal tiles of a symmetric product
    unsigned wmap = 0, wmap_diag = 0;
};

// Launch on `stream`. Returns cudaError_t as int (0 = ok), -1 for an unsupported combination.
int gemm_launch(const GemmP& p, cudaStream_t stream);

// C = beta*C + sum_s part[s]  over the tiles gemm_launch wrote (lower tiles only if lower_out)
int splitk_reduce_launch(const GemmP& p, cudaStream_t stream);

// gemm_launch that splits the contraction over otherwise idle SMs when the product has few output tiles (the latency-bound
// M x M phases at small M, Cholesky panels, triangular-inverse nodes): partial tiles go to `ws` (ws_doubles doubles, owned by
// the caller, one per stream) and are summed by splitk_reduce_launch.  Falls back to the plain launch when nothing is gained.
// The piece count is capped by ws_doubles / (batch m n): the workspace size decides how some products are split, and with it
// the order in which their partials are summed.
int gemm_launch_auto(GemmP p, cudaStream_t stream, double* ws, size_t ws_doubles);

// k split point for `tiles` equal output tiles of contraction length k on this device's SMs (multiple of 16; k = no split)
int balanced_ksplit(int tiles, int k);

// one-time: opt in to large dynamic shared memory for every instantiation
int gemm_init();

}  // namespace tsvgp
