// Blocked dense M x M factorisations built on the DMMA GEMM engine and the diagonal-block kernels.
// All matrices row-major, n a multiple of 128, explicit zeros in the unused triangle on output.
#pragma once
#include <cuda_runtime.h>

namespace tsvgp {

// In-place lower Cholesky A = L L^T (reads the lower triangle of A; upper triangle zeroed on return).
// dinv: workspace [n/128][128*128], receives the inverses of the diagonal blocks of L.
// info: device int, set to (failing pivot index + 1) if A is not positive definite (left untouched otherwise).
// Restates tf.linalg.cholesky as called at reference src/models/tsvgp.py:270,300 and src/util.py:382.
// ws / ws_doubles: optional split-K workspace (gemm_launch_auto) private to the stream; nullptr = never split.
// aux (optional): a helper stream and two events private to the caller's stream.  With it the factorisation runs with LOOK-AHEAD:
// after panel q only block column q+1 is updated on `s` (so the next diagonal block can start at once); the rest of the trailing
// update (columns >= q+2) runs on aux->s2 underneath the next diagonal-block kernel, which is one CTA and leaves 147 SMs idle.
int dense_init();   // once per process: opt in to the strip kernel's dynamic shared memory

struct CholAux { cudaStream_t s2 = nullptr; cudaEvent_t e = nullptr, f = nullptr; };
int chol_lower(double* A, long ld, int n, double* dinv, int* info, cudaStream_t s, double* ws = nullptr, size_t ws_doubles = 0,
               const CholAux* aux = nullptr);

// Linv = L^-1 for lower-triangular L.  dinv must hold the inverses of L's diagonal blocks (from chol_lower).
// tmp: workspace [ceil(n/256)*128][ld].  Turns tf.linalg.triangular_solve / cholesky_solve
// (reference tsvgp.py:271, util.py:386) into tensor-core products.
int trtri_lower(const double* L, long ld, int n, const double* dinv, double* Linv, double* tmp, cudaStream_t s, double* ws = nullptr,
                size_t ws_doubles = 0);

}  // namespace tsvgp
