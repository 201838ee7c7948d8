#include "dense.cuh"
#include "gemm.cuh"
#include "kernels.cuh"
#include "common.cuh"

namespace tsvgp {

#define TRY(x) do { int e_ = (x); if (e_) return e_; } while (0)

// ---- 32-row strip product for the Cholesky's critical path [r02] ---------------------------------------------------------------
//   C[r0 : r0+32, 0:128] = alpha * A[r0 : r0+32, 0:128] * B[0:128, 0:128]^T + beta * C          (B stored [j][k], k contiguous)
// One CTA per 32 rows, the whole 128 x 128 B in shared memory.  It replaces, per block column of chol_lower, the panel solve
// (A = C = the panel, B = the inverse of the diagonal block, lower triangular: b_lower skips its zero 8 x 8 blocks) and the update of
// the next block column (A = the panel, B = its first 128 rows, alpha = -1, beta = 1): the generic 128 x 128-tile engine needed a
// split-K launch plus a reduction kernel for each of them (4 launches, ~29 us per block column at M = 2048); these are 2 launches
// of up to n/32 CTAs.  In-place use (C == A) is safe: a CTA stages its own 32 rows completely before it stores.
constexpr int SG_LD = 132;   // 128 + 4: the 8 rows of a fragment read hit distinct banks
constexpr int SG_SMEM = (32 + 128) * SG_LD * 8;
__global__ void __launch_bounds__(256) strip_gemm_kernel(const double* __restrict__ A, long lda, const double* __restrict__ B, long ldb,
                                                         double* C, long ldc, double alpha, double beta, int b_lower) {
    PDL_PROLOGUE();
    extern __shared__ __align__(16) double sg[];
    double* sA = sg;                 // [32][SG_LD]
    double* sB = sg + 32 * SG_LD;    // [128][SG_LD]
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, g = lane >> 2, t = lane & 3;
    const long r0 = (long)blockIdx.x * 32;
    for (int u = tid; u < 32 * 64; u += 256) {
        const int r = u >> 6, c = (u & 63) * 2;
        cp_async16(sA + r * SG_LD + c, A + (r0 + r) * lda + c);
    }
    for (int u = tid; u < 128 * 64; u += 256) {
        const int r = u >> 6, c = (u & 63) * 2;
        cp_async16(sB + r * SG_LD + c, B + (long)r * ldb + c);
    }
    cp_async_commit();
    cp_async_wait<0>();
    __syncthreads();
    // warp w owns the column blocks w and 15 - w (8 columns each) of all four 8-row blocks: with a lower-triangular B the contraction
    // of column block jb stops at k = 8 (jb + 1), and (w + 1) + (16 - w) = 17 k-blocks for every warp
    const int jb0 = warp, jb1 = 15 - warp;
    const int k0max = b_lower ? 8 * (jb0 + 1) : 128, k1max = b_lower ? 8 * (jb1 + 1) : 128;
    double acc[4][2][2];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 2; ++j) { acc[i][j][0] = 0.0; acc[i][j][1] = 0.0; }
#pragma unroll 4
    for (int kk = 0; kk < k1max; kk += 4) {
        double a[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) a[i] = sA[(8 * i + g) * SG_LD + kk + t];
        const double b1 = sB[(8 * jb1 + g) * SG_LD + kk + t];
#pragma unroll
        for (int i = 0; i < 4; ++i) dmma884(acc[i][1][0], acc[i][1][1], a[i], b1);
        if (kk < k0max) {
            const double b0 = sB[(8 * jb0 + g) * SG_LD + kk + t];
#pragma unroll
            for (int i = 0; i < 4; ++i) dmma884(acc[i][0][0], acc[i][0][1], a[i], b0);
        }
    }
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 2; ++j) {
            const int col = 8 * (j ? jb1 : jb0) + 2 * t;
            double2* ptr = reinterpret_cast<double2*>(C + (r0 + 8 * i + g) * ldc + col);
            double2 o = make_double2(alpha * acc[i][j][0], alpha * acc[i][j][1]);
            if (beta != 0.0) { const double2 old = *ptr; o.x += beta * old.x; o.y += beta * old.y; }
            *ptr = o;
        }
}

int dense_init() {
    return (int)cudaFuncSetAttribute(strip_gemm_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, SG_SMEM);
}
static int strip_gemm_launch(const double* A, long lda, const double* B, long ldb, double* C, long ldc, int rows, double alpha, double beta,
                             int b_lower, cudaStream_t s) {
    launch_k(true, strip_gemm_kernel, rows / 32, 256, SG_SMEM, s, A, lda, B, ldb, C, ldc, alpha, beta, b_lower);
    return count_launch();
}

constexpr int NB = 128;
static int g_chol_outer = 512;   // outer panel width of the two-level blocking (multiple of 128)

// Right-looking with look-ahead over two streams.  Per block column q, on `s` (the critical path):
//   diag(q) -> panel(q) = A[q+1:, q] L_qq^-T -> [wait: trailing(q-1) done] -> A[q+1:, q+1] -= panel(q) panel(q)[0]^T  -> diag(q+1) ...
// and on aux->s2, once panel(q) exists:  A[q+2:, q+2:] -= panel(q)[1:] panel(q)[1:]^T  (lower tiles), hidden under diag(q+1).
// The two streams always write disjoint block columns (q+1 on `s`, >= q+2 on s2); `s` joins s2 before it returns.
static int chol_lower_lookahead(double* A, long ld, int n, double* dinv, int* info, cudaStream_t s, const CholAux& aux) {
#define CUQ(x) do { cudaError_t e_ = (x); if (e_ != cudaSuccess) return (int)e_; } while (0)
    bool f_pending = false;
    for (int q = 0; q < n; q += NB) {
        double* Aqq = A + (long)q * ld + q;
        double* Dq = dinv + (long)(q / NB) * NB * NB;
        TRY(diag_potrf_inv_launch(Aqq, ld, Dq, q / NB, info, s));
        const int below = n - (q + NB);
        if (below <= 0) break;
        double* panel = A + (long)(q + NB) * ld + q;
        TRY(strip_gemm_launch(panel, ld, Dq, NB, panel, ld, below, 1.0, 0.0, 1, s));   // panel <- panel * L_qq^-T, 32-row strips
        const int rest = below - NB;   // rows / columns from q + 2 blocks on
        if (rest > 0) {   // trailing update of the columns >= q+2 on the helper stream
            CUQ(cudaEventRecord(aux.e, s));
            CUQ(cudaStreamWaitEvent(aux.s2, aux.e, 0));
            GemmP p;
            const double* Lp = panel + (long)NB * ld;
            p.A = Lp; p.lda = ld; p.a_kc = 1;
            p.B = Lp; p.ldb = ld; p.b_kc = 1;
            p.C = A + (long)(q + 2 * NB) * ld + (q + 2 * NB); p.ldc = ld;
            p.m = rest; p.n = rest; p.k = NB;
            p.alpha = -1.0; p.beta = 1.0; p.lower_out = 1;
            // trailing(q-1) precedes it in s2's own order; block column q+1 is written on `s` meanwhile (disjoint)
            TRY(gemm_launch_auto(p, aux.s2, nullptr, 0));
        }
        // block column q+1 on the critical stream; trailing(q-1), which also wrote this column, must be complete
        if (f_pending) CUQ(cudaStreamWaitEvent(s, aux.f, 0));
        TRY(strip_gemm_launch(panel, ld, panel, ld, A + (long)(q + NB) * ld + (q + NB), ld, below, -1.0, 1.0, 0, s));
        if (rest > 0) { CUQ(cudaEventRecord(aux.f, aux.s2)); f_pending = true; }
        else f_pending = false;
    }
    if (f_pending) CUQ(cudaStreamWaitEvent(s, aux.f, 0));
#undef CUQ
    return zero_upper_launch(A, ld, n, s);
}

int chol_lower(double* A, long ld, int n, double* dinv, int* info, cudaStream_t s, double* ws, size_t ws_doubles, const CholAux* aux) {
    // measured (tools/diag_bench, profiles/diag_r02.txt): 1.12 -> 1.04 ms at n = 2048, 2.98 -> 2.90 ms at n = 4096; at n = 8192 the
    // single-level trailing updates (k = 128 per pass over the trailing matrix) lose to the two-level blocking below (12.4 vs 10.8 ms)
    if (aux && aux->s2 && n >= 4 * NB && n <= 4096) return chol_lower_lookahead(A, ld, n, dinv, info, s, *aux);
    const int OB = g_chol_outer;
    for (int P0 = 0; P0 < n; P0 += OB) {
        const int Pend = P0 + OB < n ? P0 + OB : n;
        for (int q = P0; q < Pend; q += NB) {
            double* Aqq = A + (long)q * ld + q;
            double* Dq = dinv + (long)(q / NB) * NB * NB;
            TRY(diag_potrf_inv_launch(Aqq, ld, Dq, q / NB, info, s));
            const int below = n - (q + NB);
            if (below <= 0) continue;
            double* panel = A + (long)(q + NB) * ld + q;
            {   // panel <- panel * L_qq^-T   (in place; B(k,j) = Linv[j][k])
                GemmP p;
                p.A = panel; p.lda = ld; p.a_kc = 1;
                p.B = Dq; p.ldb = NB; p.b_kc = 1;
                p.C = panel; p.ldc = ld;
                p.m = below; p.n = NB; p.k = NB;
                TRY(gemm_launch_auto(p, s, ws, ws_doubles));
            }
            const int ncols = Pend - (q + NB);
            if (ncols > 0) {   // update the rest of the outer panel: A[q+NB:, q+NB:Pend] -= panel * panel[0:ncols]^T
                GemmP p;
                p.A = panel; p.lda = ld; p.a_kc = 1;
                p.B = panel; p.ldb = ld; p.b_kc = 1;
                p.C = A + (long)(q + NB) * ld + (q + NB); p.ldc = ld;
                p.m = below; p.n = ncols; p.k = NB;
                p.alpha = -1.0; p.beta = 1.0; p.lower_out = 1;
                TRY(gemm_launch_auto(p, s, ws, ws_doubles));
            }
        }
        if (Pend < n) {   // trailing matrix -= L[Pend:, P0:Pend] L[Pend:, P0:Pend]^T
            GemmP p;
            const double* Lp = A + (long)Pend * ld + P0;
            p.A = Lp; p.lda = ld; p.a_kc = 1;
            p.B = Lp; p.ldb = ld; p.b_kc = 1;
            p.C = A + (long)Pend * ld + Pend; p.ldc = ld;
            p.m = n - Pend; p.n = n - Pend; p.k = Pend - P0;
            p.alpha = -1.0; p.beta = 1.0; p.lower_out = 1;
            TRY(gemm_launch_auto(p, s, ws, ws_doubles));
        }
    }
    return zero_upper_launch(A, ld, n, s);
}

// Bottom-up triangular inverse.  At level h (blocks) every node [lo, lo + 2h) combines its finished halves:
//   Linv[right, left] = -Linv[right, right] * L[right, left] * Linv[left, left]
// All full nodes of a level have the same shape and a constant stride, so they go out as ONE batched launch per product
// (2 launches per level instead of 2 per node); a ragged last node (n not a power of two) is launched on its own.
static int trtri_level(const double* L, long ld, int lo, int hl, int hr, int batch, long stride, double* Linv, double* tmp,
                       long tmp_stride, cudaStream_t s, double* ws, size_t ws_doubles) {
    const int mid = lo + hl;
    const int mrows = hr * NB, ncols = hl * NB;
    {   // tmp = C * Ainv,  C = L[right, left],  Ainv = Linv[left, left] (lower: B(k,j) != 0 only for k >= j)
        GemmP p;
        p.A = L + (long)mid * NB * ld + (long)lo * NB; p.lda = ld; p.a_kc = 1;
        p.B = Linv + (long)lo * NB * ld + (long)lo * NB; p.ldb = ld; p.b_kc = 0; p.b_tri = 2;
        p.C = tmp; p.ldc = ld;
        p.m = mrows; p.n = ncols; p.k = ncols;
        p.batch = batch; p.sA = stride; p.sB = stride; p.sC = tmp_stride;
        TRY(gemm_launch_auto(p, s, ws, ws_doubles));
    }
    {   // Linv[right, left] = -Binv * tmp,  Binv = Linv[right, right] (lower: A(i,k) != 0 only for k <= i)
        GemmP p;
        p.A = Linv + (long)mid * NB * ld + (long)mid * NB; p.lda = ld; p.a_kc = 1; p.a_tri = 1;
        p.B = tmp; p.ldb = ld; p.b_kc = 0;
        p.C = Linv + (long)mid * NB * ld + (long)lo * NB; p.ldc = ld;
        p.m = mrows; p.n = ncols; p.k = mrows;
        p.alpha = -1.0;
        p.batch = batch; p.sA = stride; p.sB = tmp_stride; p.sC = stride;
        TRY(gemm_launch_auto(p, s, ws, ws_doubles));
    }
    return 0;
}

int trtri_lower(const double* L, long ld, int n, const double* dinv, double* Linv, double* tmp, cudaStream_t s, double* ws, size_t ws_doubles) {
    const int nblk = n / NB;
    TRY(trtri_seed_launch(dinv, Linv, ld, n, s));
    for (int h = 1; h < nblk; h *= 2) {
        const int full = nblk / (2 * h);                 // nodes with both halves of size h
        const long stride = (long)2 * h * NB * (ld + 1);
        const long tmp_stride = (long)h * NB * ld;       // node b's scratch: rows [b*h*NB, (b+1)*h*NB) of tmp
        if (full > 0) TRY(trtri_level(L, ld, 0, h, h, full, stride, Linv, tmp, tmp_stride, s, ws, ws_doubles));
        const int lo = full * 2 * h, rem = nblk - lo;    // ragged node: left half complete, right half shorter
        if (rem > h) TRY(trtri_level(L, ld, lo, h, rem - h, 1, 0, Linv, tmp, 0, s, ws, ws_doubles));
    }
    return 0;
}

}  // namespace tsvgp
