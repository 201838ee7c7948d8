// Non-GEMM kernels of the t-SVGP path: covariance tiles, per-point likelihood statistics, M-vector products,
// diagonal-block factorisation, and small elementwise M x M utilities.  Launchers return cudaError_t as int.
#pragma once
#include <cuda_runtime.h>

namespace tsvgp {

enum { KERN_SE = 0, KERN_MATERN52 = 1, KERN_MATERN12 = 2, KERN_MATERN32 = 3 };
enum { LIK_GAUSSIAN = 0, LIK_BERNOULLI = 1, LIK_STUDENT_T = 2, LIK_SOFTMAX = 3, LIK_HETEROSKEDASTIC = 4 };
constexpr int MAX_SOFTMAX_CLASSES = 16;
constexpr int MAX_GH = 64;

struct LikSpec {
    int kind = LIK_GAUSSIAN;
    double p0 = 1.0;   // Gaussian: variance ; StudentT: scale ; heteroskedastic: scale transform (0 = exp, 1 = softplus)
    double p1 = 3.0;   // StudentT: df
    double c0 = 0.0;   // StudentT: log-density constant
    int n_gh = 20;
};

// Xs^T[d][n] = X[n][d] / ls[d]  (feature-major, leading dim ldx >= n_pad, columns n >= n zeroed) ; x2[n] = sum_d Xs^2
int scale_points_launch(const double* X, long n, int D, const double* ls, double* XsT, long ldx, double* x2, long n_pad,
                        cudaStream_t s);

// K[i][c] = k(z_i, x_{n0+c}) for i < Mp, c < ncols (multiple of 128).  Rows i >= M and columns n0+c >= n_valid are zero,
// or the identity (K[i][c] = (i == n0+c)) when pad_identity.  If alpha != null also writes
// mu_part[i/64][c] = sum_{i in 64-row group} alpha[i] K[i][c].
int kuf_launch(int kind, double variance, const double* XsT, long ldx, const double* x2, long n0, long n_valid, int ncols,
               const double* ZsT_rows /*Zs [Mp][D]*/, const double* z2, int M, int Mp, int D, const double* alpha, double* K,
               long ldk, double* mu_part, long ldmu, int pad_identity, cudaStream_t s, double* Kp = nullptr /* dk/dr2 slab */);

struct GHTable { double z[MAX_GH]; double w[MAX_GH]; };   // nodes sqrt(2) x_k and weights w_k / sqrt(pi), passed by value

struct PointArgs {
    const double* mu_part; int n_mu_part; long ldmu;   // partial means   [n_mu_part][ldmu]
    const double* q_part; int n_q_part; long ldq;      // partial |T^T k|^2 [n_q_part][ldq]   (subtracted from k(x,x); none: var = k(x,x))
    const double* q2_part = nullptr;                   // optional second set, same shape, ADDED (whitened sibling: + |LR^-1 k|^2)
    const double* y;            // [ncols] (chunk-local pointer) or null (predict)
    const double* mean_off;     // [ncols] mean_function(X) or null
    double kdiag;               // k(x,x) = kernel variance
    long n_valid;               // chunk-local number of real points (<= ncols)
    int ncols;
    double* g; double* h;       // out: d ve/d mean, clipped d ve/d var  (zero for padding columns), may be null
    double* mean_out; double* var_out;   // out (predict), may be null; written only for c < n_valid
    double* ve_blocks;          // out: per-block sum of ve   [gridDim.x]
    double* aux_blocks = nullptr;   // out (M-step): per-block [sum h, sum d ve / d likelihood parameter]   [2 * gridDim.x]
    int clip = 1;               // clip d ve / d var at -1e-8 (natgrad_step, tsvgp.py:262-263); the ELBO gradient does not
    int* flags;                 // flags[0] |= 1 if any var <= 0, or (x2 given) any mean or x2 is not finite
    const double* x2 = nullptr; // [ncols] squared norms of the scaled points (chunk-local), or null
};
// Softmax likelihood over L latents (gpflow.likelihoods.Softmax = MonteCarloLikelihood, S = num_monte_carlo_points): per point
//   ve = mean_s log softmax(f_s)[y],  f_s = mu + sqrt(var) * eps_s ;  g_l = d ve / d mu_l ;  h_l = min(d ve / d var_l, -1e-8)
// as called at reference tsvgp.py:256-263 (docs/notebooks/mnist.py:117-122).  Per-latent inputs / outputs are `*_lat` apart.
// clip = 0 (M-step gradients) leaves h_l unclipped and, with aux_blocks, adds the sum of h over the block's points and latents.
// eps: explicit standard-normal draws [S][n_total][L] (GPflow's layout) or null = Philox4x32-10 + Box-Muller keyed by (seed, draw).
// The heteroskedastic likelihood takes the same arguments (S, eps, seed and draw unused).
struct SoftmaxArgs {
    const double* mu_part; int n_mu_part; long ldmu, mu_lat;
    const double* q_part; int n_q_part; long ldq, q_lat;
    int L, S;
    const double* y;            // class labels as doubles (heteroskedastic: the observation), chunk-local
    const double* mean_off;
    double kdiag[MAX_SOFTMAX_CLASSES];   // k_l(x,x) = latent l's kernel variance
    long n_valid, n0, n_total;  // n0: global index of the chunk's first point (addresses eps / the random stream)
    int ncols;
    double* g; double* h; long gh_lat;
    double* mean_out; double* var_out; long out_lat;
    double* ve_blocks;
    int* flags;
    const double* eps;
    unsigned long long seed, draw;
    int clip = 1;                   // clip h_l at -1e-8 (natgrad_step); the ELBO gradient does not (heteroskedastic: always clipped)
    double* aux_blocks = nullptr;   // out (Softmax M-step): per 256 points [sum h over points and latents, 0], as PointArgs
    // whitened sibling (Softmax only): partial |LA^-1 k|^2 [n_q_part][ldq], one set shared by the latents and SUBTRACTED, while
    // the per-latent q_part (|LR_l^-1 k|^2) are ADDED: var_l = k(x,x) - (|LA^-1 k|^2 - |LR_l^-1 k|^2).  Null: var_l = k(x,x) - q_l
    const double* q_shared = nullptr;
    // [ncols] squared norms of the scaled points (chunk-local), or null.  Given, a point whose norm or any mean is not finite raises
    // the flag: the covariance clamps a NaN distance to a finite k, so such a point can leave every var_l finite and positive
    const double* x2 = nullptr;
};
int softmax_stats_launch(const SoftmaxArgs& a, cudaStream_t s);
// Heteroskedastic Normal likelihood over L = 2 latents (GPflow HeteroskedasticTFPConditional(Normal, scale_transform) with its
// NDiagGHQuadrature(2, n_gh)): log p(y | f) = Normal(loc = f_0, scale = T(f_1)).log_prob(y), T = exp (lik.p0 = 0) or softplus (1),
// integrated on the tensor-product grid f = mu + sqrt(v) (z_i, z_j), weights w_i w_j.  Per point: ve, g_l = d ve / d mu_l,
// h_l = min(d ve / d v_l, -1e-8); mean_out / var_out get the marginals of q(f) (predict).  One ve slot per 256 points.
int heteroskedastic_stats_launch(const LikSpec& lik, const SoftmaxArgs& a, const GHTable& gh, cudaStream_t s);
// Y [n][L] row-major -> Yt [L][ld] ; and back for outputs: src [L][ld] -> dst [n][L]
int transpose_to_latent_major_launch(const double* Y, long n, int L, double* Yt, long ld, cudaStream_t s);
int transpose_to_point_major_launch(const double* src, long ld, long n, int L, double* dst, cudaStream_t s);

// Posterior samples (tsvgp_predict_f_samples).  The standard normal eps(s, n, l) is the explicit eps [S][N][L] when given, else
// Philox4x32-10 + Box-Muller keyed by (seed, draw, point n, sample pair s / 2, latent l) — its own key, never the Softmax one.
struct SampleArgs {
    const double* eps;
    unsigned long long seed, draw;
    long N;
    int S, L;
};
// E[n][s] = eps(s, n, l) for n < N and s < S, zero elsewhere; E [Np][ld], ld even and >= S
int sample_normals_launch(const SampleArgs& a, int l, double* E, long ld, long Np, cudaStream_t s);
// out[s][n][l] = mean[n] + F[n][s]   (F [N][ldf]: the correlated draw of latent l)
int add_mean_samples_launch(const double* mean, const double* F, long ldf, long N, int S, int L, int l, double* out, cudaStream_t s);
// out[s][n][l] = mean[l][n] + sqrt(var[l][n]) eps(s, n, l)  (mean, var [L][ld])
int diag_samples_launch(const SampleArgs& a, const double* mean, const double* var, long ld, double* out, cudaStream_t s);

int point_stats_launch(const LikSpec& lik, const PointArgs& a, const GHTable& gh, cudaStream_t s);

// y[i] = alpha * sum_j A[i][j] x[j] + beta * y[i]      (row-major A [m][n], lda)
int gemv_n_launch(const double* A, long lda, int m, long n, const double* x, double alpha, double beta, double* y, cudaStream_t s);
// y[j] = sum_i A[i][j] x[i]   (uses work [nchunk][n]); deterministic two-stage
int gemv_t_launch(const double* A, long lda, int m, int n, const double* x, double* y, double* work, cudaStream_t s);

// work[c][j] = sum_{i in 64-row chunk c} A[i][j] x[i], leading dimension ldw  (partial means of a slab that already exists)
int gemv_t_part_launch(const double* A, long lda, int m, int n, const double* x, double* work, long ldw, cudaStream_t s);

// Zs[i][d] = ZsT[d][i]  (row-major copy of the scaled inducing inputs, [Mp][D])
int unpack_rows_launch(const double* ZsT, long ldz, int Mp, int D, double* Zs, cudaStream_t s);

int diag_init();   // once per device/context: opt in to the dynamic shared memory of the diagonal-block kernel
// --- diagonal blocks --------------------------------------------------------------------------------------------
// In-place lower Cholesky of the 128x128 block at A (lda) and its inverse into Dinv (ld 128, dense lower).
// info[0] = first failing global pivot index + 1 (blk_index*128 + k + 1), left untouched on success.
// Dinv must have been zero-filled once (cudaMemset) by its owner: the kernel never writes the strictly upper 32 x 32
// sub-blocks of Dinv, and leaves those of A to the caller (chol_lower zeroes the upper triangle at the end).
int diag_potrf_inv_launch(double* A, long lda, double* Dinv, int blk_index, int* info, cudaStream_t s);

// --- elementwise M x M utilities ---------------------------------------------------------------------------------
int add_diag_launch(double* A, long lda, int n, double v, cudaStream_t s);
int copy_add_diag_launch(const double* A, double* B, long ld, int n, double v, cudaStream_t s);           // B = A + v I
int mirror_lower_launch(double* A, long lda, int n, cudaStream_t s);                                       // A[j][i] = A[i][j], i > j
int flip_sym_launch(const double* W, double* Wf, long ld, int n, cudaStream_t s);                          // Wf[i][j] = W_sym[n-1-i][n-1-j], lower
int antitranspose_launch(const double* Linv, double* V, long ld, int n, cudaStream_t s);                   // V[i][j] = Linv[n-1-j][n-1-i] (lower), upper zero
int zero_upper_launch(double* A, long lda, int n, cudaStream_t s);
// L2 = -tril(P) on [0,M)^2, 0 elsewhere — skipped on the device when *bad != 0 or any of info[0..3] != 0 (failed step keeps old sites)
int finalize_sites_launch(const double* P, double* L2, long ld, int M, int Mp, const double* bad, const int* info, cudaStream_t s);
int trtri_seed_launch(const double* dinv, double* Linv, long ld, int n, cudaStream_t s);   // Linv = blockdiag(dinv[b]) (128 x 128 blocks), zero elsewhere
int dot_launch(const double* x, const double* y, int n, double* out, cudaStream_t s);
// lambda_1 <- (1-lr) lambda_1 + lr*scale*(G1 - 2 G2mZ)
int update_lambda1_launch(double* l1, const double* G1, const double* G2mZ, int n, double lr, double scale, const double* bad,
                          const int* info, cudaStream_t s);
// y = a x1 + b x2 ;  guarded y = a y + b x (skipped on the device after a failed step)
int lincomb_launch(double* y, double a, const double* x1, double b, const double* x2, int n, cudaStream_t s);
int axpby_vec_guarded_launch(double* y, const double* x, int n, double a, double b, const double* bad, const int* info, cudaStream_t s);
// y = a - b
int vsub_launch(const double* a, const double* b, double* y, int n, cudaStream_t s);

int matdot_launch(const double* A, const double* B, long ld, int n, double* out, double* part /* [128] caller-owned scratch */,
                  cudaStream_t s);   // sum_ij A_ij B_ij
int logdiag_launch(const double* A, long lda, int n, double* out, cudaStream_t s);                  // sum_i log A_ii
// P = coef*G + jitter*I on [0,M)^2, identity on the padding block
int init_update_launch(const double* G, double* P, long ld, int M, int Mp, double coef, double jitter, cudaStream_t s);
int set_scaled_identity_launch(double* A, long ld, int M, int Mp, double v, double vpad, cudaStream_t s);
int probe_vector_launch(double* v, int M, int Mp, cudaStream_t s);
// P = a P + b X on [0,M)^2 unless *bad != 0 or any info slot != 0 (guarded commit of the whitened sibling's Lambda_2)
int axpby_guarded_launch(double* P, const double* X, long ld, int M, double a, double b, const double* bad, const int* info, cudaStream_t s);
int vadd_inplace_launch(double* dst, const double* src, long n, cudaStream_t s);
int stats_tail_launch(const double* ve_blocks, long nblocks, const int* flags, const double* aux, double* out, cudaStream_t s);
// Gaussian natgrad_step, whose pass took var = k(x,x): with tr[0] = tr(P^T B P) and q = tr[0] * inv_c = sum_n |T^T k_n|^2,
// out[0] (sum ve) += half_inv_s2 * q, and out[1] (the variance flag) = 1 unless sum_n v_n = sum_kdiag - q is finite and positive
int variance_term_launch(const double* tr, double inv_c, double sum_kdiag, double half_inv_s2, double* out, cudaStream_t s);
// M-step gradient helpers (see tsvgp_elbo_grad)
// E = scale (alpha g^T - 2 U diag(h)) .* Kp, written over U (E = null) or added to E (a coupled likelihood's latents share one E)
int egrad_uf_launch(double* U, const double* Kp, long ld, int Mp, int ncols, const double* alpha, const double* g, const double* h,
                    double scale, cudaStream_t s, double* E = nullptr);
// Xa[c][0:W] = [xs - origin | 1 | (xs - origin)^2 | 0] of point n0 + c (origin [D] device vector or null); W = aug_width(D)
int xaug_launch(const double* XsT, long ldx, long n0, long nvalid, int ncols, int D, double* Xa, cudaStream_t s, const double* origin = nullptr);
inline int aug_width(int D) { return (2 * D + 1 + 127) / 128 * 128; }
int gamma_uu_launch(const double* QBQ, const double* QKQ, const double* qb, const double* qm, const double* al, const double* Kp,
                    double* Gamma, double* E, long ld, int n, double scale, cudaStream_t s);
// the whitened sibling's counterpart (tsvgp.cu, grad_epilogue_white): D = A^-1 B A^-1 - R^-1 B R^-1, W = R0^-1 A R0^-1
int gamma_uu_white_launch(const double* D, const double* W, const double* R0inv, const double* Ainv, const double* rb, const double* al,
                          const double* a0, const double* w, const double* Kp, double* Gamma, double* E, long ld, int n, double scale,
                          cudaStream_t s);

}  // namespace tsvgp
