/*
 * tsvgp.h — C ABI of libtsvgp.so: the B200 (sm_100a) implementation of t-SVGP's dual-parameterised natural-gradient
 * site update and its two read-only companions.
 *
 * The reference (AaltoML/t-SVGP) is pure Python on GPflow/TensorFlow and has NO FFI of its own; the boundary this
 * library replaces is the method surface of `t_SVGP` (reference src/models/tsvgp.py).  Each entry point below cites the
 * reference code it stands in for.  The Python mirror of that surface (t-svgp_b200/model.py) binds these symbols with
 * ctypes and hands tensors over as DLPack capsules (tsvgp_dlpack_view) — see INTEGRATION.md.
 *
 * Conventions
 *   - every array is float64, C-contiguous (row-major); num_latent_gps L = 1 in this round
 *   - every `const double*` / `double*` argument may be a HOST pointer (pageable or pinned) or a DEVICE pointer on the
 *     context's GPU; the library detects which (cudaPointerGetAttributes) and copies as needed
 *   - return value: 0 = ok, < 0 = error code below; tsvgp_last_error() gives the message.  Calls on one context are
 *     not re-entrant (one host thread per context); every call returns after its outputs are visible to the host
 *   - the library owns no caller memory; inputs are borrowed for the duration of the call (set_data copies a host
 *     minibatch to the device, or aliases a device one until the next set_data)
 *   - there is NO CPU fallback: without a CUDA device every compute entry point fails with TSVGP_ERR_CUDA
 */
#ifndef TSVGP_H
#define TSVGP_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define TSVGP_ABI_VERSION 1
#if defined(__GNUC__)
#define TSVGP_API __attribute__((visibility("default")))
#else
#define TSVGP_API
#endif

enum {
    TSVGP_OK = 0,
    TSVGP_ERR_INVALID = -1,           /* bad argument / shape (reference: tf.debugging.assert_shapes, util.py:368-372)  */
    TSVGP_ERR_CUDA = -2,              /* CUDA runtime failure, or no device                                              */
    TSVGP_ERR_NOT_POSITIVE_DEFINITE = -3, /* a Cholesky failed (reference: TF InvalidArgumentError from tf.linalg.cholesky);
                                             tsvgp_last_info() = 1-based failing pivot, LAPACK style                     */
    TSVGP_ERR_NONPOSITIVE_VARIANCE = -4,  /* some predictive variance <= 0 (reference: tf.debugging.assert_positive,
                                             tsvgp.py:113)                                                               */
    TSVGP_ERR_COMM = -5,              /* NCCL failure                                                                    */
    TSVGP_ERR_STATE = -6              /* called before the kernel / inducing points / data it needs were set             */
};

/* gpflow.kernels.{SquaredExponential,Matern52,Matern12,Matern32}; the Matern kernels take r = sqrt(max(r2, 1e-36)) as GPflow does.
 * Matern12's derivative in r2 (tsvgp_elbo_grad) is the one autodiff takes through that clamp: 0 for r2 < 1e-36.            */
enum { TSVGP_KERNEL_SE = 0, TSVGP_KERNEL_MATERN52 = 1, TSVGP_KERNEL_MATERN12 = 2, TSVGP_KERNEL_MATERN32 = 3 };
/* gpflow.likelihoods.*; TSVGP_LIK_HETEROSKEDASTIC: HeteroskedasticTFPConditional(distribution_class = Normal), see set_likelihood */
enum { TSVGP_LIK_GAUSSIAN = 0, TSVGP_LIK_BERNOULLI_PROBIT = 1, TSVGP_LIK_STUDENT_T = 2, TSVGP_LIK_SOFTMAX = 3, TSVGP_LIK_HETEROSKEDASTIC = 4 };

typedef struct tsvgp_ctx tsvgp_ctx;   /* opaque: owns one CUDA stream, device buffers, optional NCCL communicator */

/* ---- lifetime ------------------------------------------------------------------------------------------------- */
TSVGP_API int tsvgp_abi_version(void);
TSVGP_API int tsvgp_create(tsvgp_ctx** out, int device_id);          /* replaces t_SVGP.__init__ (tsvgp.py:122-157) device side    */
TSVGP_API void tsvgp_destroy(tsvgp_ctx* ctx);
TSVGP_API const char* tsvgp_last_error(const tsvgp_ctx* ctx);        /* ctx may be NULL: message of the last failed tsvgp_create    */
TSVGP_API int tsvgp_last_info(const tsvgp_ctx* ctx);                 /* failing pivot of the last TSVGP_ERR_NOT_POSITIVE_DEFINITE   */
TSVGP_API int tsvgp_set_option(tsvgp_ctx* ctx, const char* name, double value);   /* see below */

/* options: "chunk" (points per Kuf slab; 0 = automatic = 16384 points, i.e. Mp x 16384 x 8 B per slab stream — 268 MB at M = 2048,
 *          larger than the 126 MB L2: the slab is written once and re-read Mp/128 times through L2/HBM by compute-bound DMMA
 *          products, measured at ~4 % of the HBM roof), "streams" (1 to 4 ping-pong slab streams; default 2),
 * "cache_factors" (1 = keep chol(Kuu+jitter I) and the posterior factors while kernel, Z and sites are unchanged),
 * "invalidate" (any value: drop every cached factor now),
 * "route" (0 = automatic, 1 = fused: B = Kuf diag(h) Kfu then K9^-1 B K9^-1 — 2 M^2 flops per point, rounding ~ eps cond(Kuu)^2;
 *          2 = whitened: C9^-1 Kuf first, as the reference's order A = K9^-1 Kuf — 3 M^2 flops per point, rounding ~ eps cond;
 *          3 = exact: A = K9^-1 Kuf formed per slab, then the Gram product A^T diag(h) A — the reference's order literally
 *              (tsvgp.py:271-281), 4 M^2 flops per point; keeps -2 Lambda_2 positive definite where the reference's does),
 * "white" (1 = the whitened sibling t_SVGP_white, reference src/models/tsvgp_white.py: the second site argument of
 *          set_sites / get_sites / get_lambda_2 is then the full matrix Lambda_2; switching resets the sites),
 * "dist_min_m" (multi-GPU: distribute the dense M x M products over the ranks from this padded M upwards; default 4096),
 * "shard_min_m" (multi-GPU, fused route: from this padded M upwards (default 2048; needs (M/128) % ranks == 0) the statistics are
 *          reduce-scattered by tile rows, G2 = K9^-1 B K9^-1 is formed on each rank's rows and assembled by two all-gathers,
 *          instead of an all-reduce followed by the full products on every rank; a huge value switches it off),
 * "split_chains" (multi-GPU, same size gate and below dist_min_m; default 0; 1: when the Kuu + jitter I chain is joined after the
 *          pass (fused route forced or speculated) rank 0 builds the posterior factors, rank 1 the Kuu + jitter I chain, each
 *          broadcasts its result (ncclBroadcast) — every rank holds the same bits as without the split — and every rank but 0
 *          fills the wait with early slabs; pays off with row shares from tsvgp_b200.balance_weights, see DESIGN 5),
 * "route_cond_max" (automatic: fused while the power-iteration estimate of cond(Kuu + jitter I) is below this; default 1e4),
 * "route_exact_min" (automatic: exact above this estimate, whitened in between; default 1e8),
 * "mc_seed" (Softmax: key of the Monte-Carlo generator; resets the draw counter),
 * "sample_seed" (tsvgp_predict_f_samples: key of its own generator; resets its own draw counter — never touches "mc_seed"'s),
 * "speculate" (1 = automatic route: when this context's last conditioning estimate chose the fused route, run the
 *          Kuu + jitter I chain UNDERNEATH the streaming pass instead of in front of it, read the probe after the pass and
 *          repeat the pass with the right route if the estimate crossed the threshold; 0 = always probe before the pass),
 * "early_slabs" (n = Gaussian likelihood, fused route: Kuf and the constant-weight SYRK of the first slab of up to n slab
 *          streams do not depend on the posterior and are enqueued before the posterior chain; 0 = off).
 * Environment (read by tsvgp_create): TSVGP_PDL=0 plain stream order instead of programmatic dependent launch for
 * the M x M kernel chains; TSVGP_DEBUG_SYNC=1 synchronise after every launch, so that a faulting kernel is reported at its call
 * site. */

/* ---- model objects read by the path (tsvgp.py:209,268-269; GPflow kernel / likelihood / inducing attributes) ------ */
/* lengthscales: HOST pointer, n_ls = 1 (isotropic) or D (ARD).  One kernel shared by every latent (returns a context in
 * separate-kernel mode to shared mode).                                                                                */
TSVGP_API int tsvgp_set_kernel(tsvgp_ctx* ctx, int kind, double variance, const double* lengthscales, int n_ls);
/* One kernel PER LATENT (gpflow.kernels.SeparateIndependent with SharedIndependentInducingVariables): kinds, variances and
 * n_ls have L = tsvgp_num_latent entries (HOST); lengthscales holds the latents' n_ls[l] (1 or D) entries back to back.
 * Every latent then uses its own Kuu_l, Kuu_l + 1e-6 I, Kuu_l + jitter I and Kuf_l; the conditional, the KL and the site update
 * of each latent keep their form with these matrices.  Validated as tsvgp_set_kernel.  tsvgp_set_num_latent with a different L
 * drops the per-latent kernels (compute calls return TSVGP_ERR_STATE until the next set_kernels / set_kernel).  Not built:
 * option "white" = 1 and tsvgp_elbo_grad (TSVGP_ERR_INVALID).  Memory per extra latent: 5 M x M matrices and a scaled copy of
 * the resident X.                                                                                                      */
TSVGP_API int tsvgp_set_kernels(tsvgp_ctx* ctx, const int* kinds, const double* variances, const double* lengthscales, const int* n_ls);
/* Gaussian: p0 = variance.  StudentT: p0 = scale, p1 = df.  Bernoulli: inv_probit link with GPflow's 1e-3 jitter.
 * n_gh Gauss-Hermite points (<= 64; GPflow default 20); gh_x/gh_w (HOST, numpy.polynomial.hermite.hermgauss order)
 * may be NULL, in which case the library generates them.
 * Heteroskedastic: log p(y | f) = Normal(loc = f_0, scale = T(f_1)).log_prob(y) over L = 2 latents (checked at the first compute
 * call), p0 = 0: T = exp, 1: T = softplus; the expectation is the n_gh x n_gh Gauss-Hermite grid (GPflow NDiagGHQuadrature).
 * Y [N, 1] like Softmax; tsvgp_elbo_grad and option "white" are not built for it.                                      */
TSVGP_API int tsvgp_set_likelihood(tsvgp_ctx* ctx, int kind, double p0, double p1, int n_gh, const double* gh_x, const double* gh_w);
/* Z [M, D] inducing inputs (inducing_variable.Z); mean_Z [M] = mean_function(Z) or NULL for the Zero mean function     */
TSVGP_API int tsvgp_set_inducing(tsvgp_ctx* ctx, const double* Z, int M, int D, const double* mean_Z);
/* num_latent_gps = L (tsvgp.py:122-134, 276-281; default 1): L latent GPs that share the kernel and the inducing inputs, each with
 * its own site pair, in ONE context — one Kuu / Kuu + jitter I chain and one Kuf slab per launch serve all of them; the variance
 * product, the weighted SYRK and the site update run per latent.  Layouts follow the reference: lambda_1 [M, L], lambda_2_sqrt
 * [L, M, M], Y [N, L] (independent likelihood terms, summed over the latent axis) or [N, 1] class labels (Softmax), predictive
 * moments [N, L].  Resets the sites and drops the resident data.  The whitened sibling (option "white") takes any L too — Lambda_2
 * [L, M, M], tsvgp_white.py:79-89 — the Softmax likelihood included (variance gradient unclipped, as tsvgp_white.py:183-212).   */
TSVGP_API int tsvgp_set_num_latent(tsvgp_ctx* ctx, int L);
TSVGP_API int tsvgp_num_latent(const tsvgp_ctx* ctx);
/* TSVGP_LIK_SOFTMAX (gpflow.likelihoods.Softmax, docs/notebooks/mnist.py:117-122): set_likelihood with p0 = number of classes
 * (= L) and n_gh = Monte-Carlo points per data point (GPflow: 100).  GPflow draws fresh standard normals [S, N, L] in every
 * call; here they come from a counter-based generator (Philox4x32-10 + Box-Muller, option "mc_seed", a new draw per call) or,
 * for reproducible comparisons, from an explicit array eps [S, N, L] (HOST or DEVICE; used whenever a pass runs over exactly
 * N points; NULL clears it).  tsvgp_elbo and tsvgp_elbo_grad each take one draw: elbo_grad at draw k sees the draws (and
 * returns the ELBO) that tsvgp_elbo would at draw k.                                                                           */
TSVGP_API int tsvgp_set_mc_epsilon(tsvgp_ctx* ctx, const double* eps, int S, int64_t N, int L);

/* ---- DenseSites state (src/sites.py:43-80): lambda_1 [M, L], lambda_2_sqrt [L, M, M] lower triangular ------------- */
/* NULL lambda_1 / lambda_2_sqrt = the reference defaults 0 and -1e-10 * I (tsvgp.py:174-180). Upper triangle ignored.  */
TSVGP_API int tsvgp_set_sites(tsvgp_ctx* ctx, const double* lambda_1, const double* lambda_2_sqrt);
TSVGP_API int tsvgp_get_sites(tsvgp_ctx* ctx, double* lambda_1, double* lambda_2_sqrt);     /* either may be NULL                  */
TSVGP_API int tsvgp_get_lambda_2(tsvgp_ctx* ctx, double* lambda_2);                          /* L2 L2^T (tsvgp.py:197-200)          */

/* ---- data: this rank's rows of the minibatch ------------------------------------------------------------------------ */
/* X [N, D], Y [N, 1] ([N, L] for L latents with independent likelihood terms), mean_X [N] = mean_function(X) or NULL.
 * Host data is copied; device data is aliased.                                                                          */
TSVGP_API int tsvgp_set_data(tsvgp_ctx* ctx, const double* X, const double* Y, int64_t N, int D, const double* mean_X);

/* Input pipeline (stands in for the tf.data prefetch of the reference's minibatch callers, docs/notebooks/mnist.py:85,150):
 * stage_data copies the NEXT minibatch into a second set of device buffers on a copy stream and returns at once (host
 * buffers should be pinned and must stay valid until commit_staged); commit_staged makes it the resident minibatch.       */
TSVGP_API int tsvgp_stage_data(tsvgp_ctx* ctx, const double* X, const double* Y, int64_t N, int D, const double* mean_X);
TSVGP_API int tsvgp_commit_staged(tsvgp_ctx* ctx);

/* ---- the hot path ----------------------------------------------------------------------------------------------------- */
/* t_SVGP.natgrad_step (tsvgp.py:234-304) on the resident data and sites.  scale = num_data / minibatch_size or 1
 * (tsvgp.py:286-291) with minibatch_size summed over ranks.  elbo_before (may be NULL) receives the ELBO of the
 * pre-update state on the same minibatch (a by-product of the same pass).
 * TSVGP_ERR_NONPOSITIVE_VARIANCE (sites unchanged): some v_n <= 0 or non-finite.  The Gaussian likelihood's update does not
 * read v_n, so its step forms no per-point variance: it reports the error when a point of X or its predictive mean is not finite
 * and, with elbo_before, when the sum of the variances taken from the statistics is not finite and positive.       */
TSVGP_API int tsvgp_natgrad_step(tsvgp_ctx* ctx, double lr, double jitter, double scale, double* elbo_before);
/* base_SVGP.elbo (tsvgp.py:79-95) on the resident data                                                                 */
TSVGP_API int tsvgp_elbo(tsvgp_ctx* ctx, double scale, double* out);
/* base_SVGP.prior_kl (tsvgp.py:65-70): KL[q(u) || p(u)] of the current sites                                            */
TSVGP_API int tsvgp_prior_kl(tsvgp_ctx* ctx, double* out);
/* M-step: ELBO of the resident minibatch and its gradient w.r.t. the kernel variance, the lengthscales (n_ls entries, as
 * given to tsvgp_set_kernel), the inducing inputs Z [M, D] and the likelihood parameter (Gaussian: variance; StudentT:
 * scale; Bernoulli, Softmax: 0), with the sites held fixed — what the reference obtains by TensorFlow autodiff through
 * `elbo` (tsvgp.py:79-95; callers docs/notebooks/mnist.py:161-163,188-189; pinned by tests/models/test_tsvgp.py:168-188).
 * Gradients are w.r.t. the constrained (natural) parameter values; Zero mean function; any D; one kernel shared by the
 * latents.  Softmax: the derivatives of the Monte-Carlo sum for the call's draws (one per call, see tsvgp_set_mc_epsilon),
 * with h = d ve / d var unclipped; one pass over the data for all latents.  The whitened sibling (option "white") holds its
 * own sites fixed, lambda_1 and the full Lambda_2, and runs one pass per latent like the plain model, or with Softmax one pass
 * over all latents (DESIGN 10).  Collective with several ranks.  Not built for the heteroskedastic likelihood or separate kernels per latent (TSVGP_ERR_INVALID).    */
TSVGP_API int tsvgp_elbo_grad(tsvgp_ctx* ctx, double scale, double* elbo, double* d_variance, double* d_lengthscales,
                              double* d_Z, double* d_lik);
/* base_SVGP.predict_f, full_cov = False (tsvgp.py:97-114): mean_out, var_out [N, L]                                     */
TSVGP_API int tsvgp_predict_f(tsvgp_ctx* ctx, const double* Xnew, int64_t N, int D, const double* mean_X, double* mean_out, double* var_out);
/* base_SVGP.predict_f, full_cov = True (tsvgp.py:97-114 -> GPflow conditional): mean_out [N, L], cov_out [L, N, N] with
 * Sigma_l = k(X, X) - V_l^T V_l, V_l = T_l^T Kuf (DESIGN 13).  Only the diagonal of Sigma_l is checked for positivity
 * (TSVGP_ERR_NONPOSITIVE_VARIANCE).  Not collective.  Not built for the whitened sibling (TSVGP_ERR_INVALID).  The N x N
 * buffers must fit in free device memory, else TSVGP_ERR_INVALID (message: bytes needed) before anything is allocated.     */
TSVGP_API int tsvgp_predict_f_full_cov(tsvgp_ctx* ctx, const double* Xnew, int64_t N, int D, const double* mean_X,
                                       double* mean_out, double* cov_out);
/* GPModel.predict_f_samples: samples_out [S, N, L].  full_cov = 1: mean + chol(Sigma_l + 1e-6 I) eps (a failed Cholesky is
 * TSVGP_ERR_NOT_POSITIVE_DEFINITE, tsvgp_last_info() = 1-based query point); 0: mean + sqrt(var) eps (also for the whitened
 * sibling).  eps [S, N, L] (HOST or DEVICE) or NULL = Philox draws keyed by option "sample_seed", a new draw per call.
 * Not collective; the sites and cached factors are left unchanged.                                                       */
TSVGP_API int tsvgp_predict_f_samples(tsvgp_ctx* ctx, const double* Xnew, int64_t N, int D, const double* mean_X, int S,
                                      int full_cov, const double* eps, double* samples_out);
/* t_SVGP_white.predict_f_extra_data (tsvgp_white.py:134-158; whitened sibling only): predictions at Xnew after conditioning the
 * current sites on the RESIDENT minibatch (the "extra data") without changing them; jitter is the reference's argument
 * (default gpflow default_jitter = 1e-6; its test passes 0).  mean_out, var_out [N, L].  Softmax: the conditioning evaluates
 * the likelihood once, with one Monte-Carlo draw (see tsvgp_set_mc_epsilon).                                              */
TSVGP_API int tsvgp_predict_f_extra_data(tsvgp_ctx* ctx, const double* Xnew, int64_t N, int D, const double* mean_X, double jitter,
                                         double* mean_out, double* var_out);
/* t_SVGP.get_mean_chol_cov_inducing_posterior (tsvgp.py:202-212): m [M, L], chol_S [L, M, M]                           */
TSVGP_API int tsvgp_posterior(tsvgp_ctx* ctx, double* m, double* chol_S);

/* ---- multi-GPU: one context per rank, rows of the minibatch sharded over ranks, one all-reduce of the statistics ---- */
TSVGP_API int tsvgp_comm_unique_id(void* id_out_128_bytes);                                   /* ncclGetUniqueId                     */
TSVGP_API int tsvgp_comm_init(tsvgp_ctx* ctx, int world_size, int rank, const void* id_128_bytes);
TSVGP_API int tsvgp_comm_size(const tsvgp_ctx* ctx);
/* The CUDA device of the context and its main stream (a cudaStream_t): a DLPack producer is handed this stream
 * (`tensor.__dlpack__(stream=...)`) so that its pending writes are ordered before the library's first read.            */
TSVGP_API int tsvgp_device(const tsvgp_ctx* ctx);
TSVGP_API void* tsvgp_stream(const tsvgp_ctx* ctx);

/* ---- measurement ------------------------------------------------------------------------------------------------------ */
/* CUDA-event durations (ms) of the last natgrad_step, on the context's stream.  out[0..n):
 *  0 total, 1 prepare (posterior factors), 2 streaming pass, 3 all-reduce, 4 dense update, 5 number of slabs,
 *  6 kernels launched by the step, 7 route used (1 fused, 2 whitened, 3 exact), 8 estimated cond(Kuu + jitter I) (0 if not probed),
 *  9 chain split ("split_chains"): 0 = both preparation chains ran here, 1 / 2 = this rank built the posterior factors / the
 *    Kuu + jitter I chain and received the other, 3 = it received both                                                           */
TSVGP_API int tsvgp_get_timings(tsvgp_ctx* ctx, double* out, int n);
TSVGP_API int tsvgp_sync(tsvgp_ctx* ctx);
/* With option "profile" = 1 the streaming pass runs on one stream and brackets every kernel with CUDA events.  After a
 * natgrad_step, out[2*k] = summed duration (ms) and out[2*k+1] = launch count of kernel class k:
 *  0 Kuf slab, 1 variance product (triangular DMMA GEMM + column norms; not run by a Gaussian step: (0, 0)), 2 point
 *  statistics, 3 whitening GEMM, 4 weighted SYRK (DMMA), 5 Kuf g                                                        */
TSVGP_API int tsvgp_get_kernel_profile(tsvgp_ctx* ctx, double* out, int n);
/* CUDA-event stopwatch on the context's stream (every call's work, host<->device copies included, is ordered on it)   */
TSVGP_API int tsvgp_timer_start(tsvgp_ctx* ctx);
TSVGP_API int tsvgp_timer_stop(tsvgp_ctx* ctx, double* ms);      /* records, synchronises, returns the elapsed time      */
/* device staging without a tensor library: plain cudaMalloc / cudaFree / cudaMemcpy(Default) on the context's device   */
TSVGP_API void* tsvgp_device_alloc(tsvgp_ctx* ctx, size_t bytes);
TSVGP_API void tsvgp_device_free(tsvgp_ctx* ctx, void* p);
TSVGP_API int tsvgp_memcpy(tsvgp_ctx* ctx, void* dst, const void* src, size_t bytes);
TSVGP_API void* tsvgp_pinned_alloc(size_t bytes);                                             /* cudaHostAlloc, for staging buffers  */
TSVGP_API void tsvgp_pinned_free(void* p);

/* ---- DLPack hand-over ---------------------------------------------------------------------------------------------- */
typedef struct {
    void* data;          /* dl_tensor.data + byte_offset                       */
    int64_t shape[3];    /* unused trailing dims = 1                           */
    int ndim;
    int device_type;     /* 1 = kDLCPU, 2 = kDLCUDA, 3 = kDLCUDAHost, 13 = kDLCUDAManaged */
    int device_id;
} tsvgp_view;
/* Validates a `DLManagedTensor*` (float64, <= 3-D, compact row-major) taken from a "dltensor" capsule and describes it.
 * The capsule is only borrowed: the library neither renames it nor calls its deleter.                                   */
TSVGP_API int tsvgp_dlpack_view(const void* dl_managed_tensor, tsvgp_view* out);

#ifdef __cplusplus
}
#endif
#endif /* TSVGP_H */
