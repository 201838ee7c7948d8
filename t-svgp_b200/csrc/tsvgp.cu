// libtsvgp.so — C ABI (include/tsvgp.h) and step orchestration of the t-SVGP natural-gradient path on one B200.
//
// What one natgrad_step does on the device (reference: src/models/tsvgp.py:234-304, src/util.py:349-391; algebra in
// DESIGN.md):
//   prepare : K = k(Z,Z), K6 = K + 1e-6 I; W = I + L2^T K6 L2; reverse Cholesky W = Uw Uw^T; T = L2 Uw^-T (lower);
//             alpha = lambda_1 - T T^T K6 lambda_1 (= K6^-1 m_q); mZ = K alpha                      [M x M work]
//   stream  : per slab of `chunk` points, on two alternating streams:
//               Kuf slab + partial means  ->  |T^T k_n|^2 by a triangular DMMA product with a column-norm epilogue
//               -> per-point likelihood statistics (g_n, h_n, ve_n)  ->  B += Kuf diag(h) Kfu (DMMA SYRK), b += Kuf g
//             (Gaussian likelihood: g_n, h_n do not read v_n, so there is no |T^T k_n|^2; the ELBO takes sum_n |T^T k_n|^2 =
//              tr(T^T B T) / h from the statistics instead, see variance_term_from_stats)
//   reduce  : one all-reduce (NCCL) of [B | b | sum ve | flag] when the minibatch is sharded over ranks
//   update  : G2 = K9^-1 B K9^-1, G1 = K9^-1 b, lambda_1, P = (1-lr) L2 L2^T - 2 lr s G2 + jitter I, L2 = -chol(P)
// There is no CPU path: every entry point that computes needs a CUDA device.
#include "../../include/tsvgp.h"
#include "common.cuh"
#include "dense.cuh"
#include "gemm.cuh"
#include "int8_gram.cuh"
#include "kernels.cuh"
#include "nccl_dyn.h"
#include <nvtx3/nvToolsExt.h>   // header-only; ranges let ncu select the kernels of one phase (--nvtx --nvtx-include "tsvgp_stream/")

#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <string>
#include <utility>
#include <vector>
#include <mutex>
#include <thread>

namespace tsvgp {
thread_local long g_launches = 0;
int g_debug_sync = 0;
int g_pdl = 1;
thread_local int g_pdl_suspended = 0;
}
using namespace tsvgp;

namespace {

thread_local std::string g_create_error;
constexpr double GPFLOW_DEFAULT_JITTER = 1e-6;   // gpflow.config.default_jitter() (GPflow 2.2.1), tsvgp.py:209-211

inline long round_up(long v, long m) { return (v + m - 1) / m * m; }
constexpr int MAXS = 4;   // slab streams (option "streams"; default 2)

struct Pool {
    std::vector<void*> ptrs;
    cudaError_t last = cudaSuccess;
    double* get(size_t n_doubles) {
        void* p = nullptr;
        last = cudaMalloc(&p, (n_doubles ? n_doubles : 1) * sizeof(double));
        if (last != cudaSuccess) return nullptr;
        ptrs.push_back(p);
        return (double*)p;
    }
    void release() {
        for (void* p : ptrs) cudaFree(p);
        ptrs.clear();
    }
};

enum { MODE_STATS = 0, MODE_ELBO = 1, MODE_PREDICT = 2, MODE_GRAD = 3 };   // MODE_GRAD: statistics with unclipped h + dELBO/dKuf sums
enum { INFO_W = 0, INFO_K9 = 1, INFO_P = 2, INFO_S = 3, N_INFO = 4 };
enum { EV_T0 = 0, EV_PREP, EV_STREAM, EV_REDUCE, EV_DENSE, N_EV };
// device scalars
enum { SC_LOGDIAG_W = 0, SC_M_ALPHA, SC_TR_QK, SC_PK0, SC_PK1, SC_PI0, SC_PI1, SC_G_K, SC_TR_QB, SC_A_B, SC_TR_PBP, N_SCAL = 12 };
enum { ROUTE_AUTO = 0, ROUTE_FUSED = 1, ROUTE_WHITENED = 2, ROUTE_EXACT = 3 };

}  // namespace

struct tsvgp_ctx {
    int dev = 0;
    cudaStream_t s_main = nullptr, s_pp[MAXS] = {}, s_side = nullptr;
    cudaEvent_t ev_fork = nullptr, ev_join[MAXS] = {}, ev[N_EV] = {}, ev_kuu = nullptr, ev_side = nullptr;
    std::string err;
    std::mutex err_mu;            // the side-stream issue thread may report an error too
    int last_info = 0;

    // options
    long chunk_opt = 0;        // 0 = automatic
    int n_streams = 2;
    int dist_min_m = 4096;     // distribute the dense M x M products over the ranks from this (padded) M upwards
    int shard_min_m = 2048;    // from this (padded) M upwards the statistics are reduce-SCATTERED by tile rows and the two products of
    int split_chains = 0;      // 1: rank 0 builds the posterior factors, rank 1 the K9 chain, both broadcast their results (see chain_split_active)
                               // G2 = K9^-1 B K9^-1 run on each rank's rows only, assembled by two all-gathers (sharded_update)
    int async_issue = 1;       // small M: enqueue the K9 chain from a helper host thread while this thread enqueues the posterior chain
    int fuse_b = 1;            // accumulate b += Kuf g inside the SYRK kernel instead of a separate mat-vec pass over the slab
    int spread_b = 0;          // 1: ... shared by all tiles of a tile row (private slots) instead of carried by the first tile column alone.
                               // Measured (M = 2048, 262 144 rows): the SYRK launch alone 1.087 -> 1.076 ms, but the step 74.55 -> 74.63 ms
                               // (two slab streams already hide the longer first-column tiles; the extra zeroing and summing are not free)
    int balance = 1;           // split the SYRK's contraction in two pieces so that every SM gets equal work
    int cache_factors = 1;     // keep chol(K9) and the posterior factors between calls while their inputs are unchanged
    int route_opt = ROUTE_AUTO;     // statistics route: fused (B = Kuf H Kfu, then K9^-1 B K9^-1) or whitened (C9^-1 Kuf first)
    double route_cond_max = 1e4;    // auto: fused while the estimated cond(Kuu + jitter I) is below this (measured fused error
                                    // <= 4e-18 cond^2, tests/test_gpu_parity.py arbiter test: 4e-10 at the threshold)
    double route_exact_min = 1e8;   // auto: above this estimate even the two-sided product C9^-T Bw C9^-1 of the whitened route loses
                                    // the positive definiteness the reference gets from forming A = K9^-1 Kuf first and then the
                                    // Gram product A^T diag(h) A (tsvgp.py:271-281): take that order literally (4 M^2 flops per point)
    int route = ROUTE_FUSED;        // route of the current / last step
    double cond_est = 0.0;
    // The conditioning probe needs chol(K9), i.e. the whole K9 chain, before the statistics route of the pass can be chosen.  When an
    // estimate from an earlier step of this context says "fused" (the route that needs nothing of K9 inside the pass), the step
    // SPECULATES: the K9 chain runs on the side stream underneath the streaming pass instead of in front of it, the probe is read
    // after the pass, and the pass is repeated with the right route in the (rare) case the estimate crossed the threshold.
    double cond_hint = 0.0;
    bool cond_hint_valid = false;
    int speculate = 1;
    int k9_defer = 0;   // measured slower (M = 2048, 131072 rows: 41.1 vs 39.9 ms): under the pass every chain kernel waits for an SM slot
    // Gaussian likelihood, fused route: h_n is a constant, so Kuf and the SYRK of a slab do not depend on the posterior.  The first
    // slab of every slab stream is enqueued BEFORE the posterior chain (latency-bound, SMs mostly idle) and fills the idle SMs.
    int early_slabs = 1;
    int n_early = 0;
    cudaEvent_t ev_post = nullptr;
    cudaEvent_t ev_xpost = nullptr;   // posterior exchange of the chain split complete (main stream)
    cudaEvent_t ev_early0 = nullptr;  // first early slab of slab stream 0 complete
    cudaEvent_t ev_mid = nullptr;     // second slab of slab stream 0 complete (or the last one of a short pass)
    bool mark_mid = false;            // stream_pass records ev_mid
    CholAux la_main, la_side;   // look-ahead helper streams of the Cholesky factorisations on the main / side stream (dense.cuh)
    // Entry points that every rank calls together (natgrad_step, elbo, elbo_grad, predict_f_extra_data) may distribute the dense
    // M x M products over the ranks; predict_f / prior_kl / posterior may be called by one rank alone and must not hide a collective.
    bool collective_ok = false;
    bool post_collective = false;   // the cached posterior factors were built by a collective call (distributed products)

    // kernel / likelihood
    int kern_kind = -1;
    double kern_var = 1.0;
    std::vector<double> ls_host;
    LikSpec lik;
    GHTable gh;
    bool lik_set = false;
    // Separate kernels (tsvgp_set_kernels; gpflow SeparateIndependent): one kernel per latent.  Each latent owns its kernel-
    // dependent state (lengthscales, scaled inducing inputs, K, K6, the K9 chain), and select_latent() points the working views
    // (kern_kind, kern_var, ls_dev, ZsT, Zs, z2, K, K6, C9, C9inv, K9inv and the Kuf slabs) at latent l's copies, so every
    // single-latent routine runs unchanged.  Latent 0 uses the shared mode's buffers (`base`), the others live in `pks`; the
    // scaled resident data XsT/x2 hold L copies back to back.  In shared mode none of this is allocated or touched.
    struct KernelState {
        int kind = -1;
        double var = 1.0;
        std::vector<double> ls;
        double *ls_dev = nullptr, *ZsT = nullptr, *Zs = nullptr, *z2 = nullptr, *K = nullptr, *K6 = nullptr, *C9 = nullptr,
               *C9inv = nullptr, *K9inv = nullptr;
    };
    bool sep = false;
    std::vector<KernelState> lk;   // [L] in separate mode
    KernelState base;              // buffers of alloc_m_state
    Pool pks;
    int ks_Mp = 0;                 // Mp the per-latent buffers were allocated for (0: none)

    // Latent GPs sharing the kernel and the inducing inputs (num_latent_gps = L, reference tsvgp.py:276-281): one site pair, one set of
    // posterior factors and one statistics accumulator per latent, stored as [L] contiguous copies.  The per-latent pointers below
    // (lam1, L2, T, alpha, mZ, mq, scal, stats, stats2 and the per-slab mu_part / q_part / gbuf / hbuf / ve_blocks) always VIEW the
    // latent selected by select_latent(); everything kernel-dependent (K, K6, the K9 chain, the Kuf slabs) exists once.
    int L = 1, cur = 0;
    double *lam1_all = nullptr, *L2_all = nullptr, *T_all = nullptr, *alpha_all = nullptr, *mZ_all = nullptr, *mq_all = nullptr, *scal_all = nullptr;
    double *stats_all[MAXS] = {}, *stats2_all[MAXS] = {};
    double *mu_part_all[MAXS] = {}, *q_part_all[MAXS] = {}, *gbuf_all[MAXS] = {}, *hbuf_all[MAXS] = {}, *ve_all = nullptr;
    double* Yt = nullptr;      // Y [N, L] transposed to [L][n_pad] (L > 1)
    long yt_cap = 0;
    int y_cols = 1;            // columns of the resident Y: L for independent likelihood terms, 1 (class labels) for Softmax
    Pool pyt, pmc;
    double* mc_eps = nullptr;  // explicit Monte-Carlo draws [S][mc_eps_n][L] of the Softmax likelihood (tsvgp_set_mc_epsilon) or null
    long mc_eps_n = 0;
    unsigned long long mc_seed = 0x5eed5eedULL, mc_draw = 0;   // Philox key and per-call draw counter otherwise
    unsigned long long sample_seed = 0x5a3b1e5eULL, sample_draw = 0;   // the same for predict_f_samples (option "sample_seed")
    // inducing points and M x M state
    int M = 0, Mp = 0, D = 0;
    Pool pm;
    double *Zraw = nullptr, *ZsT = nullptr, *Zs = nullptr, *z2 = nullptr, *ls_dev = nullptr, *meanZ_off = nullptr;
    bool has_meanZ = false;
    double *K = nullptr, *K6 = nullptr, *L2 = nullptr, *lam1 = nullptr;
    double *Wm = nullptr, *Wf = nullptr, *V = nullptr, *T = nullptr, *X1 = nullptr, *X2 = nullptr, *C9 = nullptr, *C9inv = nullptr;
    double *G2 = nullptr, *P = nullptr, *tmp = nullptr, *dinv = nullptr, *K9inv = nullptr;
    double *stats[MAXS] = {};   // [B (Mp*Mp) | b (Mp) | tail (4)] per ping-pong stream
    double *stats2[MAXS] = {};  // second B accumulator per stream: the split-off k piece of the balanced SYRK
    double *alpha = nullptr, *mZ = nullptr, *mq = nullptr, *v1 = nullptr, *v2 = nullptr, *v3 = nullptr, *gwork = nullptr;
    double *gws = nullptr, *gws2 = nullptr;   // split-K partial-tile workspaces of the M x M products (main / side stream)
    size_t gws_doubles = 0;
    double *scal = nullptr, *red = nullptr;   // device scalars; [128] scratch of the two-stage reductions (per context)
    double jit6 = GPFLOW_DEFAULT_JITTER;   // jitter of K6 (gpflow default_jitter; predict_f_extra_data passes its own)
    int white = 0;             // 1: the whitened sibling t_SVGP_white (reference src/models/tsvgp_white.py): L2 holds the full Lambda_2
    double *C6 = nullptr, *C6inv = nullptr;   // chol(K6) and its inverse (whitened sibling)
    bool c6_valid = false, wpost_valid = false, wkl_valid = false;
    double *zaug = nullptr, *fuu = nullptr, *origin = nullptr;   // M-step: [zs | 1 | zs^2] and the Kuu counterpart of F
    double *tmp2 = nullptr, *dinv2 = nullptr, *pv1 = nullptr, *pv2 = nullptr, *gwork2 = nullptr, *scal2 = nullptr;   // side-stream workspace (K9 factor)
    bool k9inv_valid = false;  // K9inv = C9inv^T C9inv formed (on the main stream, on first use by the fused route)
    bool k9_pending = false;   // K9 work enqueued on the side stream, probe not read yet
    int* info = nullptr;    // [N_INFO]
    int* flags = nullptr;   // [2]
    bool sites_set = false, kuu_valid = false, post_valid = false, kl_valid = false, k9_valid = false;
    double k9_jitter = 0.0;
    double kl_host = 0.0;

    // data (this rank's rows)
    Pool pd;
    long N = 0, n_pad = 0;
    int dataD = 0;
    const double *X = nullptr, *Y = nullptr, *meanX = nullptr;
    double *Xown = nullptr, *Yown = nullptr, *meanXown = nullptr;
    // prefetch: the next minibatch is copied into a second set of buffers on a copy stream while the current step computes
    Pool ps;
    double *Xst = nullptr, *Yst = nullptr, *meanXst = nullptr;
    long st_cap_x = 0, st_cap_n = 0, st_N = 0;
    int st_D = 0;
    bool st_has_mean = false, st_ready = false;
    cudaStream_t s_copy = nullptr;
    cudaEvent_t ev_copy = nullptr;
    long cap_x = 0, cap_n = 0;
    int cap_yc = 1;
    double *XsT = nullptr, *x2 = nullptr;
    Pool pxs;
    long xs_cap = 0, xs_cap_n = 0;
    bool xs_valid = false;

    // slab workspace
    Pool pc;
    long chunk = 0;
    int chunk_Mp = 0;
    int chunk_route = 0;
    int slab_streams = 0;
    double *wslab[MAXS] = {};
    double *slab_all[MAXS] = {};   // [slab_lat][Mp][nc]: one Kuf slab per latent in separate mode
    int slab_lat = 1;
    double *slab[MAXS] = {}, *mu_part[MAXS] = {}, *q_part[MAXS] = {}, *q2_part[MAXS] = {}, *gbuf[MAXS] = {}, *hbuf[MAXS] = {};
    double* ve_blocks = nullptr;
    long ve_cap = 0;
    double *kpslab[MAXS] = {}, *vslab[MAXS] = {}, *uslab[MAXS] = {}, *xaug[MAXS] = {}, *fpart[MAXS] = {}, *facc[MAXS] = {};   // M-step gradient workspace
    double* aux_blocks = nullptr;
    int fsplit = 1;
    bool grad_ws = false;
    int grad_lat = 0;     // U slabs per slab stream in the gradient workspace: L for a coupled likelihood (one pass), else 1
    int waug = 128;       // columns of the augmented blocks [xs | 1 | xs^2 | 0] (xaug, zaug, facc, fuu, fpart): aug_width(D)
    double* kpart[MAXS] = {};     // split-K partial tiles of the SYRK when M is so small that its tiles cannot fill the SMs
    double* bacc[MAXS] = {};      // fused b += Kuf g shared by the tiles of a tile row: [L][2 pieces][Mp/128 tile columns][Mp] private slots
    int ksplit = 1;
    // Gaussian step, fused route: the constant-weight SYRK as an exact int8 Gram product (int8_gram.cuh) — per slab stream the
    // 16 residue planes of the slab and the residues of the lower tiles; allocated for a Gaussian model (i8_alloc)
    int8_t* i8_planes[MAXS] = {};
    uint8_t* i8_tiles[MAXS] = {};
    bool i8_alloc = false;

    // multi-GPU
    NcclComm comm = nullptr;
    int world = 1, rank = 0;

    double timings[16] = {};
    double grad_scale = 1.0;
    int profile = 0;
    std::vector<cudaEvent_t> pev;   // profile-mode event pool
    double kprof[12] = {};
    cudaEvent_t ev_sw[2] = {nullptr, nullptr};
};

namespace {

#define FAIL(code, ...)                                   \
    do {                                                  \
        char b_[512];                                     \
        snprintf(b_, sizeof b_, __VA_ARGS__);             \
        {                                                 \
            std::lock_guard<std::mutex> g_(c->err_mu);    \
            c->err = b_;                                  \
        }                                                 \
        return (code);                                    \
    } while (0)
#define CU(x)                                                                                            \
    do {                                                                                                 \
        cudaError_t e_ = (x);                                                                            \
        if (e_ != cudaSuccess) FAIL(TSVGP_ERR_CUDA, "%s: %s (%s:%d)", #x, cudaGetErrorString(e_), __FILE__, __LINE__); \
    } while (0)
#define LA(x)                                                                                                      \
    do {                                                                                                           \
        int e_ = (x);                                                                                              \
        if (e_ > 0) FAIL(TSVGP_ERR_CUDA, "%s: %s (%s:%d)", #x, cudaGetErrorString((cudaError_t)e_), __FILE__, __LINE__); \
        if (e_ < 0) FAIL(TSVGP_ERR_INVALID, "%s: unsupported launch configuration (%s:%d)", #x, __FILE__, __LINE__); \
    } while (0)
#define OK(x)                    \
    do {                         \
        int r_ = (x);            \
        if (r_ != TSVGP_OK) return r_; \
    } while (0)
#define NEED(p)                                                               \
    do {                                                                      \
        if (!(p)) FAIL(TSVGP_ERR_CUDA, "device allocation failed (%s:%d)", __FILE__, __LINE__); \
    } while (0)

int all_reduce(tsvgp_ctx* c, double* buf, size_t count);
int alloc_separate(tsvgp_ctx* c);
int ensure_posterior_white(tsvgp_ctx* c);
int posterior_one(tsvgp_ctx* c);
int ensure_kl_terms_white(tsvgp_ctx* c);
int dense_update_white(tsvgp_ctx* c, double lr, double scale);
int dense_update(tsvgp_ctx* c, double lr, double jitter, double scale, bool only_G);
double kl_white_from_scalars(const tsvgp_ctx* c, const double* sc);
bool dist_active(const tsvgp_ctx* c);
int dense_gemm(tsvgp_ctx* c, GemmP p, cudaStream_t s);
int mm_gemm(tsvgp_ctx* c, const GemmP& p, cudaStream_t s);

bool is_device_ptr(const void* p) {
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) {
        cudaGetLastError();
        return false;
    }
    return a.type == cudaMemoryTypeDevice || a.type == cudaMemoryTypeManaged;
}

// ---- latent views ---------------------------------------------------------------------------------------------------
void view_kernel_buffers(tsvgp_ctx* c, const tsvgp_ctx::KernelState& k) {
    c->ls_dev = k.ls_dev; c->ZsT = k.ZsT; c->Zs = k.Zs; c->z2 = k.z2;
    c->K = k.K; c->K6 = k.K6; c->C9 = k.C9; c->C9inv = k.C9inv; c->K9inv = k.K9inv;
}

void select_latent(tsvgp_ctx* c, int l) {
    const size_t mm = (size_t)c->Mp * c->Mp, mp = c->Mp;
    c->cur = l;
    if (c->sep && c->ks_Mp == c->Mp) {
        const tsvgp_ctx::KernelState& k = c->lk[l];
        c->kern_kind = k.kind; c->kern_var = k.var;
        view_kernel_buffers(c, k);
    }
    c->lam1 = c->lam1_all + l * mp; c->L2 = c->L2_all + l * mm; c->T = c->T_all + l * mm;
    c->alpha = c->alpha_all + l * mp; c->mZ = c->mZ_all + l * mp; c->mq = c->mq_all + l * mp; c->scal = c->scal_all + (size_t)l * N_SCAL;
    for (int s = 0; s < MAXS; ++s) {
        c->stats[s] = c->stats_all[s] + l * (mm + mp + 4);
        c->stats2[s] = c->stats2_all[s] + l * (mm + mp);
    }
    if (c->chunk > 0 && c->chunk_Mp == c->Mp) {
        const size_t nc = c->chunk;
        for (int s = 0; s < c->slab_streams; ++s) {
            c->mu_part[s] = c->mu_part_all[s] + l * (size_t)(c->Mp / 64) * nc;
            c->q_part[s] = c->q_part_all[s] + l * (size_t)(c->Mp / 128) * nc;
            c->gbuf[s] = c->gbuf_all[s] + l * nc;
            c->hbuf[s] = c->hbuf_all[s] + l * nc;
            if (c->slab_lat > 1) c->slab[s] = c->slab_all[s] + l * (size_t)c->Mp * nc;
        }
        c->ve_blocks = c->ve_all + (size_t)l * c->ve_cap;
    }
}

// ---- M-dependent state ----------------------------------------------------------------------------------------------
int alloc_m_state(tsvgp_ctx* c, int M, int D) {
    c->pm.release();
    c->M = M; c->D = D; c->Mp = (int)round_up(M, TSVGP_TILE);
    const size_t mm = (size_t)c->Mp * c->Mp, mp = c->Mp;
    Pool& p = c->pm;
    NEED(c->Zraw = p.get((size_t)M * D)); NEED(c->ZsT = p.get((size_t)D * mp)); NEED(c->Zs = p.get(mp * D));
    NEED(c->z2 = p.get(mp)); NEED(c->ls_dev = p.get(D)); NEED(c->meanZ_off = p.get(mp));
    const size_t nl = (size_t)c->L;
    NEED(c->K = p.get(mm)); NEED(c->K6 = p.get(mm)); NEED(c->L2_all = p.get(nl * mm)); NEED(c->lam1_all = p.get(nl * mp));
    NEED(c->Wm = p.get(mm)); NEED(c->Wf = p.get(mm)); NEED(c->V = p.get(mm)); NEED(c->T_all = p.get(nl * mm));
    NEED(c->X1 = p.get(mm)); NEED(c->X2 = p.get(mm)); NEED(c->C9 = p.get(mm)); NEED(c->C9inv = p.get(mm));
    NEED(c->G2 = p.get(mm)); NEED(c->P = p.get(mm)); NEED(c->K9inv = p.get(mm)); NEED(c->tmp = p.get((size_t)((c->Mp / 128 + 1) / 2) * 128 * mp));   // trtri_lower: ceil(nblk/2) block rows
    NEED(c->dinv = p.get((size_t)(c->Mp / 128) * 128 * 128));
    CU(cudaMemsetAsync(c->dinv, 0, sizeof(double) * (size_t)(c->Mp / 128) * 128 * 128, c->s_main));   // contract of diag_potrf_inv_launch
    for (int s = 0; s < MAXS; ++s) { NEED(c->stats_all[s] = p.get(nl * (mm + mp + 4))); NEED(c->stats2_all[s] = p.get(nl * (mm + mp))); }
    NEED(c->alpha_all = p.get(nl * mp)); NEED(c->mZ_all = p.get(nl * mp)); NEED(c->mq_all = p.get(nl * mp)); NEED(c->v1 = p.get(mp)); NEED(c->v2 = p.get(mp));
    NEED(c->v3 = p.get(mp)); NEED(c->gwork = p.get((size_t)(c->Mp / 64 + 1) * mp)); NEED(c->scal_all = p.get(nl * N_SCAL)); NEED(c->red = p.get(128));
    NEED(c->info = (int*)p.get(N_INFO)); NEED(c->flags = (int*)p.get(2));
    c->gws_doubles = (size_t)4 << 20;   // 32 MB per stream: up to 16 partial images of a 512 x 512 product, 4 of a 1024 x 1024 one
    NEED(c->gws = p.get(c->gws_doubles)); NEED(c->gws2 = p.get(c->gws_doubles));
    // (on the context's own stream: it is non-blocking, a legacy-stream memset would not be ordered with it)
    CU(cudaMemsetAsync(c->gws + c->gws_doubles - GEMM_WS_COUNTER_DOUBLES, 0, sizeof(double) * GEMM_WS_COUNTER_DOUBLES, c->s_main));    // tile counters
    CU(cudaMemsetAsync(c->gws2 + c->gws_doubles - GEMM_WS_COUNTER_DOUBLES, 0, sizeof(double) * GEMM_WS_COUNTER_DOUBLES, c->s_main));
    c->waug = aug_width(D);
    NEED(c->zaug = p.get(mp * c->waug)); NEED(c->fuu = p.get(mp * c->waug)); NEED(c->origin = p.get(D));
    NEED(c->C6 = p.get(mm)); NEED(c->C6inv = p.get(mm));
    c->c6_valid = c->wpost_valid = c->wkl_valid = false;
    NEED(c->tmp2 = p.get((size_t)((c->Mp / 128 + 1) / 2) * 128 * mp)); NEED(c->dinv2 = p.get((size_t)(c->Mp / 128) * 128 * 128));
    CU(cudaMemsetAsync(c->dinv2, 0, sizeof(double) * (size_t)(c->Mp / 128) * 128 * 128, c->s_main));
    CU(cudaStreamSynchronize(c->s_main));   // the side and helper streams use these buffers too
    NEED(c->pv1 = p.get(mp)); NEED(c->pv2 = p.get(mp)); NEED(c->gwork2 = p.get((size_t)(c->Mp / 64 + 1) * mp)); NEED(c->scal2 = p.get(nl * N_SCAL));
    c->sites_set = c->kuu_valid = c->post_valid = c->kl_valid = c->k9_valid = c->c6_valid = c->wpost_valid = c->wkl_valid = false;
    c->chunk = 0;   // slab workspace depends on Mp
    c->base.ls_dev = c->ls_dev; c->base.ZsT = c->ZsT; c->base.Zs = c->Zs; c->base.z2 = c->z2;
    c->base.K = c->K; c->base.K6 = c->K6; c->base.C9 = c->C9; c->base.C9inv = c->C9inv; c->base.K9inv = c->K9inv;
    c->ks_Mp = 0;
    if (c->sep) OK(alloc_separate(c));
    select_latent(c, 0);
    return TSVGP_OK;
}

// the per-latent kernel buffers of separate mode: latent 0 takes the shared mode's, latents 1.. get their own
int alloc_separate(tsvgp_ctx* c) {
    CU(cudaDeviceSynchronize());
    c->pks.release();
    const size_t mm = (size_t)c->Mp * c->Mp, mp = c->Mp;
    for (int l = 0; l < c->L; ++l) {
        tsvgp_ctx::KernelState& k = c->lk[l];
        if (l == 0) {
            k.ls_dev = c->base.ls_dev; k.ZsT = c->base.ZsT; k.Zs = c->base.Zs; k.z2 = c->base.z2;
            k.K = c->base.K; k.K6 = c->base.K6; k.C9 = c->base.C9; k.C9inv = c->base.C9inv; k.K9inv = c->base.K9inv;
            continue;
        }
        Pool& p = c->pks;
        NEED(k.ls_dev = p.get(c->D)); NEED(k.ZsT = p.get((size_t)c->D * mp)); NEED(k.Zs = p.get(mp * c->D)); NEED(k.z2 = p.get(mp));
        NEED(k.K = p.get(mm)); NEED(k.K6 = p.get(mm)); NEED(k.C9 = p.get(mm)); NEED(k.C9inv = p.get(mm)); NEED(k.K9inv = p.get(mm));
    }
    c->ks_Mp = c->Mp;
    c->kuu_valid = c->post_valid = c->kl_valid = c->k9_valid = false;
    return TSVGP_OK;
}

// back to one kernel shared by every latent (tsvgp_set_kernel, tsvgp_set_num_latent)
int drop_separate(tsvgp_ctx* c) {
    if (!c->sep) return TSVGP_OK;
    CU(cudaDeviceSynchronize());
    view_kernel_buffers(c, c->base);
    c->sep = false;
    c->lk.clear();
    c->pks.release();
    c->ks_Mp = 0;
    c->kuu_valid = c->post_valid = c->kl_valid = c->k9_valid = c->xs_valid = false;
    return TSVGP_OK;
}

int default_sites(tsvgp_ctx* c) {   // tsvgp.py:174-180 : lambda_1 = 0, lambda_2_sqrt = -1e-10 I  (every latent)
    CU(cudaMemsetAsync(c->lam1_all, 0, sizeof(double) * c->Mp * c->L, c->s_main));
    // tsvgp.py:174-180 : lambda_2_sqrt = -1e-10 I ;  tsvgp_white.py:79-85 : lambda_2 = +1e-10 I
    for (int l = 0; l < c->L; ++l)
        LA(set_scaled_identity_launch(c->L2_all + (size_t)l * c->Mp * c->Mp, c->Mp, c->M, c->Mp, c->white ? 1e-10 : -1e-10, 0.0, c->s_main));
    c->sites_set = true;
    c->post_valid = c->kl_valid = c->wpost_valid = c->wkl_valid = false;
    return TSVGP_OK;
}

int upload_lengthscales(tsvgp_ctx* c, const std::vector<double>& ls_host) {
    if (c->kern_kind < 0) FAIL(TSVGP_ERR_STATE, "kernel not set (tsvgp_set_kernel)");
    if (c->D <= 0) FAIL(TSVGP_ERR_STATE, "inducing points not set (tsvgp_set_inducing)");
    if (ls_host.size() != 1 && (int)ls_host.size() != c->D)
        FAIL(TSVGP_ERR_INVALID, "lengthscales has %zu entries, expected 1 or D=%d", ls_host.size(), c->D);
    std::vector<double> ls(c->D);
    for (int d = 0; d < c->D; ++d) ls[d] = ls_host.size() == 1 ? ls_host[0] : ls_host[d];
    CU(cudaMemcpyAsync(c->ls_dev, ls.data(), sizeof(double) * c->D, cudaMemcpyHostToDevice, c->s_main));
    CU(cudaStreamSynchronize(c->s_main));   // `ls` is a stack temporary
    return TSVGP_OK;
}

// K = k(Z,Z) (identity on the padding block), K6 = K + default_jitter I            tsvgp.py:209-211, :268
int kuu_one(tsvgp_ctx* c, const std::vector<double>& ls_host) {   // the selected latent's kernel (shared mode: the kernel)
    OK(upload_lengthscales(c, ls_host));
    cudaStream_t s = c->s_main;
    LA(scale_points_launch(c->Zraw, c->M, c->D, c->ls_dev, c->ZsT, c->Mp, c->z2, c->Mp, s));
    LA(unpack_rows_launch(c->ZsT, c->Mp, c->Mp, c->D, c->Zs, s));
    LA(kuf_launch(c->kern_kind, c->kern_var, c->ZsT, c->Mp, c->z2, 0, c->M, c->Mp, c->Zs, c->z2, c->M, c->Mp, c->D, nullptr,
                  c->K, c->Mp, nullptr, 0, 1, s));
    LA(copy_add_diag_launch(c->K, c->K6, c->Mp, c->Mp, c->jit6, s));
    return TSVGP_OK;
}

int ensure_kuu(tsvgp_ctx* c) {
    if (c->kuu_valid) return TSVGP_OK;
    if (c->M <= 0) FAIL(TSVGP_ERR_STATE, "inducing points not set (tsvgp_set_inducing)");
    if (c->sep) {   // K_l, K6_l per latent
        for (int l = 0; l < c->L; ++l) {
            select_latent(c, l);
            const int rc = kuu_one(c, c->lk[l].ls);
            if (rc != TSVGP_OK) { select_latent(c, 0); return rc; }
        }
        select_latent(c, 0);
    } else {
        OK(kuu_one(c, c->ls_host));
    }
    c->kuu_valid = true;
    c->post_valid = c->kl_valid = c->k9_valid = c->c6_valid = c->wpost_valid = c->wkl_valid = false;
    return TSVGP_OK;
}

// Posterior factors of q(u) from the dense sites (replaces posterior_from_dense_site, util.py:349-391, and the
// conditional's use of it, tsvgp.py:102-112): T, alpha, mZ, log det W.
int ensure_posterior(tsvgp_ctx* c) {
    if (c->white) return ensure_posterior_white(c);
    OK(ensure_kuu(c));
    // cached factors are reused, except that a collective call must not skip the build when this rank's cache was built by a
    // non-collective call (predict_f on one rank alone): the other ranks are about to run the distributed products' all-reduces
    if (c->post_valid && c->cache_factors && !(dist_active(c) && !c->post_collective)) return TSVGP_OK;
    if (!c->sites_set) OK(default_sites(c));
    c->post_collective = dist_active(c);
    for (int l = 0; l < c->L; ++l) {
        select_latent(c, l);
        OK(posterior_one(c));
    }
    select_latent(c, 0);
    c->post_valid = true;
    c->kl_valid = false;
    return TSVGP_OK;
}

// the factors of ONE latent (the selected one): T, alpha, m_q, mZ, log det W
int posterior_one(tsvgp_ctx* c) {
    cudaStream_t s = c->s_main;
    const int n = c->Mp;
    const long ld = c->Mp;
    {   // X1 = K6 L2
        GemmP p;
        p.A = c->K6; p.lda = ld; p.a_kc = 1;
        p.B = c->L2; p.ldb = ld; p.b_kc = 0; p.b_tri = 2;
        p.C = c->X1; p.ldc = ld; p.m = p.n = p.k = n;
        OK(dense_gemm(c, p, s));
    }
    {   // W = I + L2^T X1 (lower tiles)
        GemmP p;
        p.A = c->L2; p.lda = ld; p.a_kc = 0; p.a_tri = 2;
        p.B = c->X1; p.ldb = ld; p.b_kc = 0;
        p.C = c->Wm; p.ldc = ld; p.m = p.n = p.k = n;
        p.lower_out = 1;
        if (dist_active(c)) {
            OK(dense_gemm(c, p, s));
            LA(add_diag_launch(c->Wm, ld, n, 1.0, s));
        } else {
            LA(set_scaled_identity_launch(c->Wm, ld, n, n, 1.0, 1.0, s));
            p.beta = 1.0;
            LA(mm_gemm(c, p, s));
        }
    }
    // reverse Cholesky W = Uw Uw^T through the index flip J W J = Lr Lr^T
    LA(flip_sym_launch(c->Wm, c->Wf, ld, n, s));
    LA(chol_lower(c->Wf, ld, n, c->dinv, c->info + INFO_W, s, c->gws, c->gws_doubles, &c->la_main));
    LA(logdiag_launch(c->Wf, ld, n, c->scal + SC_LOGDIAG_W, s));
    LA(trtri_lower(c->Wf, ld, n, c->dinv, c->X2, c->tmp, s, c->gws, c->gws_doubles));
    LA(antitranspose_launch(c->X2, c->V, ld, n, s));   // V = Uw^-T (lower)
    CU(cudaMemsetAsync(c->T, 0, sizeof(double) * (size_t)n * ld, s));
    {   // T = L2 V  (lower x lower)
        GemmP p;
        p.A = c->L2; p.lda = ld; p.a_kc = 1; p.a_tri = 1;
        p.B = c->V; p.ldb = ld; p.b_kc = 0; p.b_tri = 2;
        p.C = c->T; p.ldc = ld; p.m = p.n = p.k = n;
        p.lower_out = 1;
        OK(dense_gemm(c, p, s));
    }
    // alpha = lambda_1 - T T^T K6 lambda_1
    LA(gemv_n_launch(c->K6, ld, n, n, c->lam1, 1.0, 0.0, c->v1, s));
    LA(gemv_t_launch(c->T, ld, n, n, c->v1, c->v2, c->gwork, s));
    LA(gemv_n_launch(c->T, ld, n, n, c->v2, 1.0, 0.0, c->v3, s));
    LA(vsub_launch(c->lam1, c->v3, c->alpha, n, s));
    // m_q = K6 alpha ; mZ = K alpha (+ mean_function(Z))   — predict_f(Z) of tsvgp.py:249-254 uses the un-jittered K
    LA(gemv_n_launch(c->K6, ld, n, n, c->alpha, 1.0, 0.0, c->mq, s));
    LA(gemv_n_launch(c->K, ld, n, n, c->alpha, 1.0, 0.0, c->mZ, s));
    if (c->has_meanZ) LA(vadd_inplace_launch(c->mZ, c->meanZ_off, c->M, s));
    return TSVGP_OK;
}

// KL[q(u) || p(u)] = 1/2 ( m^T alpha - tr(Q K6) + log det W )   (gauss_kl with K6; tsvgp.py:65-70). Scalars stay on the
// device until the caller's final synchronisation.
int ensure_kl_terms(tsvgp_ctx* c) {
    if (c->white) return ensure_kl_terms_white(c);
    if (c->kl_valid && c->cache_factors) return TSVGP_OK;
    cudaStream_t s = c->s_main;
    const int n = c->Mp;
    const long ld = c->Mp;
    for (int l = 0; l < c->L; ++l) {
        select_latent(c, l);
        {   // X1 = K6 T
            GemmP p;
            p.A = c->K6; p.lda = ld; p.a_kc = 1;
            p.B = c->T; p.ldb = ld; p.b_kc = 0; p.b_tri = 2;
            p.C = c->X1; p.ldc = ld; p.m = p.n = p.k = n;
            LA(mm_gemm(c, p, s));
        }
        LA(matdot_launch(c->T, c->X1, ld, n, c->scal + SC_TR_QK, c->red, s));
        LA(dot_launch(c->mq, c->alpha, n, c->scal + SC_M_ALPHA, s));
    }
    select_latent(c, 0);
    c->kl_valid = true;
    return TSVGP_OK;
}

// sc: host copy of scal_all ([L][N_SCAL]); the KL of independent q(u_l) adds up (gauss_kl sums over the latent axis)
double kl_value(const tsvgp_ctx* c, const double* sc) {
    if (c->white) return kl_white_from_scalars(c, sc);
    double kl = 0.0;
    for (int l = 0; l < c->L; ++l, sc += N_SCAL) kl += 0.5 * (sc[SC_M_ALPHA] - sc[SC_TR_QK] + 2.0 * sc[SC_LOGDIAG_W]);
    return kl;
}

constexpr int MAX_LATENT = 64;
// after a pass: [sum ve, variance flag, sum h, sum d ve / d lik] summed over the latents (the flag is the shared one)
int read_tails(tsvgp_ctx* c, double* tail /*[4]*/, double* sc /*[MAX_LATENT * N_SCAL]*/, int* info_h) {
    const size_t mm = (size_t)c->Mp * c->Mp, stride = mm + c->Mp + 4;
    double t[MAX_LATENT][4];
    cudaStream_t s = c->s_main;
    CU(cudaMemcpy2DAsync(t, 4 * sizeof(double), c->stats_all[0] + mm + c->Mp, stride * sizeof(double), 4 * sizeof(double), c->L,
                         cudaMemcpyDeviceToHost, s));
    if (sc) CU(cudaMemcpyAsync(sc, c->scal_all, sizeof(double) * N_SCAL * c->L, cudaMemcpyDeviceToHost, s));
    CU(cudaMemcpyAsync(info_h, c->info, sizeof(int) * N_INFO, cudaMemcpyDeviceToHost, s));
    CU(cudaStreamSynchronize(s));
    for (int k = 0; k < 4; ++k) tail[k] = 0.0;
    for (int l = 0; l < c->L; ++l) {
        tail[0] += t[l][0]; tail[2] += t[l][2]; tail[3] += t[l][3];
        if (t[l][1] != 0.0) tail[1] = t[l][1];
    }
    return TSVGP_OK;
}


// =====================================================================================================================
// Whitened sibling t_SVGP_white (reference src/models/tsvgp_white.py; util.py:11-88, 239-291, 394-426).  Sites (lambda_1, P) with
// P = Lambda_2 a full symmetric matrix kept in c->L2.  R = P + K6 + 1e-9 I = LR LR^T, K6 = LA LA^T:
//   mu_n = k_n^T R^-1 lambda_1 ;  v_n = k_nn - |LA^-1 k_n|^2 + |LR^-1 k_n|^2       (two triangular DMMA products per slab)
// The statistics (b, B, G1, G2) are those of the plain model; the update needs no factorisation:
//   lambda_1 <- (1-lr) lambda_1 + lr s K (G1 - 2 G2 mZ) ;  P <- (1-lr) P - 2 lr s K G2 K
// =====================================================================================================================
int ensure_posterior_white(tsvgp_ctx* c) {
    OK(ensure_kuu(c));
    if (!c->sites_set) OK(default_sites(c));
    cudaStream_t s = c->s_main;
    const int n = c->Mp;
    const long ld = n;
    if (!c->c6_valid || !c->cache_factors) {   // LA = chol(K6), LA^-1 : kernel only
        CU(cudaMemcpyAsync(c->C6, c->K6, sizeof(double) * (size_t)n * ld, cudaMemcpyDeviceToDevice, s));
        LA(chol_lower(c->C6, ld, n, c->dinv, c->info + INFO_W, s, c->gws, c->gws_doubles, &c->la_main));
        LA(trtri_lower(c->C6, ld, n, c->dinv, c->C6inv, c->tmp, s, c->gws, c->gws_doubles));
        c->c6_valid = true;
    }
    if (c->wpost_valid && c->cache_factors) return TSVGP_OK;
    for (int l = 0; l < c->L; ++l) {   // util.py:60-88 loops over the latents the same way
        select_latent(c, l);
        // R = P + K6 + 1e-9 I -> Wm = LR, T = LR^-1     (util.py:74-76, jitter default 1e-9)
        CU(cudaMemcpyAsync(c->Wm, c->K6, sizeof(double) * (size_t)n * ld, cudaMemcpyDeviceToDevice, s));
        LA(vadd_inplace_launch(c->Wm, c->L2, (long)n * ld, s));
        LA(add_diag_launch(c->Wm, ld, n, 1e-9, s));
        LA(chol_lower(c->Wm, ld, n, c->dinv, c->info + INFO_S, s, c->gws, c->gws_doubles, &c->la_main));
        LA(trtri_lower(c->Wm, ld, n, c->dinv, c->T, c->tmp, s, c->gws, c->gws_doubles));
        // alpha = R^-1 lambda_1 ; mZ = K alpha (predict_f(Z), un-jittered Kuf) ; m_q = K6 alpha
        LA(gemv_n_launch(c->T, ld, n, n, c->lam1, 1.0, 0.0, c->v1, s));
        LA(gemv_t_launch(c->T, ld, n, n, c->v1, c->alpha, c->gwork, s));
        LA(gemv_n_launch(c->K, ld, n, n, c->alpha, 1.0, 0.0, c->mZ, s));
        if (c->has_meanZ) LA(vadd_inplace_launch(c->mZ, c->meanZ_off, c->M, s));
        LA(gemv_n_launch(c->K6, ld, n, n, c->alpha, 1.0, 0.0, c->mq, s));
    }
    select_latent(c, 0);
    c->wpost_valid = true;
    c->wkl_valid = false;
    return TSVGP_OK;
}

// kl_from_precision_sites_white (util.py:239-291) with A = K6 and R0 = P + K6 (no extra jitter here): scalars
//   SC_LOGDIAG_W = sum log diag LR0 - sum log diag LA ; SC_TR_QK = |LR0^-1 LA|_F^2 ; SC_M_ALPHA = |LA^T R0^-1 lambda_1|^2
int ensure_kl_terms_white(tsvgp_ctx* c) {
    if (c->wkl_valid && c->cache_factors) return TSVGP_OK;
    cudaStream_t s = c->s_main;
    const int n = c->Mp;
    const long ld = n;
    for (int l = 0; l < c->L; ++l) {   // util.py:264-291 sums the latents' terms
        select_latent(c, l);
        CU(cudaMemcpyAsync(c->Wf, c->K6, sizeof(double) * (size_t)n * ld, cudaMemcpyDeviceToDevice, s));
        LA(vadd_inplace_launch(c->Wf, c->L2, (long)n * ld, s));
        LA(chol_lower(c->Wf, ld, n, c->dinv, c->info + INFO_P, s, c->gws, c->gws_doubles, &c->la_main));
        LA(trtri_lower(c->Wf, ld, n, c->dinv, c->V, c->tmp, s, c->gws, c->gws_doubles));       // V = LR0^-1
        LA(logdiag_launch(c->Wf, ld, n, c->scal + SC_LOGDIAG_W, s));
        LA(logdiag_launch(c->C6, ld, n, c->scal + SC_PK0, s));
        {   // X1 = LR0^-1 LA  (lower x lower)
            GemmP p;
            p.A = c->V; p.lda = ld; p.a_kc = 1; p.a_tri = 1;
            p.B = c->C6; p.ldb = ld; p.b_kc = 0; p.b_tri = 2;
            p.C = c->X1; p.ldc = ld; p.m = p.n = p.k = n;
            CU(cudaMemsetAsync(c->X1, 0, sizeof(double) * (size_t)n * ld, s));
            p.lower_out = 1;
            LA(mm_gemm(c, p, s));
        }
        LA(matdot_launch(c->X1, c->X1, ld, n, c->scal + SC_TR_QK, c->red, s));
        LA(gemv_n_launch(c->V, ld, n, n, c->lam1, 1.0, 0.0, c->v1, s));
        LA(gemv_t_launch(c->V, ld, n, n, c->v1, c->v2, c->gwork, s));   // R0^-1 lambda_1
        LA(gemv_t_launch(c->C6, ld, n, n, c->v2, c->v3, c->gwork, s));  // LA^T (.)
        LA(dot_launch(c->v3, c->v3, n, c->scal + SC_M_ALPHA, s));
    }
    select_latent(c, 0);
    c->wkl_valid = true;
    return TSVGP_OK;
}

double kl_white_from_scalars(const tsvgp_ctx* c, const double* sc) {
    double kl = 0.0;
    for (int l = 0; l < c->L; ++l, sc += N_SCAL)
        kl += 0.5 * (2.0 * (sc[SC_LOGDIAG_W] - sc[SC_PK0]) + sc[SC_TR_QK] - (double)c->Mp + sc[SC_M_ALPHA]);
    return kl;
}

// tsvgp_white.py:215-246 after the statistics are complete in stats[0]
int dense_update_white(tsvgp_ctx* c, double lr, double scale) {
    cudaStream_t s = c->s_main;
    const int n = c->Mp;
    const long ld = n;
    const size_t mm = (size_t)n * n;
    const double* bad = c->stats[0] + mm + n + 1;
    // v3 = K (G1 - 2 G2 mZ) : v2 = G1, v3 = G2 mZ were left by the shared part of the update
    LA(lincomb_launch(c->v1, 1.0, c->v2, -2.0, c->v3, n, s));          // g0 = G1 - 2 G2 mZ   (util.py:438)
    LA(gemv_n_launch(c->K, ld, n, c->M, c->v1, 1.0, 0.0, c->mq, s));   // K g0 (un-jittered Kuu, tsvgp_white.py:227,241)
    {   // X1 = K G2 ; X2 = X1 K (symmetric)
        GemmP p;
        p.A = c->K; p.lda = ld; p.a_kc = 1;
        p.B = c->G2; p.ldb = ld; p.b_kc = 0;
        p.C = c->X1; p.ldc = ld; p.m = p.n = p.k = n;
        OK(dense_gemm(c, p, s));
        GemmP q;
        q.A = c->X1; q.lda = ld; q.a_kc = 1;
        q.B = c->K; q.ldb = ld; q.b_kc = 0;
        q.C = c->X2; q.ldc = ld; q.m = q.n = q.k = n; q.lower_out = 1;
        OK(dense_gemm(c, q, s));
        LA(mirror_lower_launch(c->X2, ld, n, s));
    }
    // commit (skipped on the device after a non-positive variance or a failed factorisation)
    LA(axpby_guarded_launch(c->L2, c->X2, ld, c->M, 1.0 - lr, -2.0 * lr * scale, bad, c->info, s));
    LA(axpby_vec_guarded_launch(c->lam1, c->mq, c->M, 1.0 - lr, lr * scale, bad, c->info, s));
    return TSVGP_OK;
}

// ---- data ----------------------------------------------------------------------------------------------------------
int ensure_xs(tsvgp_ctx* c) {
    if (c->xs_valid) return TSVGP_OK;
    if (!c->X) FAIL(TSVGP_ERR_STATE, "no data resident (tsvgp_set_data)");
    OK(ensure_kuu(c));
    if (c->dataD != c->D) FAIL(TSVGP_ERR_INVALID, "X has D=%d but the inducing points have D=%d", c->dataD, c->D);
    if (c->sep) {   // one scaled copy per latent kernel, back to back: XsT [L][D][n_pad], x2 [L][n_pad]
        const long need = (long)c->L * c->D * c->n_pad, need_n = (long)c->L * c->n_pad;
        if (need > c->xs_cap || need_n > c->xs_cap_n) {
            CU(cudaStreamSynchronize(c->s_main));
            c->pxs.release();
            c->xs_cap = need; c->xs_cap_n = need_n;
            NEED(c->XsT = c->pxs.get((size_t)need)); NEED(c->x2 = c->pxs.get((size_t)need_n));
        }
        for (int l = 0; l < c->L; ++l)
            LA(scale_points_launch(c->X, c->N, c->D, c->lk[l].ls_dev, c->XsT + (size_t)l * c->D * c->n_pad, c->n_pad,
                                   c->x2 + (size_t)l * c->n_pad, c->n_pad, c->s_main));
    } else {
        LA(scale_points_launch(c->X, c->N, c->D, c->ls_dev, c->XsT, c->n_pad, c->x2, c->n_pad, c->s_main));
    }
    c->xs_valid = true;
    return TSVGP_OK;
}

long pick_chunk(const tsvgp_ctx* c) {
    long nc = c->chunk_opt;
    if (nc <= 0) nc = 16384;  // measured on B200 (profiles/): the more tiles per launch the better the SMs stay filled (per-launch fill
                              // and tail are paid half as often: 8192 -> 16384 points is -0.9 % on a cfg3 step, 12288: -0.5 %); slabs
                              // beyond the L2 cost little because both DMMA products re-read them M/128 times from L2/HBM at far
                              // below the bandwidth roof
    nc = nc / 128 * 128;
    if (nc < 128) nc = 128;
    return nc;
}

// Points per slab actually used for a pass over n_points: the allocated width `nc`, shrunk so that the slabs are equal and their
// number is a multiple of the slab streams (a 10 000-point minibatch runs as 2 x 5 120 side by side instead of 8 192 + 1 808)
long used_chunk(const tsvgp_ctx* c, long n_points, long nc, int nstr) {
    long nch = (n_points + nc - 1) / nc;
    if (c->chunk_opt > 0 || n_points <= 2048 || nstr <= 1) return nc;
    nch = round_up(nch, nstr);
    const long ncu = round_up((n_points + nch - 1) / nch, 128);
    return ncu < nc ? ncu : nc;
}

// the likelihood couples the latents (one point kernel over all of them, Y [N, 1]): Softmax, heteroskedastic Normal
inline bool coupled(const tsvgp_ctx* c) { return c->lik.kind == LIK_SOFTMAX || c->lik.kind == LIK_HETEROSKEDASTIC; }

int ensure_slabs(tsvgp_ctx* c, long n_points, bool need_grad = false) {
    const long nc = pick_chunk(c);
    const int u_lat = need_grad && coupled(c) ? c->L : 1;   // the gradient pass of a coupled likelihood keeps every latent's U
    const int nstr_used = c->profile ? 1 : (c->n_streams < 1 ? 1 : (c->n_streams > MAXS ? MAXS : c->n_streams));
    const long ncu = used_chunk(c, n_points, nc, nstr_used);
    const long nchunks = (n_points + ncu - 1) / ncu;
    const long ve_need = (nchunks + 1) * ((nc + 255) / 256);
    const bool need_w = c->route == ROUTE_WHITENED || c->route == ROUTE_EXACT;
    const int want_streams = c->profile ? 1 : (c->n_streams < 1 ? 1 : (c->n_streams > MAXS ? MAXS : c->n_streams));
    const int slab_lat = c->sep ? c->L : 1;
    const bool want_i8 = c->lik.kind == LIK_GAUSSIAN && !c->white && nc <= I8_MAX_COLS;
    if (c->chunk == nc && c->chunk_Mp == c->Mp && c->ve_cap >= ve_need && (!need_w || c->wslab[0]) && (!need_grad || (c->grad_ws && c->grad_lat >= u_lat)) &&
        c->slab_streams >= want_streams && c->slab_lat == slab_lat && c->i8_alloc == want_i8)
        return TSVGP_OK;
    CU(cudaStreamSynchronize(c->s_main));
    c->pc.release();
    for (int s = 0; s < MAXS; ++s) c->wslab[s] = nullptr;
    Pool& p = c->pc;
    const int ns = c->profile ? 1 : (c->n_streams < 1 ? 1 : (c->n_streams > MAXS ? MAXS : c->n_streams));
    c->slab_streams = ns;
    for (int s = 0; s < ns; ++s) {
        NEED(c->slab_all[s] = c->slab[s] = p.get((size_t)slab_lat * c->Mp * nc));
        if (need_w) NEED(c->wslab[s] = p.get((size_t)c->Mp * nc));
        NEED(c->mu_part_all[s] = p.get((size_t)c->L * (c->Mp / 64) * nc));
        NEED(c->q_part_all[s] = p.get((size_t)c->L * (c->Mp / 128) * nc));
        NEED(c->q2_part[s] = p.get((size_t)(c->Mp / 128) * nc));
        NEED(c->gbuf_all[s] = p.get((size_t)c->L * nc));
        NEED(c->hbuf_all[s] = p.get((size_t)c->L * nc));
    }
    {   // few output tiles (small M): split the SYRK's contraction over the idle SMs, partials reduced by a second kernel
        const int nt = c->Mp / 128, tiles = nt * (nt + 1) / 2;
        int sms = 148;
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, c->dev);
        c->ksplit = 1;
        if (tiles * 2 <= sms) {
            c->ksplit = sms / tiles;
            const int max_split = (int)(nc / 128);     // at least 8 k-tiles per piece
            if (c->ksplit > max_split) c->ksplit = max_split;
            if (c->ksplit < 2) c->ksplit = 1;
        }
        for (int s = 0; s < ns; ++s) {
            c->kpart[s] = nullptr;
            if (c->ksplit > 1) NEED(c->kpart[s] = p.get((size_t)c->ksplit * c->Mp * c->Mp));
        }
    }
    for (int s = 0; s < MAXS; ++s) { c->i8_planes[s] = nullptr; c->i8_tiles[s] = nullptr; }
    c->i8_alloc = want_i8;
    for (int s = 0; s < ns && want_i8 && c->ksplit <= 1; ++s) {   // (split-K products stay FP64)
        NEED(c->i8_planes[s] = (int8_t*)p.get((i8_plane_bytes(c->Mp, nc) + 7) / 8));
        NEED(c->i8_tiles[s] = (uint8_t*)p.get((i8_tile_bytes(c->Mp) + 7) / 8));
        LA(i8_planes_init(c->i8_planes[s], c->Mp, nc, c->s_main));
    }
    NEED(c->ve_all = p.get((size_t)c->L * ve_need));
    for (int s = 0; s < ns; ++s) NEED(c->bacc[s] = p.get((size_t)c->L * 2 * (c->Mp / 128) * c->Mp));
    c->grad_ws = false;
    c->grad_lat = 0;
    if (need_grad) {
        int sms = 148;
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, c->dev);
        c->fsplit = sms / (c->Mp / 128);
        if (c->fsplit > (int)(nc / 256)) c->fsplit = (int)(nc / 256);
        if (c->fsplit < 1) c->fsplit = 1;
        const size_t W = (size_t)c->waug;
        if (u_lat > 1) {   // U of every latent survives until the joint point kernel has run: L Mp nc doubles per slab stream
            const size_t need = ((size_t)(2 + u_lat) * c->Mp * nc + nc * W + (size_t)(c->fsplit + 1) * c->Mp * W) * ns + 2 * ve_need;
            size_t free_b = 0, total_b = 0;
            CU(cudaMemGetInfo(&free_b, &total_b));
            if (need * sizeof(double) > free_b)
                FAIL(TSVGP_ERR_INVALID, "elbo_grad with %d coupled latents at M = %d needs %zu bytes of device memory for its slab workspace, "
                     "%zu are free (option \"chunk\" narrows the slabs)", c->L, c->M, need * sizeof(double), free_b);
        }
        for (int s = 0; s < ns; ++s) {
            NEED(c->kpslab[s] = p.get((size_t)c->Mp * nc)); NEED(c->vslab[s] = p.get((size_t)c->Mp * nc));
            NEED(c->uslab[s] = p.get((size_t)u_lat * c->Mp * nc)); NEED(c->xaug[s] = p.get((size_t)nc * W));
            NEED(c->fpart[s] = p.get((size_t)c->fsplit * c->Mp * W)); NEED(c->facc[s] = p.get((size_t)c->Mp * W));
        }
        NEED(c->aux_blocks = p.get(2 * ve_need));
        c->grad_ws = true;
        c->grad_lat = u_lat;
    }
    c->ve_cap = ve_need;
    c->slab_lat = slab_lat;
    c->chunk = nc;
    c->chunk_Mp = c->Mp;
    select_latent(c, c->cur);   // the per-slab views of the selected latent
    return TSVGP_OK;
}

// The streaming pass over `N` points whose scaled, feature-major coordinates are XsT/x2.
// phase 0: the whole pass.  phase 1: set-up plus the posterior-independent head (Kuf slab and constant-weight SYRK of the first slab
// of every slab stream; Gaussian likelihood, fused route) — enqueued BEFORE the posterior chain.  phase 2: the rest of a pass whose
// phase 1 has been enqueued: the early slabs only run their posterior-dependent part (means, variance product, point statistics,
// b += Kuf g).
enum { PASS_WHOLE = 0, PASS_EARLY = 1, PASS_REST = 2 };
inline bool grad_spread_skip(const tsvgp_ctx*) { return false; }
// y / mean_out / var_out of latent l live at + l * y_stride / + l * out_stride (Y transposed to [L][n_pad]; outputs [L][n_pad_out]).
// lat_only >= 0 restricts the per-latent work to that latent (the M-step gradient pass runs latent by latent).
// Separate kernels: latent l's scaled coordinates are at XsT + l * xs_lat, x2 + l * x2_lat, and every latent builds its own slab.
int stream_pass(tsvgp_ctx* c, const double* XsT, long ldx, const double* x2, long N, const double* y, const double* mean_off,
                int mode, double* mean_out, double* var_out, int phase = PASS_WHOLE, long y_stride = 0, long out_stride = 0,
                int lat_only = -1, long xs_lat = 0, long x2_lat = 0) {
    const bool grad = mode == MODE_GRAD;
    const bool stats = mode == MODE_STATS || grad;
    if (phase != PASS_REST) OK(ensure_slabs(c, N, grad));
    const long nc = c->chunk;
    const int Mp = c->Mp;
    const int nstr = c->profile ? 1 : (c->n_streams < 1 ? 1 : (c->n_streams > MAXS ? MAXS : c->n_streams));
    const bool prof = c->profile && mode == MODE_STATS && c->L == 1;
    const int l_lo = lat_only >= 0 ? lat_only : 0, l_hi = lat_only >= 0 ? lat_only + 1 : c->L;
    const bool multi = c->L > 1;
    const bool joint = coupled(c);
    const bool sep = c->sep;
    size_t pev_used = 0;
    auto mark = [&](cudaStream_t st) -> int {   // profile mode: one event between consecutive kernels
        if (!prof) return 0;
        if (pev_used == c->pev.size()) {
            cudaEvent_t e;
            if (cudaEventCreate(&e) != cudaSuccess) return 1;
            c->pev.push_back(e);
        }
        return cudaEventRecord(c->pev[pev_used++], st) != cudaSuccess;
    };
    const long vstride = (nc + 255) / 256;
    const long ncu = used_chunk(c, N, nc, nstr);   // slab width of this pass (<= the allocated width nc, which stays the leading dimension)
    const long nchunks = (N + ncu - 1) / ncu;
    const size_t mm = (size_t)Mp * Mp;
    cudaStream_t sm = c->s_main;

    if (phase != PASS_REST) {
        CU(cudaMemsetAsync(c->flags, 0, 2 * sizeof(int), sm));
        CU(cudaMemsetAsync(c->ve_all, 0, sizeof(double) * (size_t)c->L * c->ve_cap, sm));
        if (grad) CU(cudaMemsetAsync(c->aux_blocks, 0, sizeof(double) * (size_t)(2 * nchunks * vstride), sm));
        CU(cudaEventRecord(c->ev_fork, sm));
        for (int s = 0; s < nstr; ++s) {
            CU(cudaStreamWaitEvent(c->s_pp[s], c->ev_fork, 0));
            if (stats) {   // every slab stream zeroes its own accumulators (off the main stream, which runs the posterior chain)
                CU(cudaMemsetAsync(c->stats_all[s], 0, sizeof(double) * c->L * (mm + Mp + 4), c->s_pp[s]));
                CU(cudaMemsetAsync(c->stats2_all[s], 0, sizeof(double) * c->L * (mm + Mp), c->s_pp[s]));
                if (c->spread_b) CU(cudaMemsetAsync(c->bacc[s], 0, sizeof(double) * c->L * 2 * (Mp / 128) * Mp, c->s_pp[s]));
                if (grad) CU(cudaMemsetAsync(c->facc[s], 0, sizeof(double) * (size_t)Mp * c->waug, c->s_pp[s]));
            }
        }
        c->n_early = 0;
    }
    // the weighted SYRK of one slab for the selected latent (and, fused into it, b += K g unless `with_b` is false)
    auto syrk = [&](int b, const double* stat_slab, int ncols, bool const_h, bool with_b, bool& fused_b) -> int {
        cudaStream_t s = c->s_pp[b];
        GemmP p;
        p.A = stat_slab; p.lda = nc; p.a_kc = 1;
        p.B = stat_slab; p.ldb = nc; p.b_kc = 1;
        p.C = c->stats[b]; p.ldc = Mp; p.m = p.n = Mp; p.k = ncols;
        p.beta = 1.0; p.lower_out = 1; p.kscale = c->hbuf[b];
        // Gaussian likelihood: h_n is the same constant -1/(2 s2) for every point (tsvgp.py:256-263 with the closed-form
        // variational expectation), so it multiplies the product once instead of every B fragment
        // (the whitened sibling does not clip the variance gradient, tsvgp_white.py:183-212)
        if (const_h) { p.kscale = nullptr; p.alpha = c->white ? -0.5 / c->lik.p0 : fmin(-0.5 / c->lik.p0, -1e-8); }
        const int nt = Mp / 128;
        const int ks_here = c->ksplit < ncols / 128 ? c->ksplit : ncols / 128;
        fused_b = false;
        if (const_h && c->route == ROUTE_FUSED && !c->white && ks_here <= 1 && c->i8_planes[b] && ncols <= I8_MAX_COLS) {
            // the raw covariance slab, one weight: B += alpha K K^T exactly on the int8 tensor cores (b += K g by the caller's gemv)
            LA(i8_syrk_launch(stat_slab, nc, Mp, ncols, c->kern_var, p.alpha, c->i8_planes[b], nc, c->i8_tiles[b], c->stats[b], Mp, s));
            return TSVGP_OK;
        }
        if (ks_here > 1) {
            p.ksplit = ks_here; p.part = c->kpart[b]; p.part_stride = (long)Mp * Mp;
            LA(gemm_launch(p, s));
            LA(splitk_reduce_launch(p, s));
        } else {
            const int ksp = c->balance ? balanced_ksplit(nt * (nt + 1) / 2, ncols) : ncols;
            if (ksp < ncols) { p.ksp = ksp; p.C2 = c->stats2[b]; }
            if (c->fuse_b && with_b) {   // b += K g rides on the A fragments the SYRK already holds
                p.gvec = c->gbuf[b]; p.bout = c->stats[b] + (size_t)Mp * Mp; p.bout2 = c->stats2[b] + (size_t)Mp * Mp;
                if (c->spread_b) {   // shared by the tiles of a tile row, one private slot per tile column (summed at the end of the pass)
                    double* base = c->bacc[b] + (size_t)c->cur * 2 * nt * Mp;
                    p.bout = base; p.bout2 = base + (size_t)nt * Mp; p.bstride = Mp;
                }
                fused_b = true;
            }
            LA(gemm_launch(p, s));
        }
        return TSVGP_OK;
    };
    const bool const_h_pass = c->lik.kind == LIK_GAUSSIAN && !grad;
    // Gaussian natgrad_step: g_n and h_n do not read v_n, so neither do B, b and the new sites.  The variance product is skipped
    // and the ELBO's variance term taken from B afterwards (variance_term_from_stats); the point kernel then sees var = k(x,x).
    const bool skip_var = mode == MODE_STATS && const_h_pass && !c->white;
    // ... and with one kernel every latent's B is the same matrix K diag(h) K^T: one SYRK (latent l_lo's), copied after the pass
    const bool one_syrk = stats && const_h_pass && !sep && l_hi - l_lo > 1;
    if (phase == PASS_EARLY) {
        const bool ok = mode == MODE_STATS && const_h_pass && c->route == ROUTE_FUSED && !c->white && !prof && c->ksplit <= 1 &&
                        nchunks >= 2 * nstr && !multi && !c->sep;   // (separate kernels build every slab in the pass itself)
        const int ne = ok ? (c->early_slabs < nstr ? c->early_slabs : nstr) : 0;
        for (int ci = 0; ci < ne; ++ci) {
            const long n0 = ci * ncu;
            const long nvalid = N - n0 < ncu ? N - n0 : ncu;
            const int ncols = (int)round_up(nvalid, 128);
            LA(kuf_launch(c->kern_kind, c->kern_var, XsT, ldx, x2, n0, N, ncols, c->Zs, c->z2, c->M, Mp, c->D, nullptr, c->slab[ci],
                          nc, nullptr, 0, 0, c->s_pp[ci], nullptr));
            bool fb;
            OK(syrk(ci, c->slab[ci], ncols, true, false, fb));
            if (ci == 0) CU(cudaEventRecord(c->ev_early0, c->s_pp[0]));
        }
        c->n_early = ne;
        return TSVGP_OK;
    }
    if (phase == PASS_REST) {   // the slab streams continue once the posterior factors are complete on the main stream
        CU(cudaEventRecord(c->ev_post, sm));
        for (int s = 0; s < nstr; ++s) CU(cudaStreamWaitEvent(c->s_pp[s], c->ev_post, 0));
    }
    const int n_early = phase == PASS_REST ? c->n_early : 0;

    for (long ci = 0; ci < nchunks; ++ci) {
        const int b = (int)(ci % nstr);
        cudaStream_t s = c->s_pp[b];
        const long n0 = ci * ncu;
        const long nvalid = N - n0 < ncu ? N - n0 : ncu;
        const int ncols = (int)round_up(nvalid, 128);
        const bool early = ci < n_early;   // Kuf slab and SYRK already enqueued by phase 1
        select_latent(c, l_lo);
        if (mark(s)) FAIL(TSVGP_ERR_CUDA, "profile event");
        // (a) covariance slab K[Mp x ncols] — ONE slab for all latents — and, for a single latent, the partial means
        //     sum_i alpha_i K[i][n] in the same kernel (separate kernels: per latent, below)
        if (!early && !sep)
            LA(kuf_launch(c->kern_kind, c->kern_var, XsT, ldx, x2, n0, N, ncols, c->Zs, c->z2, c->M, Mp, c->D, multi ? nullptr : c->alpha,
                          c->slab[b], nc, multi ? nullptr : c->mu_part[b], nc, 0, s, grad ? c->kpslab[b] : nullptr));
        mark(s);
        for (int l = l_lo; l < l_hi; ++l) {
            select_latent(c, l);
            if (sep)   // (a') latent l's kernel and scaled coordinates into latent l's slab, with its partial means
                LA(kuf_launch(c->kern_kind, c->kern_var, XsT + l * xs_lat, ldx, x2 + l * x2_lat, n0, N, ncols, c->Zs, c->z2, c->M, Mp,
                              c->D, c->alpha, c->slab[b], nc, c->mu_part[b], nc, 0, s, nullptr));
            else if (early || multi)   // the slab exists already: the same per-64-row partial means from a transposed mat-vec over it
                LA(gemv_t_part_launch(c->slab[b], nc, Mp, ncols, c->alpha, c->mu_part[b], nc, s));
            if (skip_var) {
                // (b) not formed: the pass needs no v_n (see skip_var)
            } else if (!c->white) {   // (b) |T^T k_n|^2 : upper-triangular T^T times the slab, reduced to column norms in the epilogue
                GemmP p;
                p.A = c->T; p.lda = Mp; p.a_kc = 0; p.a_tri = 2;
                p.B = c->slab[b]; p.ldb = nc; p.b_kc = 0;
                p.m = Mp; p.n = ncols; p.k = Mp;
                p.epilogue = grad ? EPI_STORE_COLNORM : EPI_COLNORM; p.norm_out = c->q_part[b]; p.ldn = nc;
                if (grad) { p.C = c->vslab[b]; p.ldc = nc; }   // the M-step also needs V = T^T K itself
                LA(gemm_launch(p, s));
                if (grad && joint) {   // U_l = T_l V_l now, into latent l's own U slab: V is overwritten by the next latent
                    GemmP u;
                    u.A = c->T; u.lda = Mp; u.a_kc = 1; u.a_tri = 1;
                    u.B = c->vslab[b]; u.ldb = nc; u.b_kc = 0;
                    u.C = c->uslab[b] + (size_t)l * Mp * nc; u.ldc = nc; u.m = Mp; u.n = ncols; u.k = Mp;
                    LA(gemm_launch(u, s));
                }
            } else {           // (b') whitened sibling: |LA^-1 k_n|^2 and |LR^-1 k_n|^2, two lower-triangular products (util.py:78-85).
                // The first does not depend on the latent: it is formed once per slab, into the buffer shared by the latents
                // (`q2_part`); the per-latent one goes to the latent's own `q_part`.
                for (int which = l == l_lo ? 0 : 1; which < 2; ++which) {
                    GemmP p;
                    p.A = which == 0 ? c->C6inv : c->T; p.lda = Mp; p.a_kc = 1; p.a_tri = 1;
                    p.B = c->slab[b]; p.ldb = nc; p.b_kc = 0;
                    p.m = Mp; p.n = ncols; p.k = Mp;
                    p.epilogue = EPI_COLNORM; p.norm_out = which == 0 ? c->q2_part[b] : c->q_part[b]; p.ldn = nc;
                    LA(gemm_launch(p, s));
                }
            }
            mark(s);
            if (!joint) {   // (c) marginals -> likelihood expectations and gradients, latent by latent (independent likelihood terms)
                PointArgs a;
                a.mu_part = c->mu_part[b]; a.n_mu_part = Mp / 64; a.ldmu = nc;
                a.q_part = c->white ? c->q2_part[b] : c->q_part[b]; a.n_q_part = skip_var ? 0 : Mp / 128; a.ldq = nc;   // subtracted: |LA^-1 k|^2 (white) / |T^T k|^2
                a.q2_part = c->white ? c->q_part[b] : nullptr;                                           // added:      |LR_l^-1 k|^2 (white)
                a.y = y ? y + l * y_stride + n0 : nullptr;
                a.mean_off = mean_off ? mean_off + n0 : nullptr;
                a.kdiag = c->kern_var;
                a.n_valid = nvalid; a.ncols = ncols;
                a.g = stats ? c->gbuf[b] : nullptr; a.h = stats ? c->hbuf[b] : nullptr;
                a.clip = (grad || c->white) ? 0 : 1;   // tsvgp_white.py:183-212 does not clip the variance gradient
                a.aux_blocks = grad ? c->aux_blocks + 2 * ci * vstride : nullptr;
                a.mean_out = mean_out ? mean_out + l * out_stride + n0 : nullptr; a.var_out = var_out ? var_out + l * out_stride + n0 : nullptr;
                a.ve_blocks = c->ve_blocks + ci * vstride;
                a.flags = c->flags;
                a.x2 = skip_var ? x2 + l * x2_lat + n0 : nullptr;   // no v_n to catch non-finite data: check the points themselves
                LA(point_stats_launch(c->lik, a, c->gh, s));
            }
            mark(s);
        }
        if (joint) {   // (c) Softmax / heteroskedastic: the expectation over all latents of a point at once
            select_latent(c, 0);
            SoftmaxArgs a;
            a.mu_part = c->mu_part[b]; a.n_mu_part = Mp / 64; a.ldmu = nc; a.mu_lat = (long)(Mp / 64) * nc;
            a.q_part = c->q_part[b]; a.n_q_part = Mp / 128; a.ldq = nc; a.q_lat = (long)(Mp / 128) * nc;
            a.L = c->L; a.S = c->lik.n_gh;
            a.y = y ? y + n0 : nullptr;
            a.mean_off = mean_off ? mean_off + n0 : nullptr;
            for (int l = 0; l < c->L; ++l) a.kdiag[l] = sep ? c->lk[l].var : c->kern_var;
            a.n_valid = nvalid; a.ncols = ncols; a.n0 = n0; a.n_total = N;
            a.g = stats ? c->gbuf[b] : nullptr; a.h = stats ? c->hbuf[b] : nullptr; a.gh_lat = nc;
            a.mean_out = mean_out ? mean_out + n0 : nullptr; a.var_out = var_out ? var_out + n0 : nullptr; a.out_lat = out_stride;
            a.ve_blocks = c->ve_blocks + ci * vstride;
            a.flags = c->flags;
            a.eps = (c->mc_eps && c->mc_eps_n == N) ? c->mc_eps : nullptr;
            a.seed = c->mc_seed; a.draw = c->mc_draw;
            a.clip = grad ? 0 : 1;   // the ELBO gradient takes h unclipped
            a.aux_blocks = grad ? c->aux_blocks + 2 * ci * vstride : nullptr;
            if (c->lik.kind == LIK_HETEROSKEDASTIC) LA(heteroskedastic_stats_launch(c->lik, a, c->gh, s));
            else LA(softmax_stats_launch(a, s));
        }
        if (stats) {
            // (c') whitened slab  C9^-1 K  (reference order: A = K9^-1 Kuf first, tsvgp.py:271) of the selected latent
            auto stat_slab_of = [&](const double*& out) -> int {
                out = c->slab[b];
                if ((c->route == ROUTE_WHITENED || c->route == ROUTE_EXACT) && !grad) {
                    GemmP p;
                    p.A = c->C9inv; p.lda = Mp; p.a_kc = 1; p.a_tri = 1;
                    p.B = c->slab[b]; p.ldb = nc; p.b_kc = 0;
                    p.C = c->wslab[b]; p.ldc = nc; p.m = Mp; p.n = ncols; p.k = Mp;
                    LA(gemm_launch(p, s));
                    out = c->wslab[b];
                    if (c->route == ROUTE_EXACT) {   // (c'') A = C9^-T (C9^-1 K) = K9^-1 Kuf itself, written over the covariance slab (no longer needed)
                        GemmP q;
                        q.A = c->C9inv; q.lda = Mp; q.a_kc = 0; q.a_tri = 2;
                        q.B = c->wslab[b]; q.ldb = nc; q.b_kc = 0;
                        q.C = c->slab[b]; q.ldc = nc; q.m = Mp; q.n = ncols; q.k = Mp;
                        LA(gemm_launch(q, s));
                        out = c->slab[b];
                    }
                }
                return TSVGP_OK;
            };
            const double* stat_slab = nullptr;
            if (!sep) OK(stat_slab_of(stat_slab));   // one slab (and one K9) for every latent
            mark(s);
            for (int l = l_lo; l < l_hi; ++l) {   // (d) B_l += K diag(h_l) K^T, lower tiles (already enqueued for an early slab)
                select_latent(c, l);
                if (sep) OK(stat_slab_of(stat_slab));   // latent l's slab and C9_l
                bool fused_b = false;
                if (!early && !(one_syrk && l > l_lo)) OK(syrk(b, stat_slab, ncols, const_h_pass, true, fused_b));
                mark(s);
                // (e) b += K g as its own kernel when the SYRK ran split-K or ahead of the posterior
                if (!fused_b) LA(gemv_n_launch(stat_slab, nc, Mp, ncols, c->gbuf[b], 1.0, 1.0, c->stats[b] + (size_t)Mp * Mp, s));
            }
            mark(s);
        }
        if (grad) {
            select_latent(c, l_lo);
            if (!joint) {   // U = T V = Q K  (lower-triangular T times the stored V)
                GemmP p;
                p.A = c->T; p.lda = Mp; p.a_kc = 1; p.a_tri = 1;
                p.B = c->vslab[b]; p.ldb = nc; p.b_kc = 0;
                p.C = c->uslab[b]; p.ldc = nc; p.m = Mp; p.n = ncols; p.k = Mp;
                LA(gemm_launch(p, s));
            }
            // E = scale (alpha g^T - 2 U diag(h)) .* dK/dr2   (in place), then F += E [xs | 1 | xs^2]
            LA(egrad_uf_launch(c->uslab[b], c->kpslab[b], nc, Mp, ncols, c->alpha, c->gbuf[b], c->hbuf[b], c->grad_scale, s));
            for (int l = l_lo + 1; joint && l < l_hi; ++l) {   // coupled likelihood: the latents share Kuf, so E = sum_l E_l (over U_0)
                select_latent(c, l);
                LA(egrad_uf_launch(c->uslab[b] + (size_t)l * Mp * nc, c->kpslab[b], nc, Mp, ncols, c->alpha, c->gbuf[b], c->hbuf[b],
                                   c->grad_scale, s, c->uslab[b]));
            }
            select_latent(c, l_lo);
            LA(xaug_launch(XsT, ldx, n0, nvalid, ncols, c->D, c->xaug[b], s, c->origin));
            GemmP p;
            p.A = c->uslab[b]; p.lda = nc; p.a_kc = 1;
            p.B = c->xaug[b]; p.ldb = c->waug; p.b_kc = 0;
            p.C = c->facc[b]; p.ldc = c->waug; p.m = Mp; p.n = c->waug; p.k = ncols; p.beta = 1.0;
            const int fs = c->fsplit < ncols / 256 ? c->fsplit : ncols / 256;
            if (fs > 1) {
                p.ksplit = fs; p.part = c->fpart[b]; p.part_stride = (long)Mp * c->waug;
                LA(gemm_launch(p, s));
                LA(splitk_reduce_launch(p, s));
            } else {
                LA(gemm_launch(p, s));
            }
        }
        if (c->mark_mid && ci == (nstr < nchunks - 1 ? nstr : nchunks - 1)) CU(cudaEventRecord(c->ev_mid, s));
    }
    if (prof) {   // 7 events per slab: [start, kuf, var, point, whiten, syrk, gemv]
        CU(cudaStreamSynchronize(c->s_pp[0]));
        for (int k = 0; k < 12; ++k) c->kprof[k] = 0.0;
        for (size_t e = 0; e + 6 < pev_used; e += 7)
            for (int k = 0; k < 6; ++k) {
                float ms = 0;
                cudaEventElapsedTime(&ms, c->pev[e + k], c->pev[e + k + 1]);
                if (k == 1 && skip_var) continue;
                if (k == 3 && c->route != ROUTE_WHITENED && c->route != ROUTE_EXACT) continue;
                c->kprof[2 * k] += ms;
                c->kprof[2 * k + 1] += 1.0;
            }
    }
    for (int s = 0; s < nstr; ++s) {
        CU(cudaEventRecord(c->ev_join[s], c->s_pp[s]));
        CU(cudaStreamWaitEvent(sm, c->ev_join[s], 0));
    }
    if (stats && c->spread_b && c->fuse_b && !grad_spread_skip(c)) {   // b_l += sum over streams, pieces and tile columns of the private mat-vec slots
        const int nt = Mp / 128;
        for (int l = l_lo; l < l_hi; ++l) {
            select_latent(c, l);
            for (int s = 0; s < nstr; ++s)
                LA(sum_rows_into_launch(c->bacc[s] + (size_t)l * 2 * nt * Mp, 2 * nt, Mp, c->stats[0] + mm, sm));
        }
    }
    if (stats) {   // the latents' accumulators are contiguous: one launch per pair of buffers sums all of them
        const long cnt = (long)((l_hi - l_lo) * (mm + Mp + 4)), cnt2 = (long)((l_hi - l_lo) * (mm + Mp));
        select_latent(c, l_lo);
        for (int s = 1; s < nstr; ++s) LA(vadd_inplace_launch(c->stats[0], c->stats[s], cnt, sm));
        for (int s = 1; s < nstr && grad; ++s) LA(vadd_inplace_launch(c->facc[0], c->facc[s], (long)Mp * c->waug, sm));
        for (int l = l_lo; l < l_hi && c->balance; ++l) {
            select_latent(c, l);
            for (int s = 0; s < nstr; ++s) LA(vadd_inplace_launch(c->stats[0], c->stats2[s], (long)(mm + Mp), sm));
        }
        (void)cnt2;
        for (int l = l_lo + 1; l < l_hi && one_syrk; ++l)
            CU(cudaMemcpyAsync(c->stats_all[0] + l * (mm + Mp + 4), c->stats_all[0] + l_lo * (mm + Mp + 4), sizeof(double) * mm,
                               cudaMemcpyDeviceToDevice, sm));
    }
    for (int l = l_lo; l < l_hi; ++l) {
        select_latent(c, l);
        // (a coupled likelihood's expectations and sum of h are all in latent 0's slots)
        LA(stats_tail_launch(c->ve_blocks, nchunks * vstride, c->flags, grad && (!joint || l == 0) ? c->aux_blocks : nullptr,
                             c->stats[0] + mm + Mp, sm));
    }
    select_latent(c, l_lo);
    return TSVGP_OK;
}

// the pass over the RESIDENT minibatch: Y is the transposed copy [L][n_pad] when the L latents have independent likelihood terms
int data_pass(tsvgp_ctx* c, int mode, int phase = PASS_WHOLE, int lat_only = -1) {
    const bool per_latent_y = c->L > 1 && !coupled(c);
    return stream_pass(c, c->XsT, c->n_pad, c->x2, c->N, per_latent_y ? c->Yt : c->Y, c->meanX, mode, nullptr, nullptr, phase,
                       per_latent_y ? c->n_pad : 0, 0, lat_only, c->sep ? (long)c->D * c->n_pad : 0, c->sep ? c->n_pad : 0);
}

int all_reduce(tsvgp_ctx* c, double* buf, size_t count) {
    if (c->world <= 1) return TSVGP_OK;
    NcclApi& api = nccl_api();
    int r = api.AllReduce(buf, buf, count, NCCL_FLOAT64, NCCL_SUM, c->comm, c->s_main);
    if (r != 0) FAIL(TSVGP_ERR_COMM, "ncclAllReduce: %s", api.GetErrorString ? api.GetErrorString(r) : "error");
    return TSVGP_OK;
}

// Every M x M product outside the streaming pass goes through here: few output tiles (small M, panels) are split over the idle SMs.
int mm_gemm(tsvgp_ctx* c, const GemmP& p, cudaStream_t s) {
    return gemm_launch_auto(p, s, s == c->s_side ? c->gws2 : c->gws, c->gws_doubles);
}

// An M x M product of the dense phase.  With several ranks and a large M it is DISTRIBUTED: tile rows are dealt out cyclically,
// each rank computes its rows into a zeroed C, and one all-reduce assembles the matrix on every rank (bit-identical everywhere:
// each entry is one rank's value plus zeros).  Below `dist_min_m` the product is latency-bound and stays replicated.
// Requires p.beta == 0 and every rank calling in the same order.
bool dist_active(const tsvgp_ctx* c) { return c->world > 1 && c->Mp >= c->dist_min_m && c->collective_ok; }

int dense_gemm(tsvgp_ctx* c, GemmP p, cudaStream_t s) {
    if (!dist_active(c) || p.beta != 0.0) {
        LA(mm_gemm(c, p, s));
        return TSVGP_OK;
    }
    CU(cudaMemsetAsync(p.C, 0, sizeof(double) * (size_t)p.m * p.ldc, s));
    p.row_mod = c->world; p.row_rem = c->rank;
    LA(mm_gemm(c, p, s));
    return all_reduce(c, p.C, (size_t)p.m * p.ldc);
}

// K9 = K + jitter I = C9 C9^T and C9^-1 (tsvgp.py:268-271), kept while kernel, Z and jitter are unchanged.  It depends on the
// kernel matrix only, so it is factored on a SIDE stream (own workspace) while the main stream builds the posterior factors
// from the sites; both chains are latency-bound, so running them side by side nearly halves the prepare phase.
bool k9_cached(const tsvgp_ctx* c, double jitter) { return c->k9_valid && c->k9_jitter == jitter && c->cache_factors; }

int k9_fork(tsvgp_ctx* c) {   // the side stream starts after the kernel matrix K is complete on the main stream
    CU(cudaEventRecord(c->ev_kuu, c->s_main));
    CU(cudaStreamWaitEvent(c->s_side, c->ev_kuu, 0));
    return TSVGP_OK;
}

int k9_chain(tsvgp_ctx* c, double jitter);

int start_k9(tsvgp_ctx* c, double jitter) {
    if (k9_cached(c, jitter)) return TSVGP_OK;
    OK(k9_fork(c));
    return k9_chain(c, jitter);
}

// Both chains of the prepare phase are ~40 dependent small kernels; at small M their GPU time is comparable to the time the host
// needs to enqueue them, so enqueueing them one after the other delays the second chain by the first one's issue time.  With
// `async_issue` a helper thread enqueues the K9 chain on the side stream while the calling thread enqueues the posterior chain.
struct SideIssue {
    std::thread th;
    int rc = TSVGP_OK;
    long launches = 0;
    bool active = false;
    void join_into(long& counter) {
        if (!active) return;
        th.join();
        counter += launches;
        active = false;
    }
};

int start_k9_async(tsvgp_ctx* c, double jitter, SideIssue& side) {
    if (k9_cached(c, jitter)) return TSVGP_OK;
    OK(k9_fork(c));
    if (!c->async_issue || c->Mp > 1024) return k9_chain(c, jitter);
    try {
        side.th = std::thread([c, jitter, &side]() {
            const long l0 = g_launches;
            side.rc = cudaSetDevice(c->dev) == cudaSuccess ? k9_chain(c, jitter) : TSVGP_ERR_CUDA;
            side.launches = g_launches - l0;
        });
        side.active = true;
    } catch (...) {   // no thread to be had: enqueue the chain from this thread
        return k9_chain(c, jitter);
    }
    return TSVGP_OK;
}

// One kernel's chain: K9 = K + jitter I = C9 C9^T, C9^-1, K9^-1 (when `with_inv`) and the conditioning probe into probe[N_SCAL].
// The buffers are passed explicitly: with separate kernels the chains run on the side stream, possibly issued from the helper
// thread, while the calling thread moves the latent views.
int k9_chain_one(tsvgp_ctx* c, double jitter, const double* K, double* C9, double* C9inv, double* K9inv, double* probe, bool with_inv) {
    cudaStream_t s = c->s_side;
    LA(copy_add_diag_launch(K, C9, c->Mp, c->Mp, jitter, s));
    LA(chol_lower(C9, c->Mp, c->Mp, c->dinv2, c->info + INFO_K9, s, c->gws2, c->gws_doubles, &c->la_side));
    LA(trtri_lower(C9, c->Mp, c->Mp, c->dinv2, C9inv, c->tmp2, s, c->gws2, c->gws_doubles));
    if (with_inv) {
        GemmP p;
        p.A = C9inv; p.lda = c->Mp; p.a_kc = 0; p.a_tri = 2;
        p.B = C9inv; p.ldb = c->Mp; p.b_kc = 0; p.b_tri = 2;
        p.C = K9inv; p.ldc = c->Mp; p.m = p.n = p.k = c->Mp; p.lower_out = 1;
        LA(mm_gemm(c, p, s));
        LA(mirror_lower_launch(K9inv, c->Mp, c->Mp, s));
    }
    if (c->route_opt == ROUTE_AUTO) {
        // conditioning probe: 8 power iterations each on K and on K9^-1 = C9^-T C9^-1; Rayleigh ratios of the last two
        // iterates give lambda_max(K) and 1/lambda_min(K9) (both from below)
        const int n = c->Mp;
        double *a = c->pv1, *b = c->pv2;
        LA(probe_vector_launch(a, c->M, n, s));
        for (int it = 0; it < 8; ++it) {
            if (it == 7) LA(dot_launch(a, a, c->M, probe + SC_PK0, s));
            LA(gemv_n_launch(K, n, c->M, c->M, a, 1.0, 0.0, b, s));
            double* t = a; a = b; b = t;
        }
        LA(dot_launch(a, a, c->M, probe + SC_PK1, s));
        LA(probe_vector_launch(a, c->M, n, s));
        for (int it = 0; it < 8; ++it) {
            if (it == 7) LA(dot_launch(a, a, n, probe + SC_PI0, s));
            if (with_inv) {   // K9^-1 itself is at hand (formed just above): one mat-vec per iteration instead of two
                LA(gemv_n_launch(K9inv, n, n, n, a, 1.0, 0.0, b, s));
                double* t = a; a = b; b = t;
            } else {
                LA(gemv_n_launch(C9inv, n, n, n, a, 1.0, 0.0, b, s));
                LA(gemv_t_launch(C9inv, n, n, n, b, a, c->gwork2, s));
            }
        }
        LA(dot_launch(a, a, n, probe + SC_PI1, s));
    }
    return TSVGP_OK;
}

int k9_chain(tsvgp_ctx* c, double jitter) {
    // single rank / small M: form K9^-1 in the chain, hidden behind the main stream's posterior preparation.  Separate kernels
    // always do (dense_update_one forms a missing K9^-1 once per step, not once per latent); their chains run back to back,
    // each with its own probe slots.
    const bool with_inv = !dist_active(c) || c->sep;
    c->k9inv_valid = false;
    if (c->sep) {
        for (int l = 0; l < c->L; ++l) {
            const tsvgp_ctx::KernelState& k = c->lk[l];
            OK(k9_chain_one(c, jitter, k.K, k.C9, k.C9inv, k.K9inv, c->scal2 + (size_t)l * N_SCAL, true));
        }
    } else {
        OK(k9_chain_one(c, jitter, c->K, c->C9, c->C9inv, c->K9inv, c->scal2, with_inv));
    }
    c->k9inv_valid = with_inv;
    c->k9_valid = true;
    c->k9_jitter = jitter;
    c->cond_est = 0.0;
    c->k9_pending = true;
    CU(cudaEventRecord(c->ev_side, c->s_side));
    return TSVGP_OK;
}

int route_for(const tsvgp_ctx* c, double cond) {
    if (c->route_opt != ROUTE_AUTO) return c->route_opt;
    return cond <= c->route_cond_max ? ROUTE_FUSED : (cond <= c->route_exact_min ? ROUTE_WHITENED : ROUTE_EXACT);
}

// joins the side stream, reads the conditioning probe (if one ran) and fixes the statistics route of this step
int choose_route(tsvgp_ctx* c, double jitter) {
    if (c->k9_pending) {
        if (c->route_opt == ROUTE_AUTO) {   // separate kernels: the pass takes the route of the worst-conditioned latent
            const int nk = c->sep ? c->L : 1;
            std::vector<double> scv((size_t)nk * N_SCAL);
            CU(cudaMemcpyAsync(scv.data(), c->scal2, sizeof(double) * scv.size(), cudaMemcpyDeviceToHost, c->s_side));
            CU(cudaStreamSynchronize(c->s_side));
            c->cond_est = 0.0;
            for (int l = 0; l < nk; ++l) {
                const double* sc = scv.data() + (size_t)l * N_SCAL;
                const double lmax = sqrt(sc[SC_PK1] / sc[SC_PK0]) + jitter, inv_lmin = sqrt(sc[SC_PI1] / sc[SC_PI0]);
                double e = lmax * inv_lmin;
                if (!(e == e)) e = INFINITY;   // failed factorisation: the step will report it
                if (l == 0 || e > c->cond_est) c->cond_est = e;
            }
            c->cond_hint = c->cond_est;
            c->cond_hint_valid = true;
        }
        CU(cudaStreamWaitEvent(c->s_main, c->ev_side, 0));
        c->k9_pending = false;
    }
    c->route = route_for(c, c->cond_est);
    return TSVGP_OK;
}

// tsvgp.py:268-303 after the statistics are complete in stats[0]
int dense_update_one(tsvgp_ctx* c, double lr, double jitter, double scale, bool only_G, bool G_ready = false);
int dense_update(tsvgp_ctx* c, double lr, double jitter, double scale, bool only_G) {
    for (int l = 0; l < c->L; ++l) {   // the latents' site updates are independent (tsvgp.py:293-303 per latent)
        select_latent(c, l);
        OK(dense_update_one(c, lr, jitter, scale, only_G));
    }
    if (c->L > 1 && !only_G && !c->white) {   // (the whitened sibling's update has no factorisation and commits latent by latent)
        // commit AFTER every latent has factored its -2 Lambda_2 + jitter I: the reference raises before any assign (tsvgp.py:300-303),
        // so a failure in latent l must leave the latents before l untouched too (the guards read the shared device flags)
        const size_t mm = (size_t)c->Mp * c->Mp;
        for (int l = 0; l < c->L; ++l) {
            select_latent(c, l);
            const double* bad = c->stats[0] + mm + c->Mp + 1;
            LA(update_lambda1_launch(c->lam1, c->stats2[0], c->stats2[0] + c->Mp, c->M, lr, scale, bad, c->info, c->s_main));
            LA(finalize_sites_launch(c->stats[0], c->L2, c->Mp, c->M, c->Mp, bad, c->info, c->s_main));
        }
    }
    select_latent(c, 0);
    return TSVGP_OK;
}

// Multi-GPU, fused route: instead of all-reducing B and repeating G2 = K9^-1 B K9^-1 on every rank (3 M^3 flops each), the
// statistics are reduce-scattered by tile rows, every rank forms its rows of Y = B K9^-1 and, after an all-gather of Y, its rows of
// G2 = K9^-1 Y; a second all-gather leaves the same G2 bits on every rank, so the replicated factorisation that follows stays in
// lock-step.  [b | sum ve | flag] goes through a small all-reduce.  (VERDICT r01 next #3c)
bool sharded_update_active(const tsvgp_ctx* c) {
    return c->world > 1 && c->route == ROUTE_FUSED && c->L == 1 && !c->white && c->Mp >= c->shard_min_m && (c->Mp / 128) % c->world == 0 &&
           nccl_api().ReduceScatter && nccl_api().AllGather;
}

int sharded_reduce_and_form_G(tsvgp_ctx* c) {
    cudaStream_t s = c->s_main;
    NcclApi& api = nccl_api();
    const int n = c->Mp;
    const long ld = n;
    const size_t mm = (size_t)n * n;
    const int R = n / c->world;                  // rows per rank (whole 128-row tiles)
    const size_t blk = (size_t)R * n;
    double* B = c->stats[0];
    double* bvec = c->stats[0] + mm;
    auto chk = [&](int r, const char* what) -> int {
        if (r != 0) FAIL(TSVGP_ERR_COMM, "%s: %s", what, api.GetErrorString ? api.GetErrorString(r) : "error");
        return TSVGP_OK;
    };
    LA(mirror_lower_launch(B, ld, n, s));        // complete rows: the pass accumulated lower tiles only
    double* Brows = c->X2 + (size_t)c->rank * blk;
    OK(chk(api.ReduceScatter(B, Brows, blk, NCCL_FLOAT64, NCCL_SUM, c->comm, s), "ncclReduceScatter"));
    OK(all_reduce(c, bvec, (size_t)n + 4));
    CU(cudaEventRecord(c->ev[EV_REDUCE], s));
    if (!c->k9inv_valid) {   // large M with distributed products: the K9 chain left K9^-1 = C9^-T C9^-1 to a collective product
        GemmP p;
        p.A = c->C9inv; p.lda = ld; p.a_kc = 0; p.a_tri = 2;
        p.B = c->C9inv; p.ldb = ld; p.b_kc = 0; p.b_tri = 2;
        p.C = c->K9inv; p.ldc = ld; p.m = p.n = p.k = n; p.lower_out = 1;
        OK(dense_gemm(c, p, s));
        LA(mirror_lower_launch(c->K9inv, ld, n, s));
        c->k9inv_valid = true;
    }
    {   // Y[rows] = B[rows, :] K9^-1
        GemmP p;
        p.A = Brows; p.lda = ld; p.a_kc = 1;
        p.B = c->K9inv; p.ldb = ld; p.b_kc = 0;
        p.C = c->X1 + (size_t)c->rank * blk; p.ldc = ld; p.m = R; p.n = n; p.k = n;
        LA(mm_gemm(c, p, s));
    }
    OK(chk(api.AllGather(c->X1 + (size_t)c->rank * blk, c->X1, blk, NCCL_FLOAT64, c->comm, s), "ncclAllGather"));
    {   // G2[rows] = K9^-1[rows, :] Y
        GemmP p;
        p.A = c->K9inv + (size_t)c->rank * blk; p.lda = ld; p.a_kc = 1;
        p.B = c->X1; p.ldb = ld; p.b_kc = 0;
        p.C = c->G2 + (size_t)c->rank * blk; p.ldc = ld; p.m = R; p.n = n; p.k = n;
        LA(mm_gemm(c, p, s));
    }
    OK(chk(api.AllGather(c->G2 + (size_t)c->rank * blk, c->G2, blk, NCCL_FLOAT64, c->comm, s), "ncclAllGather"));
    LA(gemv_n_launch(c->K9inv, ld, n, n, bvec, 1.0, 0.0, c->v2, s));   // G1 = K9^-1 b
    return TSVGP_OK;
}

// One rank per chain [r02].  The prepare phase of a step whose kernel matrix changed is two independent latency-bound chains: the
// posterior factors of the sites (T, alpha, m_Z) and the chain of K9 = Kuu + jitter I (C9^-1, K9^-1, conditioning probe).  Every
// rank used to run both, side by side.  With several ranks (option "split_chains") rank 0 builds the posterior factors, with its GPU
// to itself, rank 1 the K9 chain, and each BROADCASTS its result (ncclBroadcast: copies, every rank ends with the same bits as
// before); ranks 2.. build nothing.  The posterior factors travel on the main stream in front of the pass; the K9 results, which the
// fused route needs only after the pass, travel second, on the side stream, and are joined after the pass like the chain itself.
// Every rank but 0 fills the wait for the posterior factors with early slabs (posterior-independent Kuf + constant-weight SYRK):
// they may slow rank 1's K9 chain down, which is off the critical path.  Rank 0 is then the straggler by its chain time unless it gets
// fewer rows: tsvgp_b200.balance_weights (host) turns measured phase times into row shares.
// Used when the K9 chain is joined AFTER the pass anyway (fused route forced or speculated) and the dense products are replicated
// (below dist_min_m; above, the chains' products are themselves collective).
// MEASURED (cfg3, ms per step; profiles/scale_r02_n2_chains.txt, scale_r02_n8_ab.txt): 8 x B200 37.26 with both chains on every
// rank and equal rows, 36.44 with this split and balanced rows; 2 x B200 135.4-135.65 against 135.05-135.24 (both ranks have a chain).
// With equal rows the split and the early slabs do not add up (a first version with ncclSend/ncclRecv inside rank pairs: 135.8 / 135.45
// with / without early slabs against 135.4 / 135.95).
// OFF by default in the library (it needs the caller's cooperation for the row shares); bench.py switches it on for N > 1.
enum { ROLE_BOTH = 0, ROLE_POSTERIOR = 1, ROLE_K9 = 2, ROLE_NONE = 3 };
bool chain_split_active(const tsvgp_ctx* c) {
    return c->split_chains && c->world > 1 && c->L == 1 && !c->white && c->Mp >= c->shard_min_m && !dist_active(c) && nccl_api().bcast();
}
int chain_role_of(const tsvgp_ctx* c) { return c->rank == 0 ? ROLE_POSTERIOR : (c->rank == 1 ? ROLE_K9 : ROLE_NONE); }

int nccl_chk(tsvgp_ctx* c, int r, const char* what) {
    NcclApi& api = nccl_api();
    if (r != 0) FAIL(TSVGP_ERR_COMM, "%s: %s", what, api.GetErrorString ? api.GetErrorString(r) : "error");
    return TSVGP_OK;
}

// posterior factors of rank 0 -> every rank, on the main stream in front of the pass
int exchange_posterior(tsvgp_ctx* c, bool with_kl) {
    NcclApi& api = nccl_api();
    cudaStream_t s = c->s_main;
    const size_t mm = (size_t)c->Mp * c->Mp, mp = c->Mp;
    const int root = 0;
    OK(nccl_chk(c, api.GroupStart(), "ncclGroupStart"));
    int r = 0;
    r |= api.Broadcast(c->T, c->T, mm, NCCL_FLOAT64, root, c->comm, s);
    r |= api.Broadcast(c->alpha, c->alpha, mp, NCCL_FLOAT64, root, c->comm, s);
    r |= api.Broadcast(c->mZ, c->mZ, mp, NCCL_FLOAT64, root, c->comm, s);
    r |= api.Broadcast(c->mq, c->mq, mp, NCCL_FLOAT64, root, c->comm, s);
    r |= api.Broadcast(c->scal, c->scal, N_SCAL, NCCL_FLOAT64, root, c->comm, s);
    r |= api.Broadcast(c->info + INFO_W, c->info + INFO_W, 1, NCCL_INT32, root, c->comm, s);
    const int rg = api.GroupEnd();
    OK(nccl_chk(c, r ? r : rg, "ncclBroadcast (posterior factors)"));
    CU(cudaEventRecord(c->ev_xpost, s));
    if (c->rank != root) {
        c->post_valid = true;
        c->post_collective = false;
        c->kl_valid = with_kl;
    }
    return TSVGP_OK;
}

// K9 results of rank 1 -> every rank, on the side stream (rank 1: behind its chain; the others: in place of the chain)
int exchange_k9(tsvgp_ctx* c, double jitter) {
    NcclApi& api = nccl_api();
    cudaStream_t s = c->s_side;
    const size_t mm = (size_t)c->Mp * c->Mp;
    const int root = 1;
    CU(cudaStreamWaitEvent(s, c->ev_xpost, 0));   // one exchange at a time on the communicator: behind the posterior one (the urgent one)
    // ... and not before the pass is a few slabs in: an NCCL kernel that waits for its root polls on a dozen SMs, which the DMMA tiles
    // of the pass (one CTA per SM, sized for all 148) cannot share; by then rank 1's chain is complete and the transfer is immediate
    CU(cudaStreamWaitEvent(s, c->ev_mid, 0));
    OK(nccl_chk(c, api.GroupStart(), "ncclGroupStart"));
    int r = 0;
    r |= api.Broadcast(c->C9, c->C9, mm, NCCL_FLOAT64, root, c->comm, s);   // (the ELBO of a Gaussian step on another route)
    r |= api.Broadcast(c->C9inv, c->C9inv, mm, NCCL_FLOAT64, root, c->comm, s);
    r |= api.Broadcast(c->K9inv, c->K9inv, mm, NCCL_FLOAT64, root, c->comm, s);
    r |= api.Broadcast(c->scal2, c->scal2, N_SCAL, NCCL_FLOAT64, root, c->comm, s);
    r |= api.Broadcast(c->info + INFO_K9, c->info + INFO_K9, 1, NCCL_INT32, root, c->comm, s);
    const int rg = api.GroupEnd();
    OK(nccl_chk(c, r ? r : rg, "ncclBroadcast (K9 chain)"));
    if (c->rank != root) {   // the state the chain would have left
        c->k9_valid = true; c->k9_jitter = jitter; c->k9inv_valid = true;
        c->cond_est = 0.0;
        c->k9_pending = true;
    }
    CU(cudaEventRecord(c->ev_side, s));   // (re-recorded on rank 1: the join after the pass also covers its broadcast)
    return TSVGP_OK;
}

int dense_update_one(tsvgp_ctx* c, double lr, double jitter, double scale, bool only_G, bool G_ready) {
    cudaStream_t s = c->s_main;
    const int n = c->Mp;
    const long ld = c->Mp;
    const size_t mm = (size_t)n * n;
    double* B = c->stats[0];
    double* bvec = c->stats[0] + mm;
    const double* bad = c->stats[0] + mm + n + 1;
    if (!G_ready) LA(mirror_lower_launch(B, ld, n, s));
    if (G_ready) {
        // G2 (all rows, gathered) and G1 are in place
    } else if (c->route == ROUTE_FUSED) {
        if (!c->k9inv_valid) {   // K9^-1 = C9^-T C9^-1 (symmetric): two M^3 products per step instead of four; kept with chol(K9)
            GemmP p;
            p.A = c->C9inv; p.lda = ld; p.a_kc = 0; p.a_tri = 2;
            p.B = c->C9inv; p.ldb = ld; p.b_kc = 0; p.b_tri = 2;
            p.C = c->K9inv; p.ldc = ld; p.m = p.n = p.k = n; p.lower_out = 1;
            OK(dense_gemm(c, p, s));
            LA(mirror_lower_launch(c->K9inv, ld, n, s));
            c->k9inv_valid = true;
        }
        {   // X1 = K9^-1 B
            GemmP p;
            p.A = c->K9inv; p.lda = ld; p.a_kc = 1;
            p.B = B; p.ldb = ld; p.b_kc = 0;
            p.C = c->X1; p.ldc = ld; p.m = p.n = p.k = n;
            OK(dense_gemm(c, p, s));
        }
        {   // G2 = X1 K9^-1  (symmetric; lower tiles then mirrored)
            GemmP p;
            p.A = c->X1; p.lda = ld; p.a_kc = 1;
            p.B = c->K9inv; p.ldb = ld; p.b_kc = 0;
            p.C = c->G2; p.ldc = ld; p.m = p.n = p.k = n;
            p.lower_out = 1;
            OK(dense_gemm(c, p, s));
        }
        LA(gemv_n_launch(c->K9inv, ld, n, n, bvec, 1.0, 0.0, c->v2, s));   // G1 = K9^-1 b
    } else if (c->route == ROUTE_EXACT) {   // the pass accumulated G2 = A^T diag(h) A and G1 = A^T g themselves (tsvgp.py:273-281)
        CU(cudaMemcpyAsync(c->G2, B, sizeof(double) * mm, cudaMemcpyDeviceToDevice, s));
        CU(cudaMemcpyAsync(c->v2, bvec, sizeof(double) * n, cudaMemcpyDeviceToDevice, s));
    } else {
        const double* Bw = B;      // C9^-1 (Kuf H Kfu) C9^-T accumulated by the whitened pass, symmetric
        {   // X1 = C9^-T Bw
            GemmP p;
            p.A = c->C9inv; p.lda = ld; p.a_kc = 0; p.a_tri = 2;
            p.B = Bw; p.ldb = ld; p.b_kc = 0;
            p.C = c->X1; p.ldc = ld; p.m = p.n = p.k = n;
            OK(dense_gemm(c, p, s));
        }
        {   // G2 = X1 C9^-1  (symmetric)
            GemmP p;
            p.A = c->X1; p.lda = ld; p.a_kc = 1;
            p.B = c->C9inv; p.ldb = ld; p.b_kc = 0; p.b_tri = 2;
            p.C = c->G2; p.ldc = ld; p.m = p.n = p.k = n;
            p.lower_out = 1;
            OK(dense_gemm(c, p, s));
        }
        LA(gemv_t_launch(c->C9inv, ld, n, n, bvec, c->v2, c->gwork, s));   // G1 = C9^-T (C9^-1 Kuf g)
    }
    LA(mirror_lower_launch(c->G2, ld, n, s));
    LA(gemv_n_launch(c->G2, ld, n, n, c->mZ, 1.0, 0.0, c->v3, s));
    if (only_G) return TSVGP_OK;   // G2 (mirrored) in c->G2, G1 in c->v2, G2 mZ in c->v3
    if (c->white) return dense_update_white(c, lr, scale);
    // P = (1-lr) L2 L2^T - 2 lr scale G2 + jitter I                                     tsvgp.py:293-300
    // several latents: the factor and the two vectors of the lambda_1 update wait, per latent, in the (now dead) accumulators B_l and
    // stats2_l until every latent has factored (dense_update commits them together)
    double* Pl = c->L > 1 ? B : c->P;
    LA(init_update_launch(c->G2, Pl, ld, c->M, n, -2.0 * lr * scale, jitter, s));
    if (lr != 1.0) {
        GemmP p;
        p.A = c->L2; p.lda = ld; p.a_kc = 1; p.a_tri = 1;
        p.B = c->L2; p.ldb = ld; p.b_kc = 1; p.b_tri = 1;
        p.C = Pl; p.ldc = ld; p.m = p.n = p.k = n;
        p.alpha = 1.0 - lr; p.lower_out = 1;
        if (dist_active(c)) {   // (1 - lr) L2 L2^T assembled from the ranks' rows, then added
            p.C = c->X2;
            OK(dense_gemm(c, p, s));
            LA(vadd_inplace_launch(Pl, c->X2, (long)n * ld, s));
        } else {
            p.beta = 1.0;
            LA(mm_gemm(c, p, s));
        }
    }
    LA(chol_lower(Pl, ld, n, c->dinv, c->info + INFO_P, s, c->gws, c->gws_doubles, &c->la_main));
    if (c->L > 1) {
        CU(cudaMemcpyAsync(c->stats2[0], c->v2, sizeof(double) * n, cudaMemcpyDeviceToDevice, s));
        CU(cudaMemcpyAsync(c->stats2[0] + n, c->v3, sizeof(double) * n, cudaMemcpyDeviceToDevice, s));
        return TSVGP_OK;
    }
    // commit (skipped on the device if any variance was non-positive or a factorisation failed)
    LA(update_lambda1_launch(c->lam1, c->v2, c->v3, c->M, lr, scale, bad, c->info, s));
    LA(finalize_sites_launch(c->P, c->L2, ld, c->M, n, bad, c->info, s));
    return TSVGP_OK;
}

// Gaussian natgrad_step: the pass took v_n = k(x,x) (stream_pass, skip_var), so its sum of ve lacks + 1/(2 s2) sum_n |T^T k_n|^2.
// Every route's accumulator is B = c R^-1 (sum_n k_n k_n^T) R^-T, c the SYRK's constant weight, R = I (fused), C9 (whitened) or
// K9 = C9 C9^T (exact); with P = R^T T
//   sum_n |T^T k_n|^2 = tr(T^T (sum_n k_n k_n^T) T) = tr(P^T B P) / c          (one M^3 product per latent instead of M^2 per point)
// The term is added to each latent's sum of ve, and the variance flag raised unless sum_n v_n is finite and positive.  Runs on this
// rank's rows before the reduction, which then sums the corrected ve and the flags as before.
int variance_term_from_stats(tsvgp_ctx* c) {
    cudaStream_t s = c->s_main;
    const int n = c->Mp;
    const long ld = n;
    const size_t mm = (size_t)n * n;
    const double cst = fmin(-0.5 / c->lik.p0, -1e-8);   // the weight of stream_pass's constant-weight SYRK
    for (int l = 0; l < c->L; ++l) {
        select_latent(c, l);
        double* B = c->stats[0];
        LA(mirror_lower_launch(B, ld, n, s));   // (the pass accumulated lower tiles only)
        const double* P = c->T;
        if (c->route != ROUTE_FUSED) {   // X2 = C9^T T
            GemmP p;
            p.A = c->C9; p.lda = ld; p.a_kc = 0; p.a_tri = 2;
            p.B = c->T; p.ldb = ld; p.b_kc = 0; p.b_tri = 2;
            p.C = c->X2; p.ldc = ld; p.m = p.n = p.k = n;
            LA(mm_gemm(c, p, s));
            P = c->X2;
            if (c->route == ROUTE_EXACT) {   // X1 = C9 X2 = K9 T
                GemmP q;
                q.A = c->C9; q.lda = ld; q.a_kc = 1; q.a_tri = 1;
                q.B = c->X2; q.ldb = ld; q.b_kc = 0;
                q.C = c->X1; q.ldc = ld; q.m = q.n = q.k = n;
                LA(mm_gemm(c, q, s));
                P = c->X1;
            }
        }
        {   // G2 = B P  (G2 is formed again by the update)
            GemmP p;
            p.A = B; p.lda = ld; p.a_kc = 1;
            p.B = P; p.ldb = ld; p.b_kc = 0; p.b_tri = P == c->T ? 2 : 0;
            p.C = c->G2; p.ldc = ld; p.m = p.n = p.k = n;
            LA(mm_gemm(c, p, s));
        }
        LA(matdot_launch(P, c->G2, ld, n, c->scal + SC_TR_PBP, c->red, s));
        LA(variance_term_launch(c->scal + SC_TR_PBP, 1.0 / cst, (double)c->N * c->kern_var, 0.5 / c->lik.p0, B + mm + n, s));
    }
    select_latent(c, 0);
    return TSVGP_OK;
}

int check_info(tsvgp_ctx* c, const int* info_h) {
    static const char* what[N_INFO] = {"I + L2^T K6 L2 (posterior; Kuu + 1e-6 I for the whitened sibling)", "Kuu + jitter I",
                                       "-2 lambda_2 + jitter I (site update; Lambda_2 + Kuu or S_q for the whitened sibling)",
                                       "S_q (Lambda_2 + Kuu + 1e-9 I for the whitened sibling)"};
    for (int i = 0; i < N_INFO; ++i)
        if (info_h[i]) {
            c->last_info = info_h[i];
            if (i == INFO_K9) c->k9_valid = false;
            c->post_valid = c->kl_valid = c->wpost_valid = c->wkl_valid = false;
            FAIL(TSVGP_ERR_NOT_POSITIVE_DEFINITE, "Cholesky of %s failed at pivot %d", what[i], info_h[i]);
        }
    return TSVGP_OK;
}

void gauss_hermite(int n, double* x, double* w) {   // numpy.polynomial.hermite.hermgauss(n): ascending nodes, weights
    const double PIM4 = 0.7511255444649425;
    const int m = (n + 1) / 2;
    double z = 0;
    for (int i = 0; i < m; ++i) {
        if (i == 0) z = sqrt(2.0 * n + 1.0) - 1.85575 * pow(2.0 * n + 1.0, -0.16667);
        else if (i == 1) z -= 1.14 * pow((double)n, 0.426) / z;
        else if (i == 2) z = 1.86 * z - 0.86 * x[n - 1];
        else if (i == 3) z = 1.91 * z - 0.91 * x[n - 2];
        else z = 2.0 * z - x[n - 1 - (i - 2)];
        double pp = 1;
        for (int its = 0; its < 100; ++its) {
            double p1 = PIM4, p2 = 0.0;
            for (int j = 0; j < n; ++j) {
                const double p3 = p2;
                p2 = p1;
                p1 = z * sqrt(2.0 / (j + 1)) * p2 - sqrt((double)j / (j + 1)) * p3;
            }
            pp = sqrt(2.0 * n) * p2;
            const double z1 = z;
            z = z1 - p1 / pp;
            if (fabs(z - z1) <= 1e-15 * (1.0 + fabs(z))) break;
        }
        x[n - 1 - i] = z;
        x[i] = -z;
        w[i] = w[n - 1 - i] = 2.0 / (pp * pp);
    }
}

}  // namespace

// =====================================================================================================================
// C ABI
// =====================================================================================================================
extern "C" {

int tsvgp_abi_version(void) { return TSVGP_ABI_VERSION; }

int tsvgp_create(tsvgp_ctx** out, int device_id) {
    if (!out) return TSVGP_ERR_INVALID;
    *out = nullptr;
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0) {
        g_create_error = std::string("no CUDA device: ") + (e != cudaSuccess ? cudaGetErrorString(e) : "device count is 0") +
                         " — libtsvgp has no CPU fallback";
        cudaGetLastError();
        return TSVGP_ERR_CUDA;
    }
    if (device_id < 0 || device_id >= ndev) {
        g_create_error = "device_id out of range";
        return TSVGP_ERR_INVALID;
    }
    cudaDeviceProp prop;
    cudaGetDeviceProperties(&prop, device_id);
    if (prop.major != 10) {
        g_create_error = std::string("device is ") + prop.name + " (sm_" + std::to_string(prop.major) + std::to_string(prop.minor) +
                         "); libtsvgp is built for sm_100a only";
        return TSVGP_ERR_CUDA;
    }
    if (const char* dbg = getenv("TSVGP_DEBUG_SYNC")) g_debug_sync = atoi(dbg);
    if (const char* v = getenv("TSVGP_PDL")) g_pdl = atoi(v);
    tsvgp_ctx* c = new tsvgp_ctx();
    c->dev = device_id;
    bool ok = cudaSetDevice(device_id) == cudaSuccess;
    // the latency-bound M x M chains (main and side stream) outrank the slab streams, whose 1-CTA-per-SM DMMA kernels would
    // otherwise make every small chain kernel wait for a whole wave
    int prio_low = 0, prio_high = 0;
    ok = ok && cudaDeviceGetStreamPriorityRange(&prio_low, &prio_high) == cudaSuccess;
    ok = ok && cudaStreamCreateWithPriority(&c->s_main, cudaStreamNonBlocking, prio_high) == cudaSuccess;
    for (int s = 0; s < MAXS && ok; ++s) {
        ok = ok && cudaStreamCreateWithPriority(&c->s_pp[s], cudaStreamNonBlocking, prio_low) == cudaSuccess;
        ok = ok && cudaEventCreateWithFlags(&c->ev_join[s], cudaEventDisableTiming) == cudaSuccess;
    }
    ok = ok && cudaEventCreateWithFlags(&c->ev_fork, cudaEventDisableTiming) == cudaSuccess;
    ok = ok && cudaEventCreateWithFlags(&c->ev_post, cudaEventDisableTiming) == cudaSuccess;
    ok = ok && cudaEventCreateWithFlags(&c->ev_xpost, cudaEventDisableTiming) == cudaSuccess;
    ok = ok && cudaEventCreateWithFlags(&c->ev_early0, cudaEventDisableTiming) == cudaSuccess;
    ok = ok && cudaEventCreateWithFlags(&c->ev_mid, cudaEventDisableTiming) == cudaSuccess;
    // the side chain (Kuu + jitter I) yields to the main chain (posterior, site update) where they meet, and both outrank the slabs
    const int prio_mid = prio_high < prio_low - 1 ? prio_high + 1 : prio_high;
    ok = ok && cudaStreamCreateWithPriority(&c->s_side, cudaStreamNonBlocking, prio_mid) == cudaSuccess;
    for (CholAux* a : {&c->la_main, &c->la_side}) {
        ok = ok && cudaStreamCreateWithPriority(&a->s2, cudaStreamNonBlocking, a == &c->la_main ? prio_high : prio_mid) == cudaSuccess;
        ok = ok && cudaEventCreateWithFlags(&a->e, cudaEventDisableTiming) == cudaSuccess;
        ok = ok && cudaEventCreateWithFlags(&a->f, cudaEventDisableTiming) == cudaSuccess;
    }
    ok = ok && cudaEventCreateWithFlags(&c->ev_kuu, cudaEventDisableTiming) == cudaSuccess;
    ok = ok && cudaEventCreateWithFlags(&c->ev_side, cudaEventDisableTiming) == cudaSuccess;
    for (int i = 0; i < N_EV && ok; ++i) ok = ok && cudaEventCreate(&c->ev[i]) == cudaSuccess;
    ok = ok && gemm_init() == 0 && diag_init() == 0 && dense_init() == 0;
    if (!ok) {
        g_create_error = std::string("CUDA initialisation failed: ") + cudaGetErrorString(cudaGetLastError());
        delete c;
        return TSVGP_ERR_CUDA;
    }
    *out = c;
    return TSVGP_OK;
}

void tsvgp_destroy(tsvgp_ctx* c) {
    if (!c) return;
    cudaSetDevice(c->dev);
    cudaDeviceSynchronize();
    if (c->comm) nccl_api().CommDestroy(c->comm);
    c->pm.release(); c->pd.release(); c->pc.release(); c->ps.release(); c->pxs.release(); c->pyt.release(); c->pmc.release();
    c->pks.release();
    if (c->s_copy) cudaStreamDestroy(c->s_copy);
    if (c->ev_copy) cudaEventDestroy(c->ev_copy);
    for (int s = 0; s < MAXS; ++s) {
        if (c->s_pp[s]) cudaStreamDestroy(c->s_pp[s]);
        if (c->ev_join[s]) cudaEventDestroy(c->ev_join[s]);
    }
    if (c->ev_fork) cudaEventDestroy(c->ev_fork);
    if (c->ev_post) cudaEventDestroy(c->ev_post);
    if (c->ev_xpost) cudaEventDestroy(c->ev_xpost);
    if (c->ev_early0) cudaEventDestroy(c->ev_early0);
    if (c->ev_mid) cudaEventDestroy(c->ev_mid);
    if (c->ev_kuu) cudaEventDestroy(c->ev_kuu);
    if (c->ev_side) cudaEventDestroy(c->ev_side);
    if (c->s_side) cudaStreamDestroy(c->s_side);
    for (CholAux* a : {&c->la_main, &c->la_side}) {
        if (a->s2) cudaStreamDestroy(a->s2);
        if (a->e) cudaEventDestroy(a->e);
        if (a->f) cudaEventDestroy(a->f);
    }
    for (cudaEvent_t e : c->pev) cudaEventDestroy(e);
    for (int i = 0; i < 2; ++i)
        if (c->ev_sw[i]) cudaEventDestroy(c->ev_sw[i]);
    for (int i = 0; i < N_EV; ++i)
        if (c->ev[i]) cudaEventDestroy(c->ev[i]);
    if (c->s_main) cudaStreamDestroy(c->s_main);
    delete c;
}

const char* tsvgp_last_error(const tsvgp_ctx* c) { return c ? c->err.c_str() : g_create_error.c_str(); }
int tsvgp_last_info(const tsvgp_ctx* c) { return c ? c->last_info : 0; }

int tsvgp_set_option(tsvgp_ctx* c, const char* name, double value) {
    if (!c || !name) return TSVGP_ERR_INVALID;
    if (!strcmp(name, "chunk")) { c->chunk_opt = (long)value; return TSVGP_OK; }
    if (!strcmp(name, "streams")) { c->n_streams = value < 1 ? 1 : (value > MAXS ? MAXS : (int)value); return TSVGP_OK; }
    if (!strcmp(name, "route")) {
        if (value != ROUTE_AUTO && value != ROUTE_FUSED && value != ROUTE_WHITENED && value != ROUTE_EXACT)
            FAIL(TSVGP_ERR_INVALID, "route must be 0 (auto), 1 (fused), 2 (whitened) or 3 (exact)");
        c->route_opt = (int)value; c->k9_valid = false; return TSVGP_OK;
    }
    if (!strcmp(name, "mc_seed")) { c->mc_seed = (unsigned long long)value; c->mc_draw = 0; return TSVGP_OK; }
    if (!strcmp(name, "sample_seed")) { c->sample_seed = (unsigned long long)value; c->sample_draw = 0; return TSVGP_OK; }
    if (!strcmp(name, "speculate")) { c->speculate = value != 0.0; return TSVGP_OK; }
    if (!strcmp(name, "k9_defer")) { c->k9_defer = value != 0.0; return TSVGP_OK; }
    if (!strcmp(name, "early_slabs")) { c->early_slabs = value < 0 ? 0 : (int)value; return TSVGP_OK; }
    if (!strcmp(name, "route_cond_max")) { c->route_cond_max = value; return TSVGP_OK; }
    if (!strcmp(name, "route_exact_min")) { c->route_exact_min = value; return TSVGP_OK; }
    if (!strcmp(name, "white")) {   // switch the context to the whitened sibling model (resets the sites to its defaults)
        c->white = value != 0.0;
        c->sites_set = false;
        c->post_valid = c->kl_valid = c->wpost_valid = c->wkl_valid = false;
        return TSVGP_OK;
    }
    if (!strcmp(name, "dist_min_m")) { c->dist_min_m = (int)value; return TSVGP_OK; }
    if (!strcmp(name, "shard_min_m")) { c->shard_min_m = (int)value; return TSVGP_OK; }
    if (!strcmp(name, "split_chains")) { c->split_chains = value != 0.0; return TSVGP_OK; }
    if (!strcmp(name, "async_issue")) { c->async_issue = value != 0.0; return TSVGP_OK; }
    if (!strcmp(name, "fuse_b")) { c->fuse_b = value != 0.0; return TSVGP_OK; }
    if (!strcmp(name, "spread_b")) { c->spread_b = value != 0.0; return TSVGP_OK; }
    if (!strcmp(name, "balance")) { c->balance = value != 0.0; return TSVGP_OK; }
    if (!strcmp(name, "profile")) { c->profile = value != 0.0; return TSVGP_OK; }
    if (!strcmp(name, "cache_factors")) { c->cache_factors = value != 0.0; return TSVGP_OK; }
    if (!strcmp(name, "invalidate")) { c->kuu_valid = c->post_valid = c->kl_valid = c->k9_valid = c->c6_valid = c->wpost_valid = c->wkl_valid = false; return TSVGP_OK; }
    FAIL(TSVGP_ERR_INVALID, "unknown option '%s'", name);
}

int tsvgp_set_num_latent(tsvgp_ctx* c, int L) {
    if (!c) return TSVGP_ERR_INVALID;
    if (L < 1 || L > MAX_LATENT) FAIL(TSVGP_ERR_INVALID, "num_latent_gps must be in [1, %d]", MAX_LATENT);
    if (L == c->L) return TSVGP_OK;
    CU(cudaSetDevice(c->dev));
    CU(cudaDeviceSynchronize());
    if (c->sep) {   // the per-latent kernels no longer match: compute calls wait for the next set_kernels / set_kernel
        OK(drop_separate(c));
        c->kern_kind = -1;
    }
    c->L = L;
    c->k9_pending = false;
    if (c->M > 0) {   // re-allocate the per-latent state; the inducing inputs survive on the host side of the caller: re-upload needed
        std::vector<double> Z((size_t)c->M * c->D), mz(c->Mp);
        CU(cudaMemcpy(Z.data(), c->Zraw, sizeof(double) * c->M * c->D, cudaMemcpyDeviceToHost));
        CU(cudaMemcpy(mz.data(), c->meanZ_off, sizeof(double) * c->Mp, cudaMemcpyDeviceToHost));
        const int M = c->M, D = c->D;
        OK(alloc_m_state(c, M, D));
        CU(cudaMemcpy(c->Zraw, Z.data(), sizeof(double) * M * D, cudaMemcpyHostToDevice));
        CU(cudaMemcpy(c->meanZ_off, mz.data(), sizeof(double) * c->Mp, cudaMemcpyHostToDevice));
    }
    c->X = nullptr;   // the resident Y layout depends on L: set the data again
    c->y_cols = 1;
    return TSVGP_OK;
}

int tsvgp_set_mc_epsilon(tsvgp_ctx* c, const double* eps, int S, int64_t N, int L) {
    if (!c) return TSVGP_ERR_INVALID;
    CU(cudaSetDevice(c->dev));
    CU(cudaStreamSynchronize(c->s_main));
    c->pmc.release();
    c->mc_eps = nullptr; c->mc_eps_n = 0;
    if (!eps) return TSVGP_OK;
    if (S != c->lik.n_gh || L != c->L || N < 1) FAIL(TSVGP_ERR_INVALID, "epsilon must be [S = %d, N, L = %d]", c->lik.n_gh, c->L);
    NEED(c->mc_eps = c->pmc.get((size_t)S * N * L));
    CU(cudaMemcpy(c->mc_eps, eps, sizeof(double) * S * N * L, cudaMemcpyDefault));
    c->mc_eps_n = N;
    return TSVGP_OK;
}

int tsvgp_num_latent(const tsvgp_ctx* c) { return c ? c->L : 0; }

static int check_kernel(tsvgp_ctx* c, int kind, double variance, const double* lengthscales, int n_ls) {
    if (kind != TSVGP_KERNEL_SE && kind != TSVGP_KERNEL_MATERN52 && kind != TSVGP_KERNEL_MATERN12 && kind != TSVGP_KERNEL_MATERN32)
        FAIL(TSVGP_ERR_INVALID, "unknown kernel kind %d", kind);
    if (!lengthscales || n_ls < 1 || !(variance > 0.0)) FAIL(TSVGP_ERR_INVALID, "kernel needs variance > 0 and >= 1 lengthscale");
    for (int i = 0; i < n_ls; ++i)
        if (!(lengthscales[i] > 0.0)) FAIL(TSVGP_ERR_INVALID, "lengthscales must be positive");
    return TSVGP_OK;
}

int tsvgp_set_kernel(tsvgp_ctx* c, int kind, double variance, const double* lengthscales, int n_ls) {
    if (!c) return TSVGP_ERR_INVALID;
    OK(check_kernel(c, kind, variance, lengthscales, n_ls));
    if (c->sep) {
        CU(cudaSetDevice(c->dev));
        OK(drop_separate(c));
    }
    c->kern_kind = kind; c->kern_var = variance;
    c->ls_host.assign(lengthscales, lengthscales + n_ls);
    c->kuu_valid = c->post_valid = c->kl_valid = c->k9_valid = c->c6_valid = c->wpost_valid = c->wkl_valid = false;
    c->xs_valid = false;
    return TSVGP_OK;
}

int tsvgp_set_kernels(tsvgp_ctx* c, const int* kinds, const double* variances, const double* lengthscales, const int* n_ls) {
    if (!c) return TSVGP_ERR_INVALID;
    if (!kinds || !variances || !lengthscales || !n_ls) FAIL(TSVGP_ERR_INVALID, "kinds, variances, lengthscales and n_ls are required");
    std::vector<tsvgp_ctx::KernelState> ks(c->L);
    const double* ls = lengthscales;
    for (int l = 0; l < c->L; ++l) {
        OK(check_kernel(c, kinds[l], variances[l], ls, n_ls[l]));
        ks[l].kind = kinds[l]; ks[l].var = variances[l];
        ks[l].ls.assign(ls, ls + n_ls[l]);
        ls += n_ls[l];
    }
    CU(cudaSetDevice(c->dev));
    const bool fresh = !c->sep || (int)c->lk.size() != c->L;
    if (fresh) {
        CU(cudaDeviceSynchronize());
        c->sep = true;
        c->lk = std::move(ks);
        c->ks_Mp = 0;
        if (c->M > 0) OK(alloc_separate(c));
    } else {   // same latents: keep the buffers, take the new parameters
        for (int l = 0; l < c->L; ++l) { c->lk[l].kind = ks[l].kind; c->lk[l].var = ks[l].var; c->lk[l].ls = ks[l].ls; }
    }
    if (c->M > 0) select_latent(c, 0);
    c->kern_kind = c->lk[0].kind; c->kern_var = c->lk[0].var;
    c->kuu_valid = c->post_valid = c->kl_valid = c->k9_valid = c->c6_valid = c->wpost_valid = c->wkl_valid = false;
    c->xs_valid = false;
    return TSVGP_OK;
}

int tsvgp_set_likelihood(tsvgp_ctx* c, int kind, double p0, double p1, int n_gh, const double* gh_x, const double* gh_w) {
    if (!c) return TSVGP_ERR_INVALID;
    if (kind < TSVGP_LIK_GAUSSIAN || kind > TSVGP_LIK_HETEROSKEDASTIC) FAIL(TSVGP_ERR_INVALID, "unknown likelihood kind %d", kind);
    if (kind == TSVGP_LIK_HETEROSKEDASTIC && p0 != 0.0 && p0 != 1.0)
        FAIL(TSVGP_ERR_INVALID, "heteroskedastic: p0 selects the scale transform, 0 (exp) or 1 (softplus)");
    if (kind == TSVGP_LIK_SOFTMAX) {   // p0 = number of classes (= latent GPs), n_gh = Monte-Carlo points per data point
        if (p0 < 2 || p0 > MAX_SOFTMAX_CLASSES || n_gh < 1) FAIL(TSVGP_ERR_INVALID, "Softmax: 2..%d classes and >= 1 Monte-Carlo point", MAX_SOFTMAX_CLASSES);
        c->lik.kind = kind; c->lik.p0 = p0; c->lik.p1 = 0.0; c->lik.n_gh = n_gh;
        c->lik_set = true;
        return TSVGP_OK;
    }
    if (kind != TSVGP_LIK_BERNOULLI_PROBIT && kind != TSVGP_LIK_HETEROSKEDASTIC && !(p0 > 0.0)) FAIL(TSVGP_ERR_INVALID, "likelihood variance / scale must be positive");
    if (kind == TSVGP_LIK_STUDENT_T && !(p1 > 0.0)) FAIL(TSVGP_ERR_INVALID, "Student-t df must be positive");
    if (kind != TSVGP_LIK_GAUSSIAN && (n_gh < 1 || n_gh > MAX_GH)) FAIL(TSVGP_ERR_INVALID, "n_gh must be in [1, %d]", MAX_GH);
    c->lik.kind = kind; c->lik.p0 = p0; c->lik.p1 = p1; c->lik.n_gh = kind == TSVGP_LIK_GAUSSIAN ? 0 : n_gh;
    if (kind == TSVGP_LIK_STUDENT_T)   // gpflow.logdensities.student_t constant
        c->lik.c0 = lgamma((p1 + 1.0) * 0.5) - lgamma(p1 * 0.5) - 0.5 * (log(p0 * p0) + log(p1) + log(M_PI));
    if (kind != TSVGP_LIK_GAUSSIAN) {
        double x[MAX_GH], w[MAX_GH];
        if (gh_x && gh_w) { memcpy(x, gh_x, sizeof(double) * n_gh); memcpy(w, gh_w, sizeof(double) * n_gh); }
        else gauss_hermite(n_gh, x, w);
        for (int k = 0; k < n_gh; ++k) {   // gpflow.quadrature.gauss_hermite: nodes sqrt(2) x_k, weights w_k / sqrt(pi)
            c->gh.z[k] = x[k] * sqrt(2.0);
            c->gh.w[k] = w[k] / sqrt(M_PI);
        }
    }
    c->lik_set = true;
    return TSVGP_OK;
}

int tsvgp_set_inducing(tsvgp_ctx* c, const double* Z, int M, int D, const double* mean_Z) {
    if (!c) return TSVGP_ERR_INVALID;
    if (!Z || M < 1 || D < 1) FAIL(TSVGP_ERR_INVALID, "Z must be [M >= 1, D >= 1]");
    CU(cudaSetDevice(c->dev));
    if (M != c->M || D != c->D) {
        CU(cudaDeviceSynchronize());
        c->k9_pending = false;
        OK(alloc_m_state(c, M, D));
    }
    CU(cudaMemcpyAsync(c->Zraw, Z, sizeof(double) * (size_t)M * D, cudaMemcpyDefault, c->s_main));
    c->has_meanZ = mean_Z != nullptr;
    if (mean_Z) {
        CU(cudaMemsetAsync(c->meanZ_off, 0, sizeof(double) * c->Mp, c->s_main));
        CU(cudaMemcpyAsync(c->meanZ_off, mean_Z, sizeof(double) * M, cudaMemcpyDefault, c->s_main));
    }
    CU(cudaStreamSynchronize(c->s_main));
    c->kuu_valid = c->post_valid = c->kl_valid = c->k9_valid = c->c6_valid = c->wpost_valid = c->wkl_valid = false;
    return TSVGP_OK;
}

int tsvgp_set_sites(tsvgp_ctx* c, const double* lambda_1, const double* lambda_2_sqrt) {
    if (!c) return TSVGP_ERR_INVALID;
    if (c->M <= 0) FAIL(TSVGP_ERR_STATE, "inducing points not set (tsvgp_set_inducing)");
    CU(cudaSetDevice(c->dev));
    cudaStream_t s = c->s_main;
    if (!c->sites_set || (!lambda_1 && !lambda_2_sqrt)) OK(default_sites(c));
    // layouts of the reference: lambda_1 [M, L] (sites.py:56), lambda_2_sqrt [L, M, M] (sites.py:63)
    const size_t mm = (size_t)c->Mp * c->Mp;
    if (lambda_1) {
        CU(cudaMemsetAsync(c->lam1_all, 0, sizeof(double) * c->Mp * c->L, s));
        for (int l = 0; l < c->L; ++l)
            CU(cudaMemcpy2DAsync(c->lam1_all + (size_t)l * c->Mp, sizeof(double), lambda_1 + l, sizeof(double) * c->L, sizeof(double), c->M,
                                 cudaMemcpyDefault, s));
    }
    if (lambda_2_sqrt) {
        CU(cudaMemsetAsync(c->L2_all, 0, sizeof(double) * mm * c->L, s));
        for (int l = 0; l < c->L; ++l) {
            double* L2l = c->L2_all + l * mm;
            CU(cudaMemcpy2DAsync(L2l, sizeof(double) * c->Mp, lambda_2_sqrt + (size_t)l * c->M * c->M, sizeof(double) * c->M,
                                 sizeof(double) * c->M, c->M, cudaMemcpyDefault, s));
            if (!c->white) LA(zero_upper_launch(L2l, c->Mp, c->Mp, s));   // sites.py:63 — the triangular() transform keeps the lower triangle
        }
    }
    CU(cudaStreamSynchronize(s));
    c->sites_set = true;
    c->post_valid = c->kl_valid = c->wpost_valid = c->wkl_valid = false;
    return TSVGP_OK;
}

int tsvgp_get_sites(tsvgp_ctx* c, double* lambda_1, double* lambda_2_sqrt) {
    if (!c) return TSVGP_ERR_INVALID;
    if (c->M <= 0) FAIL(TSVGP_ERR_STATE, "inducing points not set (tsvgp_set_inducing)");
    CU(cudaSetDevice(c->dev));
    if (!c->sites_set) OK(default_sites(c));
    cudaStream_t s = c->s_main;
    const size_t mm = (size_t)c->Mp * c->Mp;
    for (int l = 0; l < c->L; ++l) {
        if (lambda_1)
            CU(cudaMemcpy2DAsync(lambda_1 + l, sizeof(double) * c->L, c->lam1_all + (size_t)l * c->Mp, sizeof(double), sizeof(double), c->M,
                                 cudaMemcpyDefault, s));
        if (lambda_2_sqrt)
            CU(cudaMemcpy2DAsync(lambda_2_sqrt + (size_t)l * c->M * c->M, sizeof(double) * c->M, c->L2_all + l * mm, sizeof(double) * c->Mp,
                                 sizeof(double) * c->M, c->M, cudaMemcpyDefault, s));
    }
    CU(cudaStreamSynchronize(s));
    return TSVGP_OK;
}

int tsvgp_get_lambda_2(tsvgp_ctx* c, double* lambda_2) {
    if (!c || !lambda_2) return TSVGP_ERR_INVALID;
    if (c->M <= 0) FAIL(TSVGP_ERR_STATE, "inducing points not set (tsvgp_set_inducing)");
    CU(cudaSetDevice(c->dev));
    if (!c->sites_set) OK(default_sites(c));
    cudaStream_t s = c->s_main;
    const int n = c->Mp;
    if (c->white) {   // the whitened sibling stores Lambda_2 itself, [L, M, M]
        for (int l = 0; l < c->L; ++l)
            CU(cudaMemcpy2DAsync(lambda_2 + (size_t)l * c->M * c->M, sizeof(double) * c->M, c->L2_all + (size_t)l * n * n, sizeof(double) * n,
                                 sizeof(double) * c->M, c->M, cudaMemcpyDefault, s));
        CU(cudaStreamSynchronize(s));
        return TSVGP_OK;
    }
    for (int l = 0; l < c->L; ++l) {   // [L, M, M]
        const double* L2l = c->L2_all + (size_t)l * n * n;
        GemmP p;   // L2 L2^T (tsvgp.py:197-200), lower tiles then mirrored
        p.A = L2l; p.lda = n; p.a_kc = 1; p.a_tri = 1;
        p.B = L2l; p.ldb = n; p.b_kc = 1; p.b_tri = 1;
        p.C = c->X2; p.ldc = n; p.m = p.n = p.k = n; p.lower_out = 1;
        LA(mm_gemm(c, p, s));
        LA(mirror_lower_launch(c->X2, n, n, s));
        CU(cudaMemcpy2DAsync(lambda_2 + (size_t)l * c->M * c->M, sizeof(double) * c->M, c->X2, sizeof(double) * n, sizeof(double) * c->M, c->M,
                             cudaMemcpyDefault, s));
    }
    CU(cudaStreamSynchronize(s));
    return TSVGP_OK;
}

int tsvgp_set_data(tsvgp_ctx* c, const double* X, const double* Y, int64_t N, int D, const double* mean_X) {
    if (!c) return TSVGP_ERR_INVALID;
    if (!X || !Y || N < 1) FAIL(TSVGP_ERR_INVALID, "X [N >= 1, D] and Y [N] are required");
    if (c->D > 0 && D != c->D) FAIL(TSVGP_ERR_INVALID, "X has D=%d but the inducing points have D=%d", D, c->D);
    CU(cudaSetDevice(c->dev));
    cudaStream_t s = c->s_main;
    const long npad = round_up(N, 128);
    // Y is [N, L] for L latents with independent likelihood terms (tsvgp.py:256-259 sums over the latent axis), [N, 1] class labels
    // for the Softmax likelihood (set the likelihood before the data)
    const int ycols = (c->L > 1 && !coupled(c)) ? c->L : 1;
    if (npad > c->cap_n || (long)N * D > c->cap_x || ycols > c->cap_yc) {   // (re)allocate the owned staging and scaled-coordinate buffers
        CU(cudaStreamSynchronize(s));
        c->pd.release();
        c->cap_n = npad; c->cap_x = (long)N * D; c->cap_yc = ycols;
        NEED(c->Xown = c->pd.get((size_t)N * D)); NEED(c->Yown = c->pd.get((size_t)npad * ycols)); NEED(c->meanXown = c->pd.get(npad));
    }
    if (npad > c->xs_cap_n || (long)D * npad > c->xs_cap) {
        CU(cudaStreamSynchronize(s));
        c->pxs.release();
        c->xs_cap_n = npad; c->xs_cap = (long)D * npad;
        NEED(c->XsT = c->pxs.get((size_t)D * npad)); NEED(c->x2 = c->pxs.get(npad));
    }
    if (is_device_ptr(X)) c->X = X;
    else { CU(cudaMemcpyAsync(c->Xown, X, sizeof(double) * (size_t)N * D, cudaMemcpyHostToDevice, s)); c->X = c->Xown; }
    if (is_device_ptr(Y)) c->Y = Y;
    else { CU(cudaMemcpyAsync(c->Yown, Y, sizeof(double) * N * ycols, cudaMemcpyHostToDevice, s)); c->Y = c->Yown; }
    c->y_cols = ycols;
    if (ycols > 1) {   // latent-major copy: every latent's point kernel reads its own contiguous column
        if ((long)npad * ycols > c->yt_cap) {
            CU(cudaStreamSynchronize(s));
            c->pyt.release();
            c->yt_cap = (long)npad * ycols;
            NEED(c->Yt = c->pyt.get((size_t)c->yt_cap));
        }
        LA(transpose_to_latent_major_launch(c->Y, N, ycols, c->Yt, npad, s));
    }
    if (!mean_X) c->meanX = nullptr;
    else if (is_device_ptr(mean_X)) c->meanX = mean_X;
    else { CU(cudaMemcpyAsync(c->meanXown, mean_X, sizeof(double) * N, cudaMemcpyHostToDevice, s)); c->meanX = c->meanXown; }
    c->N = N; c->n_pad = npad;
    c->dataD = D;
    c->xs_valid = false;
    return TSVGP_OK;
}

int tsvgp_stage_data(tsvgp_ctx* c, const double* X, const double* Y, int64_t N, int D, const double* mean_X) {
    if (!c) return TSVGP_ERR_INVALID;
    if (c->L > 1 && !coupled(c)) FAIL(TSVGP_ERR_INVALID, "stage_data with num_latent_gps > 1: use set_data");
    if (!X || !Y || N < 1) FAIL(TSVGP_ERR_INVALID, "X [N >= 1, D] and Y [N] are required");
    if (c->D > 0 && D != c->D) FAIL(TSVGP_ERR_INVALID, "X has D=%d but the inducing points have D=%d", D, c->D);
    CU(cudaSetDevice(c->dev));
    if (!c->s_copy) {
        CU(cudaStreamCreateWithFlags(&c->s_copy, cudaStreamNonBlocking));
        CU(cudaEventCreateWithFlags(&c->ev_copy, cudaEventDisableTiming));
    }
    const long npad = round_up(N, 128);
    if (npad > c->st_cap_n || (long)N * D > c->st_cap_x) {
        CU(cudaStreamSynchronize(c->s_copy));
        c->ps.release();
        c->st_cap_n = npad; c->st_cap_x = (long)N * D;
        NEED(c->Xst = c->ps.get((size_t)N * D)); NEED(c->Yst = c->ps.get(npad)); NEED(c->meanXst = c->ps.get(npad));
    }
    CU(cudaMemcpyAsync(c->Xst, X, sizeof(double) * (size_t)N * D, cudaMemcpyDefault, c->s_copy));
    CU(cudaMemcpyAsync(c->Yst, Y, sizeof(double) * N, cudaMemcpyDefault, c->s_copy));
    if (mean_X) CU(cudaMemcpyAsync(c->meanXst, mean_X, sizeof(double) * N, cudaMemcpyDefault, c->s_copy));
    CU(cudaEventRecord(c->ev_copy, c->s_copy));
    c->st_N = N; c->st_D = D; c->st_has_mean = mean_X != nullptr; c->st_ready = true;
    return TSVGP_OK;
}

int tsvgp_commit_staged(tsvgp_ctx* c) {
    if (!c) return TSVGP_ERR_INVALID;
    if (!c->st_ready) FAIL(TSVGP_ERR_STATE, "no staged minibatch (tsvgp_stage_data)");
    CU(cudaSetDevice(c->dev));
    CU(cudaStreamWaitEvent(c->s_main, c->ev_copy, 0));
    // the staged buffers become the resident ones; the old resident buffers become the next staging area
    std::swap(c->Xown, c->Xst); std::swap(c->Yown, c->Yst); std::swap(c->meanXown, c->meanXst);
    std::swap(c->cap_x, c->st_cap_x);
    std::swap(c->pd.ptrs, c->ps.ptrs);
    const long npad = round_up(c->st_N, 128);
    // XsT / x2 stay with the context (pool pd owned them before the swap): re-home them if their capacity is too small
    if (npad > c->xs_cap_n || (long)c->st_D * npad > c->xs_cap) {
        CU(cudaStreamSynchronize(c->s_main));
        c->pxs.release();
        c->xs_cap_n = npad; c->xs_cap = (long)c->st_D * npad;
        NEED(c->XsT = c->pxs.get((size_t)c->st_D * npad)); NEED(c->x2 = c->pxs.get(npad));
    }
    std::swap(c->cap_n, c->st_cap_n);
    c->X = c->Xown; c->Y = c->Yown; c->meanX = c->st_has_mean ? c->meanXown : nullptr;
    c->N = c->st_N; c->n_pad = npad; c->dataD = c->st_D;
    c->xs_valid = false;
    c->st_ready = false;
    return TSVGP_OK;
}

static int require_model(tsvgp_ctx* c, bool need_data) {
    if (c->kern_kind < 0) FAIL(TSVGP_ERR_STATE, "kernel not set (tsvgp_set_kernel)");
    if (!c->lik_set) FAIL(TSVGP_ERR_STATE, "likelihood not set (tsvgp_set_likelihood)");
    if (c->M <= 0) FAIL(TSVGP_ERR_STATE, "inducing points not set (tsvgp_set_inducing)");
    if (need_data && !c->X) FAIL(TSVGP_ERR_STATE, "no data resident (tsvgp_set_data)");
    if (c->lik.kind == LIK_SOFTMAX && (int)c->lik.p0 != c->L)
        FAIL(TSVGP_ERR_INVALID, "Softmax with %d classes needs num_latent_gps = %d (tsvgp_set_num_latent), not %d", (int)c->lik.p0, (int)c->lik.p0, c->L);
    if (c->white && c->lik.kind == LIK_SOFTMAX) FAIL(TSVGP_ERR_INVALID, "the whitened sibling model is not built for the Softmax likelihood");
    if (c->lik.kind == LIK_HETEROSKEDASTIC && c->L != 2)
        FAIL(TSVGP_ERR_INVALID, "the heteroskedastic likelihood needs num_latent_gps = 2 (loc, scale), not %d", c->L);
    if (c->white && c->lik.kind == LIK_HETEROSKEDASTIC)
        FAIL(TSVGP_ERR_INVALID, "the whitened sibling model is not built for the heteroskedastic likelihood");
    if (c->white && c->sep) FAIL(TSVGP_ERR_INVALID, "the whitened sibling model is not built for separate kernels per latent");
    if (need_data && c->y_cols != ((c->L > 1 && !coupled(c)) ? c->L : 1))
        FAIL(TSVGP_ERR_STATE, "the resident Y has %d column(s): set the likelihood and num_latent_gps before the data", c->y_cols);
    return TSVGP_OK;
}

int tsvgp_natgrad_step(tsvgp_ctx* c, double lr, double jitter, double scale, double* elbo_before) {
    if (!c) return TSVGP_ERR_INVALID;
    OK(require_model(c, true));
    CU(cudaSetDevice(c->dev));
    cudaStream_t s = c->s_main;
    const long launches0 = g_launches;
    const size_t mm = (size_t)c->Mp * c->Mp;
    CU(cudaMemsetAsync(c->info, 0, sizeof(int) * N_INFO, s));
    CU(cudaEventRecord(c->ev[EV_T0], s));
    c->collective_ok = true;
    OK(ensure_xs(c));
    OK(ensure_kuu(c));
    int chain_role = 0;   // ROLE_*: 0 both chains here; 1 / 2: this rank built the posterior factors / the K9 chain; 3: neither (received both)
    {
        SideIssue side;
        struct PdlGuard { ~PdlGuard() { g_pdl_suspended = 0; } } pdl_guard;
        const bool k9_runs = !k9_cached(c, jitter);
        int rc = TSVGP_OK;
        // When is the K9 chain joined?  The fused route needs nothing of it inside the pass, so if the route is fused — forced, or
        // SPECULATED from this context's last conditioning estimate — the chain runs underneath the pass and is joined after it
        // (where the probe is read and the guess checked).  Whitened / exact passes need C9^-1: join first, as does a first step.
        bool join_before = true;
        if (k9_runs && (c->route_opt == ROUTE_FUSED ||
                        (c->route_opt == ROUTE_AUTO && c->speculate && c->cond_hint_valid && route_for(c, c->cond_hint) == ROUTE_FUSED))) {
            c->route = ROUTE_FUSED;
            join_before = false;
        }
        // ... and when does it start?  Side by side with the posterior chain the two latency-bound chains slow each other down
        // (measured at M = 2048: posterior chain 2.6 ms alone, 3.4 ms beside the K9 chain, programmatic launch suspended).  When the
        // chain is only needed after the pass it therefore starts once the posterior chain is complete and runs under the pass.
        // several ranks: the two chains are split over the ranks of a pair and exchanged (chain_split_active)
        const bool split = k9_runs && !join_before && c->sites_set && chain_split_active(c);
        chain_role = split ? chain_role_of(c) : ROLE_BOTH;
        const bool k9_here = chain_role == ROLE_BOTH || chain_role == ROLE_K9, post_here = chain_role == ROLE_BOTH || chain_role == ROLE_POSTERIOR;
        const bool defer_k9 = k9_runs && !join_before && c->k9_defer && c->Mp >= 2048 && !split;
        if (c->Mp >= 2048 && k9_runs && !defer_k9 && !split) g_pdl_suspended = 1;   // two concurrent chains of large kernels: see common.cuh
        if (!defer_k9 && k9_here) rc = start_k9_async(c, jitter, side);
        if (rc == TSVGP_OK && !k9_runs) rc = choose_route(c, jitter);   // cached factors: the route is known at once
        c->n_early = 0;
        // split chains: no early slabs on the rank that builds the posterior factors — every rank waits for that chain
        const bool early = rc == TSVGP_OK && c->early_slabs && (!k9_runs || !join_before) && c->route == ROUTE_FUSED && (!split || !post_here);
        if (early) rc = data_pass(c, MODE_STATS, PASS_EARLY);
        if (rc == TSVGP_OK && post_here) rc = ensure_posterior(c);
        if (rc == TSVGP_OK && post_here && elbo_before) rc = ensure_kl_terms(c);
        if (rc == TSVGP_OK && split) {
            // a receiver's broadcast kernel polls on SMs until rank 0 delivers: it is launched when the first early slab is done
            // (one slab's Kuf + SYRK is about as long as the posterior chain), not underneath it
            if (!post_here && c->n_early > 0) CU(cudaStreamWaitEvent(s, c->ev_early0, 0));
            rc = exchange_posterior(c, elbo_before != nullptr);   // rank 0: behind its chain; the others receive
        }
        if (rc == TSVGP_OK && defer_k9) rc = start_k9(c, jitter);   // forks from the main stream HERE: behind the posterior chain
        side.join_into(g_launches);
        if (rc != TSVGP_OK) return rc;
        if (side.rc != TSVGP_OK) return side.rc;
        if (k9_runs && join_before) OK(choose_route(c, jitter));
        CU(cudaEventRecord(c->ev[EV_PREP], s));
        nvtxRangePushA("tsvgp_stream");
        c->mark_mid = split;
        const int rc_pass = data_pass(c, MODE_STATS, early ? PASS_REST : PASS_WHOLE);
        c->mark_mid = false;
        nvtxRangePop();
        OK(rc_pass);
        if (split) OK(exchange_k9(c, jitter));   // second on the communicator, on the side stream, once the pass is a few slabs in
        if (k9_runs && !join_before) {   // join the K9 chain, read the probe, repeat the pass if the guess was wrong
            const int guessed = c->route;
            OK(choose_route(c, jitter));
            if (c->route != guessed)
                OK(data_pass(c, MODE_STATS));
        }
    }
    if (elbo_before && c->lik.kind == LIK_GAUSSIAN && !c->white) OK(variance_term_from_stats(c));
    CU(cudaEventRecord(c->ev[EV_STREAM], s));
    struct NvtxRange { NvtxRange(const char* n) { nvtxRangePushA(n); } ~NvtxRange() { nvtxRangePop(); } } nvtx_dense("tsvgp_dense");
    if (sharded_update_active(c)) {
        OK(sharded_reduce_and_form_G(c));   // records EV_REDUCE after the reduce-scatter
        OK(dense_update_one(c, lr, jitter, scale, false, true));
    } else {
        OK(all_reduce(c, c->stats_all[0], c->L * (mm + c->Mp + 4)));
        CU(cudaEventRecord(c->ev[EV_REDUCE], s));
        OK(dense_update(c, lr, jitter, scale, false));
    }
    CU(cudaEventRecord(c->ev[EV_DENSE], s));

    double tail[4];
    std::vector<double> scv((size_t)c->L * N_SCAL);
    double* sc = scv.data();
    int info_h[N_INFO];
    OK(read_tails(c, tail, sc, info_h));
    ++c->mc_draw;
    // the step consumed the posterior factors of the old sites
    c->post_valid = c->kl_valid = c->wpost_valid = c->wkl_valid = false;
    float ms = 0;
    for (int i = 0; i < 4; ++i) { cudaEventElapsedTime(&ms, c->ev[i], c->ev[i + 1]); c->timings[1 + i] = ms; }
    cudaEventElapsedTime(&ms, c->ev[EV_T0], c->ev[EV_DENSE]);
    c->timings[0] = ms;
    {
        const int nstr_t = c->profile ? 1 : (c->n_streams < 1 ? 1 : (c->n_streams > MAXS ? MAXS : c->n_streams));
        const long ncu_t = used_chunk(c, c->N, c->chunk, nstr_t);
        c->timings[5] = (double)((c->N + ncu_t - 1) / ncu_t);
    }
    c->timings[6] = (double)(g_launches - launches0);
    c->timings[7] = (double)c->route;
    c->timings[8] = c->cond_est;
    c->timings[9] = (double)chain_role;
    OK(check_info(c, info_h));
    if (tail[1] != 0.0) {
        c->post_valid = c->kl_valid = c->wpost_valid = c->wkl_valid = false;
        FAIL(TSVGP_ERR_NONPOSITIVE_VARIANCE, "predict_f: non-positive predictive variance (sites unchanged)");
    }
    if (elbo_before) *elbo_before = scale * tail[0] - kl_value(c, sc);
    return TSVGP_OK;
}

int tsvgp_elbo(tsvgp_ctx* c, double scale, double* out) {
    if (!c || !out) return TSVGP_ERR_INVALID;
    OK(require_model(c, true));
    CU(cudaSetDevice(c->dev));
    c->collective_ok = true;    // every rank calls elbo together (it all-reduces the expectations)
    cudaStream_t s = c->s_main;
    const size_t mm = (size_t)c->Mp * c->Mp;
    CU(cudaMemsetAsync(c->info, 0, sizeof(int) * N_INFO, s));
    OK(ensure_xs(c));
    OK(ensure_posterior(c));
    OK(ensure_kl_terms(c));
    OK(data_pass(c, MODE_ELBO));
    for (int l = 0; l < c->L; ++l) OK(all_reduce(c, c->stats_all[0] + l * (mm + c->Mp + 4) + mm + c->Mp, 4));
    double tail[4];
    std::vector<double> scv((size_t)c->L * N_SCAL);
    int info_h[N_INFO];
    OK(read_tails(c, tail, scv.data(), info_h));
    ++c->mc_draw;
    OK(check_info(c, info_h));
    if (tail[1] != 0.0) FAIL(TSVGP_ERR_NONPOSITIVE_VARIANCE, "predict_f: non-positive predictive variance");
    *out = scale * tail[0] - kl_value(c, scv.data());
    return TSVGP_OK;
}

int tsvgp_prior_kl(tsvgp_ctx* c, double* out) {
    if (!c || !out) return TSVGP_ERR_INVALID;
    OK(require_model(c, false));
    CU(cudaSetDevice(c->dev));
    c->collective_ok = false;   // may be called by one rank alone: no hidden collective (replicated products)
    cudaStream_t s = c->s_main;
    CU(cudaMemsetAsync(c->info, 0, sizeof(int) * N_INFO, s));
    OK(ensure_posterior(c));
    OK(ensure_kl_terms(c));
    std::vector<double> scv((size_t)c->L * N_SCAL);
    int info_h[N_INFO];
    CU(cudaMemcpyAsync(scv.data(), c->scal_all, sizeof(double) * N_SCAL * c->L, cudaMemcpyDeviceToHost, s));
    CU(cudaMemcpyAsync(info_h, c->info, sizeof info_h, cudaMemcpyDeviceToHost, s));
    CU(cudaStreamSynchronize(s));
    OK(check_info(c, info_h));
    *out = kl_value(c, scv.data());
    return TSVGP_OK;
}

// The dense epilogue of the gradient of ONE latent, after the pass has accumulated its statistics: *elbo = scale * sum ve_l - KL_l
// (a coupled likelihood: latent 0 carries the whole expectation and sum of h), the kernel-variance and likelihood terms, and
// F_uu = E_uu [zs | 1 | zs^2] on the host.  Reuses X1 (the KL terms are recomputed on the next call).
static int grad_epilogue(tsvgp_ctx* c, int lat, double scale, double* elbo, double* d_variance, double* d_lik, std::vector<double>& Fuu) {
    cudaStream_t s = c->s_main;
    const int n = c->Mp, M = c->M, D = c->D, W = c->waug;
    const long ld = n;
    const size_t mm = (size_t)n * n;
    select_latent(c, lat);
    OK(all_reduce(c, c->stats[0], mm + n + 4));
    double* B = c->stats[0];
    double* bvec = c->stats[0] + mm;
    LA(mirror_lower_launch(B, ld, n, s));
    {   // Q = T T^T  (symmetric, = (Lambda_2^-1 + K6)^-1)
        GemmP p;
        p.A = c->T; p.lda = ld; p.a_kc = 1; p.a_tri = 1;
        p.B = c->T; p.ldb = ld; p.b_kc = 1; p.b_tri = 1;
        p.C = c->Wm; p.ldc = ld; p.m = p.n = p.k = n; p.lower_out = 1;
        LA(mm_gemm(c, p, s));
    }
    LA(mirror_lower_launch(c->Wm, ld, n, s));
    auto full_gemm = [&](const double* A, const double* Bm, double* C) {   // C = A * Bm, all symmetric-or-full row-major
        GemmP p;
        p.A = A; p.lda = ld; p.a_kc = 1;
        p.B = Bm; p.ldb = ld; p.b_kc = 0;
        p.C = C; p.ldc = ld; p.m = p.n = p.k = n;
        return mm_gemm(c, p, s);
    };
    LA(full_gemm(c->Wm, B, c->X1));        // Q B
    LA(full_gemm(c->X1, c->Wm, c->X2));    // Q B Q
    LA(full_gemm(c->Wm, c->K6, c->G2));    // Q K6
    LA(full_gemm(c->G2, c->Wm, c->P));     // Q K6 Q
    LA(gemv_n_launch(c->Wm, ld, n, n, bvec, 1.0, 0.0, c->v1, s));     // Q b
    LA(gemv_n_launch(c->Wm, ld, n, n, c->mq, 1.0, 0.0, c->v2, s));    // Q m_q
    // dk/dr2 of Kuu (K itself is recomputed into a scratch matrix: V is not needed once T exists)
    LA(kuf_launch(c->kern_kind, c->kern_var, c->ZsT, n, c->z2, 0, M, n, c->Zs, c->z2, M, n, D, nullptr, c->V, n, nullptr, 0, 0, s, c->Wf));
    LA(gamma_uu_launch(c->X2, c->P, c->v1, c->v2, c->alpha, c->Wf, c->X1, c->G2, ld, n, scale, s));   // X1 = Gamma, G2 = E_uu
    LA(matdot_launch(c->X1, c->K, ld, n, c->scal + SC_G_K, c->red, s));
    LA(matdot_launch(c->Wm, B, ld, n, c->scal + SC_TR_QB, c->red, s));
    LA(dot_launch(c->alpha, bvec, n, c->scal + SC_A_B, s));
    LA(xaug_launch(c->ZsT, n, 0, M, n, D, c->zaug, s, c->origin));
    {   // F_uu = E_uu [zs | 1 | zs^2]
        GemmP p;
        p.A = c->G2; p.lda = ld; p.a_kc = 1;
        p.B = c->zaug; p.ldb = W; p.b_kc = 0;
        p.C = c->fuu; p.ldc = W; p.m = n; p.n = W; p.k = n;
        LA(mm_gemm(c, p, s));
    }
    Fuu.resize((size_t)n * W);
    double tail[4], sc[N_SCAL];
    int info_h[N_INFO];
    CU(cudaMemcpyAsync(Fuu.data(), c->fuu, sizeof(double) * n * W, cudaMemcpyDeviceToHost, s));
    CU(cudaMemcpyAsync(tail, c->stats[0] + mm + n, sizeof tail, cudaMemcpyDeviceToHost, s));
    CU(cudaMemcpyAsync(sc, c->scal, sizeof sc, cudaMemcpyDeviceToHost, s));
    CU(cudaMemcpyAsync(info_h, c->info, sizeof info_h, cudaMemcpyDeviceToHost, s));
    CU(cudaStreamSynchronize(s));
    c->kl_valid = false;   // X1 was reused
    OK(check_info(c, info_h));
    if (tail[1] != 0.0) FAIL(TSVGP_ERR_NONPOSITIVE_VARIANCE, "predict_f: non-positive predictive variance");
    *elbo = scale * tail[0] - 0.5 * (sc[SC_M_ALPHA] - sc[SC_TR_QK] + 2.0 * sc[SC_LOGDIAG_W]);
    *d_variance = (scale * (sc[SC_A_B] - 2.0 * sc[SC_TR_QB]) + sc[SC_G_K]) / c->kern_var + scale * tail[2];
    *d_lik = scale * tail[3];
    return TSVGP_OK;
}

// Lengthscale and Z gradients from F_uf = E_uf [xs | 1 | xs^2] (summed over the points) and F_uu (host, row stride waug):
// d r2 / d lengthscale_d = -2 delta_d^2 / l_d, d r2 / d z_id = 2 delta_d / l_d with delta = zs - xs (scaled coordinates);
// sums over points expanded through F:  sum_n E delta = zs S1 - EX ; sum E delta^2 = zs^2 S1 - 2 zs EX + C2
static int f_to_grads(tsvgp_ctx* c, const std::vector<double>& origin, const std::vector<double>& Fuf, const std::vector<double>& Fuu,
                      std::vector<double>& dls, std::vector<double>& dZ) {
    cudaStream_t s = c->s_main;
    const int n = c->Mp, M = c->M, D = c->D, W = c->waug;
    std::vector<double> Zs((size_t)n * D), ls(D);
    CU(cudaMemcpyAsync(Zs.data(), c->Zs, sizeof(double) * n * D, cudaMemcpyDeviceToHost, s));
    CU(cudaMemcpyAsync(ls.data(), c->ls_dev, sizeof(double) * D, cudaMemcpyDeviceToHost, s));
    CU(cudaStreamSynchronize(s));
    dZ.assign((size_t)M * D, 0.0);
    dls.assign(D, 0.0);
    for (int d = 0; d < D; ++d) {
        double acc = 0.0;
        for (int i = 0; i < M; ++i) {
            const double z = Zs[(size_t)i * D + d] - origin[d];   // F was accumulated in the same shifted coordinates
            const double* fu = &Fuf[(size_t)i * W];
            const double* fz = &Fuu[(size_t)i * W];
            acc += z * z * fu[D] - 2.0 * z * fu[d] + fu[D + 1 + d];
            acc += z * z * fz[D] - 2.0 * z * fz[d] + fz[D + 1 + d];
            dZ[(size_t)i * D + d] = (2.0 / ls[d]) * (z * fu[D] - fu[d]) + (4.0 / ls[d]) * (z * fz[D] - fz[d]);
        }
        dls[d] = -(2.0 / ls[d]) * acc;
    }
    return TSVGP_OK;
}

// F_uf of the last gradient pass, all-reduced over the ranks, to the host
static int read_fuf(tsvgp_ctx* c, std::vector<double>& Fuf) {
    const size_t cnt = (size_t)c->Mp * c->waug;
    OK(all_reduce(c, c->facc[0], cnt));
    Fuf.resize(cnt);
    CU(cudaMemcpyAsync(Fuf.data(), c->facc[0], sizeof(double) * cnt, cudaMemcpyDeviceToHost, c->s_main));
    CU(cudaStreamSynchronize(c->s_main));
    return TSVGP_OK;
}

// ELBO terms and gradients of ONE latent with independent likelihood terms: its own pass, then its epilogue
static int elbo_grad_one(tsvgp_ctx* c, int lat, double scale, const std::vector<double>& origin, double* elbo, double* d_variance,
                         std::vector<double>& dls, std::vector<double>& dZ, double* d_lik) {
    c->grad_scale = scale;
    OK(data_pass(c, MODE_GRAD, PASS_WHOLE, lat));
    select_latent(c, lat);
    std::vector<double> Fuf, Fuu;
    OK(read_fuf(c, Fuf));
    OK(grad_epilogue(c, lat, scale, elbo, d_variance, d_lik, Fuu));
    return f_to_grads(c, origin, Fuf, Fuu, dls, dZ);
}

// A coupled likelihood (Softmax): ONE pass over all latents (the point kernel needs every latent's moments of the same points),
// then the epilogue per latent.  Kuf is shared, so F_uf holds the sum over the latents already and the F_uu add up.
static int elbo_grad_coupled(tsvgp_ctx* c, double scale, const std::vector<double>& origin, double* elbo, double* d_variance,
                             std::vector<double>& dls, std::vector<double>& dZ, double* d_lik) {
    c->grad_scale = scale;
    OK(data_pass(c, MODE_GRAD));
    std::vector<double> Fuf, Fuu, Fuu_sum;
    OK(read_fuf(c, Fuf));
    double e_sum = 0.0, dv_sum = 0.0, dl_sum = 0.0;
    for (int l = 0; l < c->L; ++l) {
        double e = 0.0, dv = 0.0, dl = 0.0;
        OK(grad_epilogue(c, l, scale, &e, &dv, &dl, Fuu));
        if (l == 0) Fuu_sum = Fuu;
        else for (size_t i = 0; i < Fuu.size(); ++i) Fuu_sum[i] += Fuu[i];
        e_sum += e; dv_sum += dv; dl_sum += dl;
    }
    *elbo = e_sum; *d_variance = dv_sum; *d_lik = dl_sum;
    return f_to_grads(c, origin, Fuf, Fuu_sum, dls, dZ);
}

int tsvgp_elbo_grad(tsvgp_ctx* c, double scale, double* elbo, double* d_variance, double* d_lengthscales, double* d_Z, double* d_lik) {
    if (!c || !elbo || !d_variance || !d_lengthscales || !d_Z || !d_lik) return TSVGP_ERR_INVALID;
    OK(require_model(c, true));
    if (c->white) FAIL(TSVGP_ERR_INVALID, "elbo_grad is not available for the whitened sibling model");
    if (c->lik.kind == LIK_HETEROSKEDASTIC) FAIL(TSVGP_ERR_INVALID, "elbo_grad is not built for the heteroskedastic likelihood");
    if (c->sep) FAIL(TSVGP_ERR_INVALID, "elbo_grad is not built for separate kernels per latent");
    CU(cudaSetDevice(c->dev));
    c->collective_ok = true;
    cudaStream_t s = c->s_main;
    const int M = c->M, D = c->D;
    CU(cudaMemsetAsync(c->info, 0, sizeof(int) * N_INFO, s));
    OK(ensure_xs(c));
    OK(ensure_posterior(c));
    OK(ensure_kl_terms(c));
    // common origin of the scaled coordinates: the centroid of the inducing inputs (see xaug_kernel)
    std::vector<double> origin(D, 0.0);
    {
        std::vector<double> Zs((size_t)c->Mp * D);
        CU(cudaMemcpyAsync(Zs.data(), c->Zs, sizeof(double) * c->Mp * D, cudaMemcpyDeviceToHost, s));
        CU(cudaStreamSynchronize(s));
        for (int i = 0; i < M; ++i)
            for (int d = 0; d < D; ++d) origin[d] += Zs[(size_t)i * D + d] / M;
        CU(cudaMemcpyAsync(c->origin, origin.data(), sizeof(double) * D, cudaMemcpyHostToDevice, s));
        CU(cudaStreamSynchronize(s));
    }
    // the ELBO is additive over the latents (shared kernel: the expectations sum over the latent axis, the KL over the independent
    // q(u_l); tsvgp.py:65-95), and so is every gradient
    double e_sum = 0.0, dv_sum = 0.0, dl_sum = 0.0;
    std::vector<double> dls_sum(D, 0.0), dZ_sum((size_t)M * D, 0.0), dls, dZ;
    if (coupled(c)) {
        const int rc = elbo_grad_coupled(c, scale, origin, &e_sum, &dv_sum, dls_sum, dZ_sum, &dl_sum);
        select_latent(c, 0);
        if (rc != TSVGP_OK) return rc;
        ++c->mc_draw;   // one Monte-Carlo draw per call, as tsvgp_elbo: the ELBO returned here at draw k is elbo's at draw k
    } else {
        for (int l = 0; l < c->L; ++l) {
            double e = 0.0, dv = 0.0, dl = 0.0;
            const int rc = elbo_grad_one(c, l, scale, origin, &e, &dv, dls, dZ, &dl);
            select_latent(c, 0);
            if (rc != TSVGP_OK) return rc;
            e_sum += e; dv_sum += dv; dl_sum += dl;
            for (int d = 0; d < D; ++d) dls_sum[d] += dls[d];
            for (size_t i = 0; i < dZ.size(); ++i) dZ_sum[i] += dZ[i];
        }
    }
    *elbo = e_sum; *d_variance = dv_sum; *d_lik = dl_sum;
    if (c->ls_host.size() == 1) {
        double t = 0.0;
        for (int d = 0; d < D; ++d) t += dls_sum[d];
        CU(cudaMemcpy(d_lengthscales, &t, sizeof(double), cudaMemcpyDefault));
    } else {
        CU(cudaMemcpy(d_lengthscales, dls_sum.data(), sizeof(double) * D, cudaMemcpyDefault));
    }
    CU(cudaMemcpy(d_Z, dZ_sum.data(), sizeof(double) * (size_t)M * D, cudaMemcpyDefault));
    return TSVGP_OK;
}

// the query points scaled by the kernel's lengthscales; separate kernels: one copy per latent, xsT [L][D][ld], x2 [L][ld]
static int scale_query(tsvgp_ctx* c, const double* X, long N, int D, double* xsT, long ld, double* x2) {
    if (!c->sep) {
        LA(scale_points_launch(X, N, D, c->ls_dev, xsT, ld, x2, ld, c->s_main));
        return TSVGP_OK;
    }
    for (int l = 0; l < c->L; ++l)
        LA(scale_points_launch(X, N, D, c->lk[l].ls_dev, xsT + (size_t)l * D * ld, ld, x2 + (size_t)l * ld, ld, c->s_main));
    return TSVGP_OK;
}

int tsvgp_predict_f(tsvgp_ctx* c, const double* Xnew, int64_t N, int D, const double* mean_X, double* mean_out, double* var_out) {
    if (!c) return TSVGP_ERR_INVALID;
    if (!Xnew || !mean_out || !var_out || N < 1) FAIL(TSVGP_ERR_INVALID, "Xnew [N >= 1, D], mean_out [N], var_out [N] are required");
    OK(require_model(c, false));
    if (D != c->D) FAIL(TSVGP_ERR_INVALID, "Xnew has D=%d but the inducing points have D=%d", D, c->D);
    CU(cudaSetDevice(c->dev));
    c->collective_ok = false;   // predict_f needs no collective (DESIGN 6): one rank may call it alone
    cudaStream_t s = c->s_main;
    CU(cudaMemsetAsync(c->info, 0, sizeof(int) * N_INFO, s));
    OK(ensure_posterior(c));
    const long npad = round_up(N, 128);
    Pool tp;
    struct Rel { Pool& p; cudaStream_t s; ~Rel() { cudaStreamSynchronize(s); p.release(); } } rel{tp, s};
    double *xd = nullptr, *xsT, *x2, *md, *vd, *moff = nullptr;
    const double* xsrc = Xnew;
    if (!is_device_ptr(Xnew)) {
        NEED(xd = tp.get((size_t)N * D));
        CU(cudaMemcpyAsync(xd, Xnew, sizeof(double) * (size_t)N * D, cudaMemcpyHostToDevice, s));
        xsrc = xd;
    }
    const int L = c->L, nk = c->sep ? L : 1;
    NEED(xsT = tp.get((size_t)nk * D * npad)); NEED(x2 = tp.get((size_t)nk * npad)); NEED(md = tp.get((size_t)L * npad)); NEED(vd = tp.get((size_t)L * npad));
    if (mean_X) {
        NEED(moff = tp.get(npad));
        CU(cudaMemcpyAsync(moff, mean_X, sizeof(double) * N, cudaMemcpyDefault, s));
    }
    OK(scale_query(c, xsrc, N, D, xsT, npad, x2));
    OK(stream_pass(c, xsT, npad, x2, N, nullptr, moff, MODE_PREDICT, md, vd, PASS_WHOLE, 0, npad, -1, c->sep ? (long)D * npad : 0,
                   c->sep ? npad : 0));
    double tail[4];
    int info_h[N_INFO];
    if (L == 1) {
        CU(cudaMemcpyAsync(mean_out, md, sizeof(double) * N, cudaMemcpyDefault, s));
        CU(cudaMemcpyAsync(var_out, vd, sizeof(double) * N, cudaMemcpyDefault, s));
    } else {   // [L][npad] on the device -> the reference's [N, L]
        double *mt, *vt;
        NEED(mt = tp.get((size_t)N * L)); NEED(vt = tp.get((size_t)N * L));
        LA(transpose_to_point_major_launch(md, npad, N, L, mt, s));
        LA(transpose_to_point_major_launch(vd, npad, N, L, vt, s));
        CU(cudaMemcpyAsync(mean_out, mt, sizeof(double) * N * L, cudaMemcpyDefault, s));
        CU(cudaMemcpyAsync(var_out, vt, sizeof(double) * N * L, cudaMemcpyDefault, s));
    }
    OK(read_tails(c, tail, nullptr, info_h));
    OK(check_info(c, info_h));
    if (tail[1] != 0.0) FAIL(TSVGP_ERR_NONPOSITIVE_VARIANCE, "predict_f: non-positive predictive variance");
    return TSVGP_OK;
}

// The N x N path (DESIGN 13): cov_out != null -> predict_f(full_cov = True), mean_out [N, L], cov_out [L, N, N]; otherwise
// predict_f_samples, samples_out [S, N, L].  Per latent l, in one Np x Np buffer:
//   Sigma = k(X, X) (identity on the padding) ;  V = T_l^T Kuf ;  Sigma -= V^T V (lower tiles)
//   covariance: mirror, copy [0, N)^2 out ;  samples: chol(Sigma + 1e-6 I) E_l + mean
// The moments come from predict_f's own pass, so the means are predict_f's bits and the marginal variances are checked there.
static int predict_full(tsvgp_ctx* c, const double* Xnew, int64_t N, int D, const double* mean_X, double* mean_out, double* cov_out,
                        int S, int full_cov, const double* eps, double* samples_out) {
    OK(require_model(c, false));
    if (D != c->D) FAIL(TSVGP_ERR_INVALID, "Xnew has D=%d but the inducing points have D=%d", D, c->D);
    const bool want_cov = cov_out != nullptr;
    if (c->white && full_cov)
        FAIL(TSVGP_ERR_INVALID, "full_cov is not built for the whitened sibling: its conditional computes the diagonal only "
                                "(tsvgp_white.py:122-132)");
    CU(cudaSetDevice(c->dev));
    c->collective_ok = false;   // like predict_f: one rank may call it alone, so every product below stays on this GPU
    cudaStream_t s = c->s_main;
    const int L = c->L, Mp = c->Mp;
    const long Np = round_up(N, 128), Sp = want_cov ? 0 : round_up(S, 128);
    const bool x_host = !is_device_ptr(Xnew), eps_host = eps && !is_device_ptr(eps);
    const bool out_host = !want_cov && !is_device_ptr(samples_out);
    const int nk = c->sep ? L : 1;   // scaled copies of the query points (one per latent kernel)
    {   // every temporary below, counted before the first allocation
        size_t need = (size_t)nk * (D * Np + Np) + 2 * (size_t)L * Np + (mean_X ? Np : 0) + (x_host ? (size_t)N * D : 0) + (size_t)N * L;
        if (full_cov) need += (size_t)Np * D + 2 * (size_t)Mp * Np + (size_t)Np * Np;
        if (full_cov && !want_cov) need += (size_t)Np * 128 + 2 * (size_t)Np * Sp + L;
        if (eps_host) need += (size_t)S * N * L;
        if (out_host) need += (size_t)S * N * L;
        size_t free_b = 0, total_b = 0;
        CU(cudaMemGetInfo(&free_b, &total_b));
        if (need * sizeof(double) > free_b)
            FAIL(TSVGP_ERR_INVALID, "%s at N = %lld needs %zu bytes of device memory, %zu are free",
                 want_cov ? "predict_f(full_cov = True)" : "predict_f_samples", (long long)N, need * sizeof(double), free_b);
    }
    CU(cudaMemsetAsync(c->info, 0, sizeof(int) * N_INFO, s));
    OK(ensure_posterior(c));
    Pool tp;
    struct Rel { Pool& p; cudaStream_t s; ~Rel() { cudaStreamSynchronize(s); p.release(); } } rel{tp, s};
    double *xsT, *x2, *md, *vd, *moff = nullptr;
    const double* xsrc = Xnew;
    if (x_host) {
        double* xd;
        NEED(xd = tp.get((size_t)N * D));
        CU(cudaMemcpyAsync(xd, Xnew, sizeof(double) * (size_t)N * D, cudaMemcpyHostToDevice, s));
        xsrc = xd;
    }
    NEED(xsT = tp.get((size_t)nk * D * Np)); NEED(x2 = tp.get((size_t)nk * Np)); NEED(md = tp.get((size_t)L * Np)); NEED(vd = tp.get((size_t)L * Np));
    if (mean_X) {
        NEED(moff = tp.get(Np));
        CU(cudaMemcpyAsync(moff, mean_X, sizeof(double) * N, cudaMemcpyDefault, s));
    }
    OK(scale_query(c, xsrc, N, D, xsT, Np, x2));
    OK(stream_pass(c, xsT, Np, x2, N, nullptr, moff, MODE_PREDICT, md, vd, PASS_WHOLE, 0, Np, -1, c->sep ? (long)D * Np : 0,
                   c->sep ? Np : 0));   // exactly predict_f's moments

    SampleArgs sa;
    sa.eps = eps; sa.seed = c->sample_seed; sa.draw = c->sample_draw; sa.N = N; sa.S = S; sa.L = L;
    double* out_d = samples_out;
    if (!want_cov) {
        ++c->sample_draw;   // a new draw per call
        if (eps_host) {
            double* e;
            NEED(e = tp.get((size_t)S * N * L));
            CU(cudaMemcpyAsync(e, eps, sizeof(double) * (size_t)S * N * L, cudaMemcpyHostToDevice, s));
            sa.eps = e;
        }
        if (out_host) NEED(out_d = tp.get((size_t)S * N * L));
    }
    int* chol_info = nullptr;   // [L]: failing pivot of chol(Sigma_l + 1e-6 I), 1-based = query point
    if (!full_cov) {
        LA(diag_samples_launch(sa, md, vd, Np, out_d, s));
    } else {
        double *xr, *kuf, *V, *Sig, *dinv = nullptr, *E = nullptr, *F = nullptr;
        NEED(xr = tp.get((size_t)Np * D)); NEED(kuf = tp.get((size_t)Mp * Np)); NEED(V = tp.get((size_t)Mp * Np));
        NEED(Sig = tp.get((size_t)Np * Np));
        auto build_kuf = [&](const double* xs, const double* xx) -> int {   // the query points as the row operand of k(X, X); Kuf
            LA(unpack_rows_launch(xs, Np, (int)Np, D, xr, s));
            LA(kuf_launch(c->kern_kind, c->kern_var, xs, Np, xx, 0, N, (int)Np, c->Zs, c->z2, c->M, Mp, D, nullptr, kuf, Np, nullptr, 0, 0, s));
            return TSVGP_OK;
        };
        if (!c->sep) OK(build_kuf(xsT, x2));   // one kernel: built once for every latent
        if (!want_cov) {
            NEED(dinv = tp.get((size_t)Np * 128)); NEED(E = tp.get((size_t)Np * Sp)); NEED(F = tp.get((size_t)Np * Sp));
            NEED(chol_info = (int*)tp.get(L));
            CU(cudaMemsetAsync(dinv, 0, sizeof(double) * (size_t)Np * 128, s));   // contract of diag_potrf_inv_launch
            CU(cudaMemsetAsync(chol_info, 0, sizeof(int) * L, s));
        }
        for (int l = 0; l < L; ++l) {
            select_latent(c, l);
            const double* xs_l = xsT + (size_t)(c->sep ? l : 0) * D * Np;
            const double* x2_l = x2 + (size_t)(c->sep ? l : 0) * Np;
            if (c->sep) OK(build_kuf(xs_l, x2_l));   // latent l's kernel
            // Sigma = k(X, X), recomputed per latent instead of keeping a second N x N copy
            LA(kuf_launch(c->kern_kind, c->kern_var, xs_l, Np, x2_l, 0, N, (int)Np, xr, x2_l, (int)N, (int)Np, D, nullptr, Sig, Np, nullptr, 0, 1, s));
            {   // V = T^T Kuf  (the variance product of the pass, stored)
                GemmP p;
                p.A = c->T; p.lda = Mp; p.a_kc = 0; p.a_tri = 2;
                p.B = kuf; p.ldb = Np; p.b_kc = 0;
                p.C = V; p.ldc = Np; p.m = Mp; p.n = (int)Np; p.k = Mp;
                LA(mm_gemm(c, p, s));
            }
            {   // Sigma -= V^T V  (lower tiles; split-K over idle SMs when Np is small)
                GemmP p;
                p.A = V; p.lda = Np; p.a_kc = 0;
                p.B = V; p.ldb = Np; p.b_kc = 0;
                p.C = Sig; p.ldc = Np; p.m = p.n = (int)Np; p.k = Mp;
                p.alpha = -1.0; p.beta = 1.0; p.lower_out = 1;
                LA(mm_gemm(c, p, s));
            }
            if (want_cov) {
                LA(mirror_lower_launch(Sig, Np, (int)Np, s));
                CU(cudaMemcpy2DAsync(cov_out + (size_t)l * N * N, sizeof(double) * N, Sig, sizeof(double) * Np, sizeof(double) * N, N,
                                     cudaMemcpyDefault, s));
                continue;
            }
            // gpflow sample_mvn: chol(Sigma + default_jitter I) eps.  The padding block stays the identity (V's padding columns are 0)
            LA(add_diag_launch(Sig, Np, (int)Np, GPFLOW_DEFAULT_JITTER, s));
            LA(chol_lower(Sig, Np, (int)Np, dinv, chol_info + l, s, c->gws, c->gws_doubles, &c->la_main));
            LA(sample_normals_launch(sa, l, E, Sp, Np, s));
            GemmP p;   // F = C E
            p.A = Sig; p.lda = Np; p.a_kc = 1; p.a_tri = 1;
            p.B = E; p.ldb = Sp; p.b_kc = 0;
            p.C = F; p.ldc = Sp; p.m = (int)Np; p.n = (int)Sp; p.k = (int)Np;
            LA(mm_gemm(c, p, s));
            LA(add_mean_samples_launch(md + (size_t)l * Np, F, Sp, N, S, L, l, out_d, s));
        }
        select_latent(c, 0);
    }
    if (want_cov) {
        if (L == 1) {
            CU(cudaMemcpyAsync(mean_out, md, sizeof(double) * N, cudaMemcpyDefault, s));
        } else {   // [L][Np] on the device -> the reference's [N, L]
            double* mt;
            NEED(mt = tp.get((size_t)N * L));
            LA(transpose_to_point_major_launch(md, Np, N, L, mt, s));
            CU(cudaMemcpyAsync(mean_out, mt, sizeof(double) * N * L, cudaMemcpyDefault, s));
        }
    } else if (out_host) {
        CU(cudaMemcpyAsync(samples_out, out_d, sizeof(double) * (size_t)S * N * L, cudaMemcpyDeviceToHost, s));
    }
    std::vector<int> chol_h(chol_info ? L : 0);
    if (chol_info) CU(cudaMemcpyAsync(chol_h.data(), chol_info, sizeof(int) * L, cudaMemcpyDeviceToHost, s));
    double tail[4];
    int info_h[N_INFO];
    OK(read_tails(c, tail, nullptr, info_h));   // synchronises
    OK(check_info(c, info_h));
    if (tail[1] != 0.0) FAIL(TSVGP_ERR_NONPOSITIVE_VARIANCE, "predict_f: non-positive predictive variance");
    for (int l = 0; l < (int)chol_h.size(); ++l)
        if (chol_h[l]) {
            c->last_info = chol_h[l];
            FAIL(TSVGP_ERR_NOT_POSITIVE_DEFINITE, "Cholesky of Sigma + 1e-6 I (latent %d) failed at query point %d", l, chol_h[l]);
        }
    return TSVGP_OK;
}

int tsvgp_predict_f_full_cov(tsvgp_ctx* c, const double* Xnew, int64_t N, int D, const double* mean_X, double* mean_out, double* cov_out) {
    if (!c) return TSVGP_ERR_INVALID;
    if (!Xnew || !mean_out || !cov_out || N < 1) FAIL(TSVGP_ERR_INVALID, "Xnew [N >= 1, D], mean_out [N, L], cov_out [L, N, N] are required");
    return predict_full(c, Xnew, N, D, mean_X, mean_out, cov_out, 0, 1, nullptr, nullptr);
}

int tsvgp_predict_f_samples(tsvgp_ctx* c, const double* Xnew, int64_t N, int D, const double* mean_X, int S, int full_cov,
                            const double* eps, double* samples_out) {
    if (!c) return TSVGP_ERR_INVALID;
    if (!Xnew || !samples_out || N < 1 || S < 1) FAIL(TSVGP_ERR_INVALID, "Xnew [N >= 1, D] and samples_out [S >= 1, N, L] are required");
    return predict_full(c, Xnew, N, D, mean_X, nullptr, nullptr, S, full_cov != 0, eps, samples_out);
}

int tsvgp_predict_f_extra_data(tsvgp_ctx* c, const double* Xnew, int64_t N, int D, const double* mean_X, double jitter,
                               double* mean_out, double* var_out) {
    if (!c) return TSVGP_ERR_INVALID;
    if (!c->white) FAIL(TSVGP_ERR_STATE, "predict_f_extra_data belongs to the whitened sibling model (option \"white\")");
    OK(require_model(c, true));
    CU(cudaSetDevice(c->dev));
    cudaStream_t s = c->s_main;
    const int n = c->Mp;
    const long ld = n;
    const size_t mm = (size_t)n * n;
    // (1) natural parameters of the resident (extra) data under the current sites: tsvgp_white.py:183-212
    c->collective_ok = true;
    CU(cudaMemsetAsync(c->info, 0, sizeof(int) * N_INFO, s));
    OK(ensure_xs(c));
    OK(ensure_kuu(c));
    OK(start_k9(c, 1e-9));
    OK(ensure_posterior(c));
    OK(choose_route(c, 1e-9));
    OK(data_pass(c, MODE_STATS));
    select_latent(c, 0);
    OK(all_reduce(c, c->stats_all[0], (size_t)c->L * (mm + n + 4)));
    {   // the reference calls predict_f on the extra data here (assert_positive, failed Cholesky raise): check before going on,
        // the nested predict_f below clears the flags
        double tail[4];
        int info_h[N_INFO];
        OK(read_tails(c, tail, nullptr, info_h));
        OK(check_info(c, info_h));
        if (tail[1] != 0.0) FAIL(TSVGP_ERR_NONPOSITIVE_VARIANCE, "predict_f_extra_data: non-positive predictive variance at the extra data");
    }
    // (2) K_j = Kuu + jitter I ; combined sites lambda_1 + K_j g0, Lambda_2 - 2 K_j G2 K_j, latent by latent (tsvgp_white.py:144-150).
    // The current sites of latent l wait in its own accumulator B_l / b_l, dead once G2_l and G1_l are formed.
    struct Restore {   // every exit path puts the sites, K6 and its jitter back
        tsvgp_ctx* c; double jit_saved; int n; size_t mm; cudaStream_t s; int saved;
        ~Restore() {
            for (int l = 0; l < saved; ++l) {
                const double* bak = c->stats_all[0] + (size_t)l * (mm + n + 4);
                cudaMemcpyAsync(c->L2_all + (size_t)l * mm, bak, sizeof(double) * mm, cudaMemcpyDeviceToDevice, s);
                cudaMemcpyAsync(c->lam1_all + (size_t)l * n, bak + mm, sizeof(double) * n, cudaMemcpyDeviceToDevice, s);
            }
            c->jit6 = jit_saved;
            copy_add_diag_launch(c->K, c->K6, n, n, c->jit6, s);
            c->c6_valid = c->wpost_valid = c->wkl_valid = false;
            cudaStreamSynchronize(s);
            select_latent(c, 0);
        }
    } restore{c, c->jit6, n, mm, s, 0};
    c->jit6 = jitter;
    LA(copy_add_diag_launch(c->K, c->K6, n, n, jitter, s));   // (the statistics below use chol(K + 1e-9 I) and m_Z only)
    c->c6_valid = c->wpost_valid = c->wkl_valid = false;
    for (int l = 0; l < c->L; ++l) {
        select_latent(c, l);
        OK(dense_update_one(c, 1.0, 1e-9, 1.0, true, false));
        LA(lincomb_launch(c->v1, 1.0, c->v2, -2.0, c->v3, n, s));          // g0 = G1 - 2 G2 mZ
        CU(cudaMemcpyAsync(c->stats[0], c->L2, sizeof(double) * mm, cudaMemcpyDeviceToDevice, s));
        CU(cudaMemcpyAsync(c->stats[0] + mm, c->lam1, sizeof(double) * n, cudaMemcpyDeviceToDevice, s));
        restore.saved = l + 1;
        LA(gemv_n_launch(c->K6, ld, n, c->M, c->v1, 1.0, 0.0, c->mq, s));
        LA(axpby_vec_guarded_launch(c->lam1, c->mq, c->M, 1.0, 1.0, nullptr, nullptr, s));
        GemmP p;
        p.A = c->K6; p.lda = ld; p.a_kc = 1;
        p.B = c->G2; p.ldb = ld; p.b_kc = 0;
        p.C = c->X1; p.ldc = ld; p.m = p.n = p.k = n;
        LA(mm_gemm(c, p, s));
        GemmP q;
        q.A = c->X1; q.lda = ld; q.a_kc = 1;
        q.B = c->K6; q.ldb = ld; q.b_kc = 0;
        q.C = c->X2; q.ldc = ld; q.m = q.n = q.k = n; q.lower_out = 1;
        LA(mm_gemm(c, q, s));
        LA(mirror_lower_launch(c->X2, ld, n, s));
        LA(axpby_guarded_launch(c->L2, c->X2, ld, c->M, 1.0, -2.0, nullptr, nullptr, s));
    }
    select_latent(c, 0);
    // (3) the conditional at Xnew with the combined sites; `restore` puts everything back as it was
    return tsvgp_predict_f(c, Xnew, N, D, mean_X, mean_out, var_out);
}

int tsvgp_posterior(tsvgp_ctx* c, double* m, double* chol_S) {
    if (!c) return TSVGP_ERR_INVALID;
    OK(require_model(c, false));
    CU(cudaSetDevice(c->dev));
    c->collective_ok = false;
    cudaStream_t s = c->s_main;
    const int n = c->Mp;
    CU(cudaMemsetAsync(c->info, 0, sizeof(int) * N_INFO, s));
    OK(ensure_posterior(c));
    if (m)   // m_q [M, L]
        for (int l = 0; l < c->L; ++l)
            CU(cudaMemcpy2DAsync(m + l, sizeof(double) * c->L, c->mq_all + (size_t)l * c->Mp, sizeof(double), sizeof(double), c->M,
                                 cudaMemcpyDefault, s));
    if (chol_S && c->white) {   // S_l = (LR_l^-1 K6)^T (LR_l^-1 K6)   (util.py:421-424), chol_S [L, M, M]
        for (int l = 0; l < c->L; ++l) {
            GemmP p;
            p.A = c->T_all + (size_t)l * n * n; p.lda = n; p.a_kc = 1; p.a_tri = 1;
            p.B = c->K6; p.ldb = n; p.b_kc = 0;
            p.C = c->X1; p.ldc = n; p.m = p.n = p.k = n;
            LA(mm_gemm(c, p, s));
            GemmP q;
            q.A = c->X1; q.lda = n; q.a_kc = 0;
            q.B = c->X1; q.ldb = n; q.b_kc = 0;
            q.C = c->X2; q.ldc = n; q.m = q.n = q.k = n; q.lower_out = 1;
            LA(mm_gemm(c, q, s));
            c->wkl_valid = false;
            LA(chol_lower(c->X2, n, n, c->dinv, c->info + INFO_P, s, c->gws, c->gws_doubles, &c->la_main));
            CU(cudaMemcpy2DAsync(chol_S + (size_t)l * c->M * c->M, sizeof(double) * c->M, c->X2, sizeof(double) * n, sizeof(double) * c->M, c->M,
                                 cudaMemcpyDefault, s));
        }
    } else if (chol_S) {   // S_l = K6_l - (K6_l T_l)(K6_l T_l)^T   (util.py:387-388), chol_S [L, M, M]
        for (int l = 0; l < c->L; ++l) {
            select_latent(c, l);
            GemmP p;
            p.A = c->K6; p.lda = n; p.a_kc = 1;
            p.B = c->T_all + (size_t)l * n * n; p.ldb = n; p.b_kc = 0; p.b_tri = 2;
            p.C = c->X1; p.ldc = n; p.m = p.n = p.k = n;
            LA(mm_gemm(c, p, s));
            c->kl_valid = false;   // X1 is shared with the KL terms
            CU(cudaMemcpyAsync(c->X2, c->K6, sizeof(double) * (size_t)n * n, cudaMemcpyDeviceToDevice, s));
            GemmP q;
            q.A = c->X1; q.lda = n; q.a_kc = 1;
            q.B = c->X1; q.ldb = n; q.b_kc = 1;
            q.C = c->X2; q.ldc = n; q.m = q.n = q.k = n;
            q.alpha = -1.0; q.beta = 1.0; q.lower_out = 1;
            LA(mm_gemm(c, q, s));
            LA(chol_lower(c->X2, n, n, c->dinv, c->info + INFO_S, s, c->gws, c->gws_doubles, &c->la_main));
            CU(cudaMemcpy2DAsync(chol_S + (size_t)l * c->M * c->M, sizeof(double) * c->M, c->X2, sizeof(double) * n, sizeof(double) * c->M, c->M,
                                 cudaMemcpyDefault, s));
        }
        select_latent(c, 0);
    }
    int info_h[N_INFO];
    CU(cudaMemcpyAsync(info_h, c->info, sizeof info_h, cudaMemcpyDeviceToHost, s));
    CU(cudaStreamSynchronize(s));
    return check_info(c, info_h);
}

int tsvgp_comm_unique_id(void* id_out_128_bytes) {
    NcclApi& api = nccl_api();
    if (!api.ok() || !id_out_128_bytes) return TSVGP_ERR_COMM;
    NcclUniqueId id;
    if (api.GetUniqueId(&id) != 0) return TSVGP_ERR_COMM;
    memcpy(id_out_128_bytes, &id, sizeof id);
    return TSVGP_OK;
}

int tsvgp_comm_init(tsvgp_ctx* c, int world_size, int rank, const void* id_128_bytes) {
    if (!c) return TSVGP_ERR_INVALID;
    if (world_size < 1 || rank < 0 || rank >= world_size || !id_128_bytes) FAIL(TSVGP_ERR_INVALID, "bad world_size / rank / id");
    NcclApi& api = nccl_api();
    if (!api.ok()) FAIL(TSVGP_ERR_COMM, "libnccl.so.2 could not be loaded: %s", dlerror());
    CU(cudaSetDevice(c->dev));
    NcclUniqueId id;
    memcpy(&id, id_128_bytes, sizeof id);
    int r = api.CommInitRank(&c->comm, world_size, id, rank);
    if (r != 0) FAIL(TSVGP_ERR_COMM, "ncclCommInitRank: %s", api.GetErrorString ? api.GetErrorString(r) : "error");
    c->world = world_size; c->rank = rank;
    return TSVGP_OK;
}

int tsvgp_comm_size(const tsvgp_ctx* c) { return c ? c->world : 0; }
int tsvgp_device(const tsvgp_ctx* c) { return c ? c->dev : -1; }
void* tsvgp_stream(const tsvgp_ctx* c) { return c ? (void*)c->s_main : nullptr; }

int tsvgp_get_timings(tsvgp_ctx* c, double* out, int n) {
    if (!c || !out) return TSVGP_ERR_INVALID;
    for (int i = 0; i < n; ++i) out[i] = i < 16 ? c->timings[i] : 0.0;
    return TSVGP_OK;
}

int tsvgp_get_kernel_profile(tsvgp_ctx* c, double* out, int n) {
    if (!c || !out) return TSVGP_ERR_INVALID;
    for (int i = 0; i < n; ++i) out[i] = i < 12 ? c->kprof[i] : 0.0;
    return TSVGP_OK;
}

int tsvgp_timer_start(tsvgp_ctx* c) {
    if (!c) return TSVGP_ERR_INVALID;
    CU(cudaSetDevice(c->dev));
    for (int i = 0; i < 2; ++i)
        if (!c->ev_sw[i]) CU(cudaEventCreate(&c->ev_sw[i]));
    CU(cudaEventRecord(c->ev_sw[0], c->s_main));
    return TSVGP_OK;
}

int tsvgp_timer_stop(tsvgp_ctx* c, double* ms) {
    if (!c || !ms || !c->ev_sw[1]) return TSVGP_ERR_INVALID;
    CU(cudaSetDevice(c->dev));
    CU(cudaEventRecord(c->ev_sw[1], c->s_main));
    CU(cudaEventSynchronize(c->ev_sw[1]));
    float f = 0;
    CU(cudaEventElapsedTime(&f, c->ev_sw[0], c->ev_sw[1]));
    *ms = f;
    return TSVGP_OK;
}

void* tsvgp_device_alloc(tsvgp_ctx* c, size_t bytes) {
    if (!c || cudaSetDevice(c->dev) != cudaSuccess) return nullptr;
    void* p = nullptr;
    if (cudaMalloc(&p, bytes ? bytes : 1) != cudaSuccess) { cudaGetLastError(); return nullptr; }
    return p;
}

void tsvgp_device_free(tsvgp_ctx* c, void* p) {
    if (c && p && cudaSetDevice(c->dev) == cudaSuccess) cudaFree(p);
}

int tsvgp_memcpy(tsvgp_ctx* c, void* dst, const void* src, size_t bytes) {
    if (!c || !dst || !src) return TSVGP_ERR_INVALID;
    CU(cudaSetDevice(c->dev));
    CU(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDefault, c->s_main));
    CU(cudaStreamSynchronize(c->s_main));
    return TSVGP_OK;
}

int tsvgp_sync(tsvgp_ctx* c) {
    if (!c) return TSVGP_ERR_INVALID;
    CU(cudaSetDevice(c->dev));
    CU(cudaStreamSynchronize(c->s_main));
    return TSVGP_OK;
}

void* tsvgp_pinned_alloc(size_t bytes) {
    void* p = nullptr;
    if (cudaHostAlloc(&p, bytes ? bytes : 1, cudaHostAllocDefault) != cudaSuccess) { cudaGetLastError(); return nullptr; }
    return p;
}
void tsvgp_pinned_free(void* p) { if (p) cudaFreeHost(p); }

// --- DLPack (dlpack.h v0.8 layout) -------------------------------------------------------------------------------
typedef struct { int32_t device_type; int32_t device_id; } DLDevice_;
typedef struct { uint8_t code; uint8_t bits; uint16_t lanes; } DLDataType_;
typedef struct {
    void* data; DLDevice_ device; int32_t ndim; DLDataType_ dtype; int64_t* shape; int64_t* strides; uint64_t byte_offset;
} DLTensor_;

int tsvgp_dlpack_view(const void* dl_managed_tensor, tsvgp_view* out) {
    if (!dl_managed_tensor || !out) return TSVGP_ERR_INVALID;
    const DLTensor_* t = (const DLTensor_*)dl_managed_tensor;   // DLManagedTensor begins with its DLTensor
    if (t->dtype.code != 2 /* kDLFloat */ || t->dtype.bits != 64 || t->dtype.lanes != 1) return TSVGP_ERR_INVALID;
    if (t->ndim < 1 || t->ndim > 3) return TSVGP_ERR_INVALID;
    int64_t expect = 1;
    for (int i = t->ndim - 1; i >= 0; --i) {   // compact row-major (strides may be NULL)
        if (t->strides && t->shape[i] > 1 && t->strides[i] != expect) return TSVGP_ERR_INVALID;
        expect *= t->shape[i];
    }
    out->data = (char*)t->data + t->byte_offset;
    out->ndim = t->ndim;
    for (int i = 0; i < 3; ++i) out->shape[i] = i < t->ndim ? t->shape[i] : 1;
    out->device_type = t->device.device_type;
    out->device_id = t->device.device_id;
    return TSVGP_OK;
}

}  // extern "C"
