// Non-GEMM kernels of the t-SVGP natural-gradient path (see kernels.cuh).  sm_100a.
#include "kernels.cuh"
#include "common.cuh"
#include <math.h>

namespace tsvgp {

// =====================================================================================================================
// Covariance tiles.  Restates GPflow 2.2.1 stationaries.py / utilities/ops.py::square_distance (SURVEY Appendix B):
//   Xs = X / lengthscales ;  r2 = |xs|^2 + |zs|^2 - 2 xs.zs  (expansion form, not clipped for SE)
//   SE: variance * exp(-r2/2) ;  Matern52: r = sqrt(max(r2,1e-36)), variance (1 + sqrt5 r + 5/3 r^2) exp(-sqrt5 r)
//   Matern32: variance (1 + sqrt3 r) exp(-sqrt3 r) ;  Matern12: variance exp(-r)   (same r)
// called by the reference at src/models/tsvgp.py:209,268,269 and inside gpflow.conditionals.conditional (:103).
// =====================================================================================================================
__global__ void scale_points_kernel(const double* __restrict__ X, long n, int D, const double* __restrict__ ls,
                                    double* __restrict__ XsT, long ldx, double* __restrict__ x2, long n_pad) {
    const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_pad) return;
    double s = 0.0;
    if (i < n) {
        for (int d = 0; d < D; ++d) {
            const double v = X[i * D + d] / ls[d];
            XsT[(long)d * ldx + i] = v;
            s = fma(v, v, s);
        }
    } else {
        for (int d = 0; d < D; ++d) XsT[(long)d * ldx + i] = 0.0;
    }
    x2[i] = s;
}

int scale_points_launch(const double* X, long n, int D, const double* ls, double* XsT, long ldx, double* x2, long n_pad,
                        cudaStream_t s) {
    if (n_pad <= 0) return 0;
    scale_points_kernel<<<(unsigned)((n_pad + 255) / 256), 256, 0, s>>>(X, n, D, ls, XsT, ldx, x2, n_pad);
    return count_launch();
}

__global__ void unpack_rows_kernel(const double* __restrict__ ZsT, long ldz, int Mp, int D, double* __restrict__ Zs) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= Mp) return;
    for (int d = 0; d < D; ++d) Zs[(long)i * D + d] = ZsT[(long)d * ldz + i];
}
int unpack_rows_launch(const double* ZsT, long ldz, int Mp, int D, double* Zs, cudaStream_t s) {
    unpack_rows_kernel<<<(Mp + 255) / 256, 256, 0, s>>>(ZsT, ldz, Mp, D, Zs);
    return count_launch();
}

// ---- branch-free FP64 math for the covariance epilogue (the CUDA library calls carry slow-path branches and re-materialise
// their constants per call site; here the constants live in registers across the whole tile) ---------------------------
// exp(x) for x <= ~0 (clamped at -700): Cody-Waite reduction by ln2, degree-13 Taylor on |f| <= 0.347 (truncation 4e-18).
__device__ __forceinline__ double exp_nonpos(double x) {
    x = fmax(x, -700.0);
    const double t = fma(x, 1.4426950408889634074, 6755399441055744.0);   // 1.5 * 2^52 : rint in the low mantissa bits
    const int n = __double2loint(t);
    const double fn = t - 6755399441055744.0;
    double f = fma(fn, -6.93147180369123816490e-01, x);
    f = fma(fn, -1.90821492927058770002e-10, f);
    double p = 1.6059043836821613e-10;            // 1/13!
    p = fma(p, f, 2.08767569878681e-09);          // 1/12!
    p = fma(p, f, 2.505210838544172e-08);         // 1/11!
    p = fma(p, f, 2.755731922398589e-07);         // 1/10!
    p = fma(p, f, 2.7557319223985893e-06);        // 1/9!
    p = fma(p, f, 2.48015873015873e-05);          // 1/8!
    p = fma(p, f, 1.984126984126984e-04);         // 1/7!
    p = fma(p, f, 1.388888888888889e-03);         // 1/6!
    p = fma(p, f, 8.333333333333333e-03);         // 1/5!
    p = fma(p, f, 4.1666666666666664e-02);        // 1/4!
    p = fma(p, f, 1.6666666666666666e-01);        // 1/3!
    p = fma(p, f, 0.5);
    p = fma(p, f, 1.0);
    p = fma(p, f, 1.0);
    return p * __hiloint2double((n + 1023) << 20, 0);
}
// sqrt(m) for normal m > 0: hardware reciprocal-sqrt seed, two Newton steps, one residual correction
__device__ __forceinline__ double sqrt_pos(double m) {
    double y;
    asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(m));
    const double hm = 0.5 * m;
    y = y * fma(-hm * y, y, 1.5);
    y = y * fma(-hm * y, y, 1.5);
    double r = m * y;
    const double e = fma(-r, r, m);
    return fma(0.5 * y, e, r);
}

// k(r2) and, when asked, dk/d(r2)  (SE: -k/2 ; Matern-5/2: -(5/6) variance (1 + sqrt5 r) exp(-sqrt5 r) ;
// Matern-3/2: -(3/2) variance exp(-sqrt3 r) ; Matern-1/2: -k / (2 r) for r2 >= 1e-36, else 0)
template <int KIND, bool DERIV>
__device__ __forceinline__ double cov_from_r2(double r2, double variance, double& dk) {
    if (KIND == KERN_SE) {
        const double k = variance * exp_nonpos(-0.5 * r2);
        if (DERIV) dk = -0.5 * k;
        return k;
    } else if (KIND == KERN_MATERN12) {
        // GPflow: variance exp(-r), r = sqrt(max(r2, 1e-36)).  The derivative is the one TensorFlow's autodiff takes through the
        // clamp: 1 / (2 r) below it would put -5e17 variance into the M-step's E at a coincident point (r2 = 0 exactly when a
        // point equals an inducing input: x2, z2 and x.z come from the same fma chain)
        const double r = sqrt_pos(fmax(r2, 1e-36));
        const double k = variance * exp_nonpos(-r);
        if (DERIV) dk = r2 >= 1e-36 ? -0.5 * k / r : 0.0;
        return k;
    } else if (KIND == KERN_MATERN32) {
        const double r = sqrt_pos(fmax(r2, 1e-36));
        const double sqrt3 = 1.73205080756887729353;
        const double e = variance * exp_nonpos(-sqrt3 * r);
        if (DERIV) dk = -1.5 * e;
        return fma(sqrt3, r, 1.0) * e;
    } else {
        const double r = sqrt_pos(fmax(r2, 1e-36));
        const double sqrt5 = 2.23606797749978969641;
        const double e = variance * exp_nonpos(-sqrt5 * r);
        if (DERIV) dk = (-5.0 / 6.0) * fma(sqrt5, r, 1.0) * e;
        return fma(5.0 / 3.0, r * r, fma(sqrt5, r, 1.0)) * e;
    }
}

constexpr int KUF_DC = 16;   // feature chunk staged in shared memory
constexpr int KUF_ROWS = 64; // inducing rows per CTA: 4 thread groups of 16 rows; each thread owns 16 rows x 2 columns

template <int KIND, bool DERIV>
__global__ void __launch_bounds__(256, 2) kuf_kernel(double variance, const double* __restrict__ XsT, long ldx,
                                                     const double* __restrict__ x2, long n0, long n_valid,
                                                     const double* __restrict__ Zs, const double* __restrict__ z2, int M, int D,
                                                     const double* __restrict__ alpha, double* __restrict__ K, long ldk,
                                                     double* __restrict__ mu_part, long ldmu, int pad_identity,
                                                     double* __restrict__ Kp) {
    __shared__ __align__(128) double sx[KUF_DC][128];
    __shared__ __align__(128) double sz[KUF_ROWS][KUF_DC];
    __shared__ double smu[4][128];
    __shared__ __align__(8) uint64_t tma_bar;
    const int tid = threadIdx.x, tx = tid & 63, ty = tid >> 6;
    const long c0 = (long)blockIdx.x * 128;          // chunk-local first column of this tile
    const int ibase = blockIdx.y * KUF_ROWS, rbase = ty * 16;
    if (tid == 0) {
        mbar_init(&tma_bar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");   // make the initialised barrier visible to the async proxy
    }
    uint32_t tma_phase = 0;

    double dot[16][2];
#pragma unroll
    for (int r = 0; r < 16; ++r) { dot[r][0] = 0.0; dot[r][1] = 0.0; }

    for (int dc = 0; dc < D; dc += KUF_DC) {
        const int dlen = min(KUF_DC, D - dc);
        __syncthreads();   // previous chunk consumed (and the barrier initialised)
        // X and Z tiles are staged by TMA bulk copies (one 1 KB row of scaled coordinates per feature, one feature chunk per
        // inducing row) whenever the pieces are 16-byte multiples; otherwise (odd D, e.g. D = 1) by plain loads
        const bool tma_ok = (dlen & 1) == 0 && (D & 1) == 0;
        if (tma_ok) {
            if (tid < 32) {
                if (tid == 0) mbar_expect_tx(&tma_bar, (uint32_t)(dlen * 128 * 8 + KUF_ROWS * dlen * 8));
                __syncwarp();
                for (int d = tid; d < dlen; d += 32) tma_bulk_g2s(&sx[d][0], XsT + (long)(dc + d) * ldx + n0 + c0, 128 * 8, &tma_bar);
                for (int r = tid; r < KUF_ROWS; r += 32)
                    tma_bulk_g2s(&sz[r][0], Zs + (long)(ibase + r) * D + dc, (uint32_t)(dlen * 8), &tma_bar);
            }
            if (dlen < KUF_DC) {   // zero the unused feature slots once (they are never overwritten by the bulk copies)
                for (int e = tid; e < (KUF_DC - dlen) * 128; e += 256) sx[dlen + (e >> 7)][e & 127] = 0.0;
                for (int e = tid; e < KUF_ROWS * (KUF_DC - dlen); e += 256) sz[e / (KUF_DC - dlen)][dlen + e % (KUF_DC - dlen)] = 0.0;
            }
            mbar_wait(&tma_bar, tma_phase);
            tma_phase ^= 1;
            __syncthreads();   // the zero fill above
        } else {
            for (int e = tid; e < KUF_DC * 128; e += 256) {
                const int d = e >> 7, c = e & 127;
                sx[d][c] = d < dlen ? XsT[(long)(dc + d) * ldx + n0 + c0 + c] : 0.0;
            }
            for (int e = tid; e < KUF_ROWS * KUF_DC; e += 256) {
                const int r = e / KUF_DC, d = e % KUF_DC;
                sz[r][d] = d < dlen ? Zs[(long)(ibase + r) * D + dc + d] : 0.0;
            }
            __syncthreads();
        }
        const int dl4 = (dlen + 3) & ~3;
        for (int d4 = 0; d4 < dl4; d4 += 4) {
            double xa[4], xb[4];
#pragma unroll
            for (int d = 0; d < 4; ++d) { xa[d] = sx[d4 + d][tx]; xb[d] = sx[d4 + d][tx + 64]; }
#pragma unroll
            for (int r = 0; r < 16; ++r) {
                const double2* zp = reinterpret_cast<const double2*>(&sz[rbase + r][d4]);
                const double2 z01 = zp[0], z23 = zp[1];
                double a = dot[r][0], b = dot[r][1];
                a = fma(xa[0], z01.x, a); b = fma(xb[0], z01.x, b);
                a = fma(xa[1], z01.y, a); b = fma(xb[1], z01.y, b);
                a = fma(xa[2], z23.x, a); b = fma(xb[2], z23.x, b);
                a = fma(xa[3], z23.y, a); b = fma(xb[3], z23.y, b);
                dot[r][0] = a; dot[r][1] = b;
            }
        }
    }

    const long na = n0 + c0 + tx, nb = na + 64;       // global point indices of this thread's two columns
    const double xa2 = x2[na], xb2 = x2[nb];
    const bool oka = na < n_valid, okb = nb < n_valid;
    double mua = 0.0, mub = 0.0;
#pragma unroll
    for (int r = 0; r < 16; ++r) {
        const int i = ibase + rbase + r;
        const double zi2 = z2[i];
        double dka = 0.0, dkb = 0.0;
        double ka = cov_from_r2<KIND, DERIV>(fma(-2.0, dot[r][0], xa2 + zi2), variance, dka);
        double kb = cov_from_r2<KIND, DERIV>(fma(-2.0, dot[r][1], xb2 + zi2), variance, dkb);
        const bool row_ok = i < M;
        if (!(row_ok && oka)) { ka = (pad_identity && (long)i == na) ? 1.0 : 0.0; dka = 0.0; }
        if (!(row_ok && okb)) { kb = (pad_identity && (long)i == nb) ? 1.0 : 0.0; dkb = 0.0; }
        K[(long)i * ldk + c0 + tx] = ka;
        K[(long)i * ldk + c0 + tx + 64] = kb;
        if (DERIV) {
            Kp[(long)i * ldk + c0 + tx] = dka;
            Kp[(long)i * ldk + c0 + tx + 64] = dkb;
        }
        if (alpha) {
            const double al = alpha[i];
            mua = fma(al, ka, mua);
            mub = fma(al, kb, mub);
        }
    }
    if (alpha) {
        smu[ty][tx] = mua;
        smu[ty][tx + 64] = mub;
        __syncthreads();
        if (tid < 128) mu_part[(long)blockIdx.y * ldmu + c0 + tid] = (smu[0][tid] + smu[1][tid]) + (smu[2][tid] + smu[3][tid]);
    }
}

int kuf_launch(int kind, double variance, const double* XsT, long ldx, const double* x2, long n0, long n_valid, int ncols,
               const double* Zs, const double* z2, int M, int Mp, int D, const double* alpha, double* K, long ldk,
               double* mu_part, long ldmu, int pad_identity, cudaStream_t s, double* Kp) {
    dim3 grid(ncols / 128, Mp / KUF_ROWS);
#define KUF_ARGS variance, XsT, ldx, x2, n0, n_valid, Zs, z2, M, D, alpha, K, ldk, mu_part, ldmu, pad_identity, Kp
    if (kind == KERN_SE && !Kp) kuf_kernel<KERN_SE, false><<<grid, 256, 0, s>>>(KUF_ARGS);
    else if (kind == KERN_SE) kuf_kernel<KERN_SE, true><<<grid, 256, 0, s>>>(KUF_ARGS);
    else if (kind == KERN_MATERN52 && !Kp) kuf_kernel<KERN_MATERN52, false><<<grid, 256, 0, s>>>(KUF_ARGS);
    else if (kind == KERN_MATERN52) kuf_kernel<KERN_MATERN52, true><<<grid, 256, 0, s>>>(KUF_ARGS);
    else if (kind == KERN_MATERN12 && !Kp) kuf_kernel<KERN_MATERN12, false><<<grid, 256, 0, s>>>(KUF_ARGS);
    else if (kind == KERN_MATERN12) kuf_kernel<KERN_MATERN12, true><<<grid, 256, 0, s>>>(KUF_ARGS);
    else if (kind == KERN_MATERN32 && !Kp) kuf_kernel<KERN_MATERN32, false><<<grid, 256, 0, s>>>(KUF_ARGS);
    else if (kind == KERN_MATERN32) kuf_kernel<KERN_MATERN32, true><<<grid, 256, 0, s>>>(KUF_ARGS);
    else return -1;
#undef KUF_ARGS
    return count_launch();
}

// =====================================================================================================================
// Per-point q(f) marginals -> likelihood expectations and their gradients.
// Restates gpflow.likelihoods (Gaussian closed form; ScalarLikelihood 20-point Gauss-Hermite for Bernoulli-probit and
// StudentT) as called at reference src/models/tsvgp.py:88 and :256-259, with the gradients of the quadrature sum written
// analytically instead of tf.GradientTape, and the clip of :262-263 (g_var <= -1e-8).
// =====================================================================================================================

template <int LIK>
__device__ __forceinline__ void logp_and_grad(double f, double y, const LikSpec& lk, double& lp, double& dlp) {
    if (LIK == LIK_BERNOULLI) {
        // inv_probit with GPflow's 1e-3 jitter; logp = log(where(y == 1, p, 1 - p))
        const double p = 0.5 * (1.0 + erf(f * 0.70710678118654752440)) * (1.0 - 2e-3) + 1e-3;
        const double dp = (1.0 - 2e-3) * exp(-0.5 * f * f) * 0.39894228040143267794;
        if (y == 1.0) { lp = log(p); dlp = dp / p; }
        else { lp = log(1.0 - p); dlp = -dp / (1.0 - p); }
    } else {
        // StudentT: c0 - (df+1)/2 * log(1 + ((y-f)/scale)^2 / df)
        const double r = y - f;
        const double q = r / lk.p0;
        lp = lk.c0 - 0.5 * (lk.p1 + 1.0) * log(1.0 + (1.0 / lk.p1) * (q * q));
        dlp = (lk.p1 + 1.0) * r / (lk.p1 * lk.p0 * lk.p0 + r * r);
    }
}

template <int LIK>
__global__ void __launch_bounds__(256) point_stats_kernel(LikSpec lk, PointArgs a, GHTable gh) {
    __shared__ double sred[8];
    const int c = blockIdx.x * 256 + threadIdx.x;
    double ve = 0.0, hsum = 0.0, lsum = 0.0;
    if (c < a.ncols) {
        const bool valid = c < a.n_valid;
        double mu = 0.0, q = 0.0;
        for (int p = 0; p < a.n_mu_part; ++p) mu += a.mu_part[(long)p * a.ldmu + c];
        for (int p = 0; p < a.n_q_part; ++p) q += a.q_part[(long)p * a.ldq + c];
        if (a.q2_part) {
            double q2 = 0.0;
            for (int p = 0; p < a.n_q_part; ++p) q2 += a.q2_part[(long)p * a.ldq + c];
            q -= q2;   // var = k(x,x) - |LA^-1 k|^2 + |LR^-1 k|^2   (reference util.py:83-85)
        }
        const double mean = mu + (a.mean_off ? a.mean_off[c] : 0.0);
        const double var = a.kdiag - q;
        // with x2 (the Gaussian natgrad_step, which forms no v_n): non-finite data raises the flag that keeps the step from
        // committing (the covariance clamps a NaN distance to a finite k, so a NaN in X shows in x2, not in the mean)
        if (valid && (!(var > 0.0) || (a.x2 && !(isfinite(mean) && isfinite(a.x2[c]))))) atomicOr(a.flags, 1);
        if (valid && a.mean_out) { a.mean_out[c] = mean; a.var_out[c] = var; }
        double gm = 0.0, gv = 0.0;
        if (valid && a.y) {
            const double y = a.y[c];
            if (LIK == LIK_GAUSSIAN) {
                const double s2 = lk.p0, r = y - mean;
                ve = -0.5 * 1.83787706640934548356 - 0.5 * log(s2) - 0.5 * (r * r + var) / s2;
                gm = r / s2;
                gv = -0.5 / s2;
            } else {
                const double sd = sqrt(var);
                double gs = 0.0;
                for (int k = 0; k < lk.n_gh; ++k) {
                    const double f = mean + sd * gh.z[k];
                    double lp, dlp;
                    logp_and_grad<LIK>(f, y, lk, lp, dlp);
                    const double wd = gh.w[k] * dlp;
                    ve = fma(gh.w[k], lp, ve);
                    gm += wd;
                    gs = fma(wd, gh.z[k], gs);
                }
                gv = gs / (2.0 * sd);
            }
            if (a.clip) gv = fmin(gv, -1e-8);
            hsum = gv;
            if (a.aux_blocks) {   // d ve / d likelihood parameter (Gaussian: variance ; Student-t: scale), M-step gradients
                if (LIK == LIK_GAUSSIAN) {
                    const double s2 = lk.p0, r = y - mean;
                    lsum = -0.5 / s2 + 0.5 * (r * r + var) / (s2 * s2);
                } else if (LIK == LIK_STUDENT_T) {
                    const double sd = sqrt(var), sc = lk.p0, df = lk.p1;
                    for (int k = 0; k < lk.n_gh; ++k) {
                        const double rr = y - (mean + sd * gh.z[k]);
                        lsum = fma(gh.w[k], -1.0 / sc + (df + 1.0) * rr * rr / (sc * (df * sc * sc + rr * rr)), lsum);
                    }
                }
            }
        }
        if (a.g) { a.g[c] = valid ? gm : 0.0; a.h[c] = valid ? gv : 0.0; }
        if (!valid) ve = 0.0;
    }
    if (a.aux_blocks) {
        __shared__ double sred2[2][8];
        hsum = warp_sum(hsum);
        lsum = warp_sum(lsum);
        if ((threadIdx.x & 31) == 0) { sred2[0][threadIdx.x >> 5] = hsum; sred2[1][threadIdx.x >> 5] = lsum; }
        __syncthreads();
        if (threadIdx.x == 0) {
            double s0 = 0.0, s1 = 0.0;
            for (int w = 0; w < 8; ++w) { s0 += sred2[0][w]; s1 += sred2[1][w]; }
            a.aux_blocks[2 * blockIdx.x] = s0;
            a.aux_blocks[2 * blockIdx.x + 1] = s1;
        }
    }
    if (a.ve_blocks) {
        ve = warp_sum(ve);
        if ((threadIdx.x & 31) == 0) sred[threadIdx.x >> 5] = ve;
        __syncthreads();
        if (threadIdx.x == 0) {
            double s = 0.0;
            for (int w = 0; w < 8; ++w) s += sred[w];
            a.ve_blocks[blockIdx.x] = s;
        }
    }
}

int point_stats_launch(const LikSpec& lik, const PointArgs& a, const GHTable& g_gh, cudaStream_t s) {
    const int grid = (a.ncols + 255) / 256;
    switch (lik.kind) {
        case LIK_GAUSSIAN: point_stats_kernel<LIK_GAUSSIAN><<<grid, 256, 0, s>>>(lik, a, g_gh); break;
        case LIK_BERNOULLI: point_stats_kernel<LIK_BERNOULLI><<<grid, 256, 0, s>>>(lik, a, g_gh); break;
        case LIK_STUDENT_T: point_stats_kernel<LIK_STUDENT_T><<<grid, 256, 0, s>>>(lik, a, g_gh); break;
        default: return -1;
    }
    return count_launch();
}

// ---- Softmax (Monte Carlo) ------------------------------------------------------------------------------------------------
__device__ __forceinline__ void philox4x32_10(unsigned c0, unsigned c1, unsigned c2, unsigned c3, unsigned k0, unsigned k1, unsigned (&out)[4]) {
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        const unsigned hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
        const unsigned hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
        c0 = hi1 ^ c1 ^ k0; c1 = lo1; c2 = hi0 ^ c3 ^ k1; c3 = lo0;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
    out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}
// two standard normals from one Philox block: 2 x 53-bit uniforms -> Box-Muller
__device__ __forceinline__ void normal_pair(unsigned long long seed, unsigned long long draw, unsigned long long point, unsigned s, unsigned lp,
                                            double& z0, double& z1) {
    unsigned r[4];
    philox4x32_10((unsigned)point, (unsigned)(point >> 32), s, lp ^ (unsigned)(draw << 8), (unsigned)seed ^ (unsigned)(draw >> 24),
                  (unsigned)(seed >> 32), r);
    const double u0 = ((double)(((unsigned long long)r[0] << 21) ^ (r[1] >> 11)) + 0.5) * (1.0 / 9007199254740992.0);
    const double u1 = ((double)(((unsigned long long)r[2] << 21) ^ (r[3] >> 11)) + 0.5) * (1.0 / 9007199254740992.0);
    const double rad = sqrt(-2.0 * log(u0));
    double sn, cs;
    sincospi(2.0 * u1, &sn, &cs);
    z0 = rad * cs; z1 = rad * sn;
}

__global__ void __launch_bounds__(128) softmax_stats_kernel(SoftmaxArgs a) {
    __shared__ double sred[4];
    const int c = blockIdx.x * 128 + threadIdx.x;
    double ve = 0.0, hsum = 0.0;
    if (c < a.ncols) {
        const bool valid = c < a.n_valid;
        double mu[MAX_SOFTMAX_CLASSES], sd[MAX_SOFTMAX_CLASSES], gm[MAX_SOFTMAX_CLASSES], gs[MAX_SOFTMAX_CLASSES];
        bool bad = false;
        const double off = a.mean_off ? a.mean_off[c] : 0.0;
        double qs = 0.0;
        if (a.q_shared)
            for (int p = 0; p < a.n_q_part; ++p) qs += a.q_shared[(long)p * a.ldq + c];
        if (a.x2) bad = !isfinite(a.x2[c]);
        for (int l = 0; l < a.L; ++l) {
            double m = 0.0, q = 0.0;
            for (int p = 0; p < a.n_mu_part; ++p) m += a.mu_part[l * a.mu_lat + (long)p * a.ldmu + c];
            for (int p = 0; p < a.n_q_part; ++p) q += a.q_part[l * a.q_lat + (long)p * a.ldq + c];
            // (the whitened sibling rounds as point_stats_kernel does: k(x,x) - (|LA^-1 k|^2 - |LR_l^-1 k|^2), util.py:83-85)
            const double var = a.q_shared ? a.kdiag[l] - (qs - q) : a.kdiag[l] - q;
            mu[l] = m + off;
            bad = bad || !(var > 0.0) || (a.x2 && !isfinite(mu[l]));
            sd[l] = sqrt(var);
            gm[l] = 0.0; gs[l] = 0.0;
            if (valid && a.mean_out) { a.mean_out[l * a.out_lat + c] = mu[l]; a.var_out[l * a.out_lat + c] = var; }
        }
        if (valid && bad) atomicOr(a.flags, 1);
        if (valid && a.y && !bad) {
            const int yc = (int)a.y[c];
            const unsigned long long point = (unsigned long long)(a.n0 + c);
            for (int s = 0; s < a.S; ++s) {
                double f[MAX_SOFTMAX_CLASSES], e[MAX_SOFTMAX_CLASSES], fmax_ = -1e300;
                for (int l = 0; l < a.L; l += 2) {
                    double z0, z1;
                    if (a.eps) {
                        const double* ep = a.eps + ((long)s * a.n_total + (long)point) * a.L + l;
                        z0 = ep[0]; z1 = l + 1 < a.L ? ep[1] : 0.0;
                    } else {
                        normal_pair(a.seed, a.draw, point, (unsigned)s, (unsigned)(l >> 1), z0, z1);
                    }
                    e[l] = z0; f[l] = fma(sd[l], z0, mu[l]); fmax_ = fmax(fmax_, f[l]);
                    if (l + 1 < a.L) { e[l + 1] = z1; f[l + 1] = fma(sd[l + 1], z1, mu[l + 1]); fmax_ = fmax(fmax_, f[l + 1]); }
                }
                double den = 0.0;
                for (int l = 0; l < a.L; ++l) { f[l] = exp(f[l] - fmax_); den += f[l]; }
                // log softmax(f)[y] = (f_y - max) - log(den) ; d / d f_l = [l == y] - p_l
                const double fy = (yc >= 0 && yc < a.L) ? log(f[yc]) : 0.0;
                ve += fy - log(den);
                const double inv = 1.0 / den;
                for (int l = 0; l < a.L; ++l) {
                    const double d = (l == yc ? 1.0 : 0.0) - f[l] * inv;
                    gm[l] += d;
                    gs[l] = fma(d, e[l], gs[l]);
                }
            }
            const double invS = 1.0 / (double)a.S;
            ve *= invS;
            for (int l = 0; l < a.L; ++l) {
                gm[l] *= invS;
                gs[l] = gs[l] * invS / (2.0 * sd[l]);
                if (a.clip) gs[l] = fmin(gs[l], -1e-8);
            }
        } else {
            for (int l = 0; l < a.L; ++l) gs[l] = (valid && a.y && a.clip) ? -1e-8 : 0.0;
        }
        if (a.g)
            for (int l = 0; l < a.L; ++l) { a.g[l * a.gh_lat + c] = valid ? gm[l] : 0.0; a.h[l * a.gh_lat + c] = valid ? gs[l] : 0.0; }
        if (a.aux_blocks && valid)
            for (int l = 0; l < a.L; ++l) hsum += gs[l];
        if (!valid) ve = 0.0;
    }
    ve = warp_sum(ve);
    if ((threadIdx.x & 31) == 0) sred[threadIdx.x >> 5] = ve;
    __syncthreads();
    if (threadIdx.x == 0 && a.ve_blocks) {
        const double s2 = (sred[0] + sred[1]) + (sred[2] + sred[3]);
        // ve_blocks holds one slot per 256 points (point_stats_kernel's layout): two 128-thread blocks share one
        atomicAdd(a.ve_blocks + (blockIdx.x >> 1), s2);
    }
    if (a.aux_blocks) {   // sum of h for the s sum_n h term of the kernel-variance gradient; same slots and order as ve_blocks
        __syncthreads();
        hsum = warp_sum(hsum);
        if ((threadIdx.x & 31) == 0) sred[threadIdx.x >> 5] = hsum;
        __syncthreads();
        if (threadIdx.x == 0) atomicAdd(a.aux_blocks + 2 * (blockIdx.x >> 1), (sred[0] + sred[1]) + (sred[2] + sred[3]));
    }
}
int softmax_stats_launch(const SoftmaxArgs& a, cudaStream_t s) {
    if (a.L < 2 || a.L > MAX_SOFTMAX_CLASSES || a.S < 1) return -1;
    softmax_stats_kernel<<<(a.ncols + 127) / 128, 128, 0, s>>>(a);
    return count_launch();
}

// ---- heteroskedastic Normal (2-D Gauss-Hermite) ------------------------------------------------------------------------
// The integrand of every sum below is a product of a function of f_0 and one of f_1, so each double sum over the n_gh x n_gh
// grid is the product of two single sums (the same value up to rounding).  With r = y - f_0, s = T(f_1), D = T'(f_1) / s and
// E0[.] = sum_i w_i (.)(f_0 = mu_0 + sd_0 z_i), E1[.] = sum_j w_j (.)(f_1 = mu_1 + sd_1 z_j):
//   ve = -1/2 log(2 pi) E0[1] E1[1] - E0[1] E1[log s] - 1/2 E0[r^2] E1[s^-2]
//   d log p / d f_0 = r s^-2                     ->  g_0 = E0[r] E1[s^-2] ;            h_0 = E0[r z] E1[s^-2] / (2 sd_0)
//   d log p / d f_1 = D (r^2 s^-2 - 1)           ->  g_1 = E0[r^2] E1[D s^-2] - E0[1] E1[D]
//                                                    h_1 = (E0[r^2] E1[D s^-2 z] - E0[1] E1[D z]) / (2 sd_1)
// (the pattern of the one-latent quadratures: d / d v_l = sum w d log p / d f_l z_l / (2 sd_l)).
__global__ void __launch_bounds__(256) heteroskedastic_stats_kernel(LikSpec lk, SoftmaxArgs a, GHTable gh) {
    __shared__ double sred[8];
    const int c = blockIdx.x * 256 + threadIdx.x;
    double ve = 0.0;
    if (c < a.ncols) {
        const bool valid = c < a.n_valid;
        double mu[2], var[2];
        for (int l = 0; l < 2; ++l) {
            double m = 0.0, q = 0.0;
            for (int p = 0; p < a.n_mu_part; ++p) m += a.mu_part[l * a.mu_lat + (long)p * a.ldmu + c];
            for (int p = 0; p < a.n_q_part; ++p) q += a.q_part[l * a.q_lat + (long)p * a.ldq + c];
            mu[l] = m;
            var[l] = a.kdiag[l] - q;
            if (valid && a.mean_out) { a.mean_out[l * a.out_lat + c] = mu[l]; a.var_out[l * a.out_lat + c] = var[l]; }
        }
        const bool bad = !(var[0] > 0.0) || !(var[1] > 0.0);
        if (valid && bad) atomicOr(a.flags, 1);
        double g0 = 0.0, g1 = 0.0, h0 = -1e-8, h1 = -1e-8;
        if (valid && a.y && !bad) {
            const double y = a.y[c], sd0 = sqrt(var[0]), sd1 = sqrt(var[1]);
            double s0 = 0.0, er = 0.0, er2 = 0.0, erz = 0.0;
            double s1 = 0.0, elog = 0.0, eb = 0.0, edb = 0.0, edbz = 0.0, ed = 0.0, edz = 0.0;
            for (int k = 0; k < lk.n_gh; ++k) {
                const double w = gh.w[k], z = gh.z[k];
                const double r = y - fma(sd0, z, mu[0]);
                s0 += w;
                er = fma(w, r, er);
                er2 = fma(w, r * r, er2);
                erz = fma(w, r * z, erz);
                const double f1 = fma(sd1, z, mu[1]);
                double logs, d;
                if (lk.p0 == 0.0) {   // exp: log s = f_1, T' / T = 1
                    logs = f1;
                    d = 1.0;
                } else {              // softplus(f) = log(1 + e^f), stable form; T' = sigmoid(f)
                    const double e = exp(-fabs(f1));
                    const double sp = fmax(f1, 0.0) + log1p(e);
                    logs = log(sp);
                    d = (f1 >= 0.0 ? 1.0 : e) / ((1.0 + e) * sp);
                }
                const double b = exp(-2.0 * logs);
                s1 += w;
                elog = fma(w, logs, elog);
                eb = fma(w, b, eb);
                edb = fma(w, d * b, edb);
                edbz = fma(w, d * b * z, edbz);
                ed = fma(w, d, ed);
                edz = fma(w, d * z, edz);
            }
            ve = -0.91893853320467274178 * s0 * s1 - s0 * elog - 0.5 * er2 * eb;
            g0 = er * eb;
            h0 = fmin(erz * eb / (2.0 * sd0), -1e-8);
            g1 = er2 * edb - s0 * ed;
            h1 = fmin((er2 * edbz - s0 * edz) / (2.0 * sd1), -1e-8);
        }
        if (!(valid && a.y)) h0 = h1 = 0.0;
        if (a.g) {
            a.g[c] = valid ? g0 : 0.0; a.h[c] = valid ? h0 : 0.0;
            a.g[a.gh_lat + c] = valid ? g1 : 0.0; a.h[a.gh_lat + c] = valid ? h1 : 0.0;
        }
        if (!valid) ve = 0.0;
    }
    if (a.ve_blocks) {
        ve = warp_sum(ve);
        if ((threadIdx.x & 31) == 0) sred[threadIdx.x >> 5] = ve;
        __syncthreads();
        if (threadIdx.x == 0) {
            double s = 0.0;
            for (int w = 0; w < 8; ++w) s += sred[w];
            a.ve_blocks[blockIdx.x] = s;
        }
    }
}
int heteroskedastic_stats_launch(const LikSpec& lik, const SoftmaxArgs& a, const GHTable& gh, cudaStream_t s) {
    if (a.L != 2 || lik.n_gh < 1 || lik.n_gh > MAX_GH) return -1;
    heteroskedastic_stats_kernel<<<(a.ncols + 255) / 256, 256, 0, s>>>(lik, a, gh);
    return count_launch();
}

// ---- posterior samples ------------------------------------------------------------------------------------------------------
// eps(2 sp, n, l) and eps(2 sp + 1, n, l): one Philox block gives both draws of a sample pair
__device__ __forceinline__ void sample_pair(const SampleArgs& a, long n, int sp, int l, double& z0, double& z1) {
    const int s0 = 2 * sp;
    if (a.eps) {
        z0 = a.eps[((long)s0 * a.N + n) * a.L + l];
        z1 = s0 + 1 < a.S ? a.eps[((long)(s0 + 1) * a.N + n) * a.L + l] : 0.0;
    } else {
        normal_pair(a.seed, a.draw, (unsigned long long)n, (unsigned)sp, (unsigned)l, z0, z1);
    }
}

__global__ void __launch_bounds__(256) sample_normals_kernel(SampleArgs a, int l, double* __restrict__ E, long ld, long Np) {
    const long half = ld >> 1;
    const long t = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= Np * half) return;
    const long n = t / half;
    const int sp = (int)(t - n * half);
    double z0 = 0.0, z1 = 0.0;
    if (n < a.N && 2 * sp < a.S) {
        sample_pair(a, n, sp, l, z0, z1);
        if (2 * sp + 1 >= a.S) z1 = 0.0;
    }
    *reinterpret_cast<double2*>(E + n * ld + 2 * sp) = make_double2(z0, z1);
}
int sample_normals_launch(const SampleArgs& a, int l, double* E, long ld, long Np, cudaStream_t s) {
    if (ld & 1) return -1;
    const long threads = Np * (ld >> 1);
    sample_normals_kernel<<<(unsigned)((threads + 255) / 256), 256, 0, s>>>(a, l, E, ld, Np);
    return count_launch();
}

__global__ void __launch_bounds__(256) add_mean_samples_kernel(const double* __restrict__ mean, const double* __restrict__ F, long ldf,
                                                               long N, int S, int L, int l, double* __restrict__ out) {
    const long t = (long)blockIdx.x * blockDim.x + threadIdx.x;   // sample index fastest: coalesced reads of F's rows
    if (t >= N * S) return;
    const long n = t / S;
    const int smp = (int)(t - n * S);
    out[((long)smp * N + n) * L + l] = mean[n] + F[n * ldf + smp];
}
int add_mean_samples_launch(const double* mean, const double* F, long ldf, long N, int S, int L, int l, double* out, cudaStream_t s) {
    add_mean_samples_kernel<<<(unsigned)((N * S + 255) / 256), 256, 0, s>>>(mean, F, ldf, N, S, L, l, out);
    return count_launch();
}

__global__ void __launch_bounds__(256) diag_samples_kernel(SampleArgs a, const double* __restrict__ mean, const double* __restrict__ var,
                                                           long ld, double* __restrict__ out) {
    const int pairs = (a.S + 1) >> 1;
    const long t = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= a.N * pairs) return;
    const long n = t / pairs;
    const int sp = (int)(t - n * pairs);
    for (int l = 0; l < a.L; ++l) {
        double z0, z1;
        sample_pair(a, n, sp, l, z0, z1);
        const double mu = mean[(long)l * ld + n], sd = sqrt(var[(long)l * ld + n]);
        out[((long)(2 * sp) * a.N + n) * a.L + l] = fma(sd, z0, mu);
        if (2 * sp + 1 < a.S) out[((long)(2 * sp + 1) * a.N + n) * a.L + l] = fma(sd, z1, mu);
    }
}
int diag_samples_launch(const SampleArgs& a, const double* mean, const double* var, long ld, double* out, cudaStream_t s) {
    const long threads = a.N * ((a.S + 1) / 2);
    diag_samples_kernel<<<(unsigned)((threads + 255) / 256), 256, 0, s>>>(a, mean, var, ld, out);
    return count_launch();
}

__global__ void transpose_to_latent_major_kernel(const double* __restrict__ Y, long n, int L, double* __restrict__ Yt, long ld) {
    const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    for (int l = 0; l < L; ++l) Yt[l * ld + i] = Y[i * L + l];
}
int transpose_to_latent_major_launch(const double* Y, long n, int L, double* Yt, long ld, cudaStream_t s) {
    transpose_to_latent_major_kernel<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(Y, n, L, Yt, ld);
    return count_launch();
}
__global__ void transpose_to_point_major_kernel(const double* __restrict__ src, long ld, long n, int L, double* __restrict__ dst) {
    const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    for (int l = 0; l < L; ++l) dst[i * L + l] = src[l * ld + i];
}
int transpose_to_point_major_launch(const double* src, long ld, long n, int L, double* dst, cudaStream_t s) {
    transpose_to_point_major_kernel<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(src, ld, n, L, dst);
    return count_launch();
}

// =====================================================================================================================
// M-vector products
// =====================================================================================================================
__global__ void __launch_bounds__(256) gemv_n_kernel(const double* __restrict__ A, long lda, int m, long n,
                                                     const double* __restrict__ x, double alpha, double beta,
                                                     double* __restrict__ y) {
    PDL_PROLOGUE();
    const int row = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (row >= m) return;
    const double* a = A + (long)row * lda;
    double s0 = 0.0, s1 = 0.0;
    long j = lane * 2;
    for (; j + 1 < n; j += 64) {
        const double2 av = *reinterpret_cast<const double2*>(a + j);
        const double2 xv = *reinterpret_cast<const double2*>(x + j);
        s0 = fma(av.x, xv.x, s0);
        s1 = fma(av.y, xv.y, s1);
    }
    if (j < n) s0 = fma(a[j], x[j], s0);
    const double s = warp_sum(s0 + s1);
    if (lane == 0) y[row] = alpha * s + (beta != 0.0 ? beta * y[row] : 0.0);
}

// long rows (the b += Kuf g mat-vec over a slab: n = points per slab): one CTA per row, four 16-byte loads in flight per thread
__global__ void __launch_bounds__(256) gemv_n_wide_kernel(const double* __restrict__ A, long lda, int m, long n,
                                                          const double* __restrict__ x, double alpha, double beta,
                                                          double* __restrict__ y) {
    PDL_PROLOGUE();
    __shared__ double sred[8];
    const int row = blockIdx.x;
    const double* a = A + (long)row * lda;
    double s0 = 0.0, s1 = 0.0, s2 = 0.0, s3 = 0.0;
    long j = threadIdx.x * 2;
    for (; j + 1 + 3 * 512 < n; j += 4 * 512) {
        const double2 a0 = *reinterpret_cast<const double2*>(a + j), a1 = *reinterpret_cast<const double2*>(a + j + 512);
        const double2 a2 = *reinterpret_cast<const double2*>(a + j + 1024), a3 = *reinterpret_cast<const double2*>(a + j + 1536);
        const double2 x0 = *reinterpret_cast<const double2*>(x + j), x1 = *reinterpret_cast<const double2*>(x + j + 512);
        const double2 x2 = *reinterpret_cast<const double2*>(x + j + 1024), x3 = *reinterpret_cast<const double2*>(x + j + 1536);
        s0 = fma(a0.x, x0.x, s0); s0 = fma(a0.y, x0.y, s0);
        s1 = fma(a1.x, x1.x, s1); s1 = fma(a1.y, x1.y, s1);
        s2 = fma(a2.x, x2.x, s2); s2 = fma(a2.y, x2.y, s2);
        s3 = fma(a3.x, x3.x, s3); s3 = fma(a3.y, x3.y, s3);
    }
    for (; j + 1 < n; j += 512) {
        const double2 av = *reinterpret_cast<const double2*>(a + j);
        const double2 xv = *reinterpret_cast<const double2*>(x + j);
        s0 = fma(av.x, xv.x, s0); s0 = fma(av.y, xv.y, s0);
    }
    if (j < n) s0 = fma(a[j], x[j], s0);
    double v = warp_sum((s0 + s1) + (s2 + s3));
    if ((threadIdx.x & 31) == 0) sred[threadIdx.x >> 5] = v;
    __syncthreads();
    if (threadIdx.x == 0) {
        double t = 0.0;
#pragma unroll
        for (int w = 0; w < 8; ++w) t += sred[w];
        y[row] = alpha * t + (beta != 0.0 ? beta * y[row] : 0.0);
    }
}

int gemv_n_launch(const double* A, long lda, int m, long n, const double* x, double alpha, double beta, double* y, cudaStream_t s) {
    if (n >= 4096 && (n & 1) == 0 && (lda & 1) == 0) launch_k(true, gemv_n_wide_kernel, m, 256, 0, s, A, lda, m, n, x, alpha, beta, y);
    else launch_k(true, gemv_n_kernel, (m + 7) / 8, 256, 0, s, A, lda, m, n, x, alpha, beta, y);
    return count_launch();
}

__global__ void __launch_bounds__(128) gemv_t_part_kernel(const double* __restrict__ A, long lda, int m, int n,
                                                          const double* __restrict__ x, double* __restrict__ work) {
    PDL_PROLOGUE();
    const int j = blockIdx.x * 128 + threadIdx.x;
    const int i0 = blockIdx.y * 64;
    if (j >= n) return;
    double s = 0.0;
    const int i1 = min(i0 + 64, m);
    for (int i = i0; i < i1; ++i) s = fma(A[(long)i * lda + j], x[i], s);
    work[(long)blockIdx.y * n + j] = s;
}
// the partial stage alone, with its own leading dimension: work[chunk][j] = sum over the 64-row chunk of A[i][j] x[i]  (the layout
// kuf_kernel gives its partial means)
__global__ void __launch_bounds__(128) gemv_t_part_ld_kernel(const double* __restrict__ A, long lda, int m, int n,
                                                             const double* __restrict__ x, double* __restrict__ work, long ldw) {
    PDL_PROLOGUE();
    const int j = blockIdx.x * 128 + threadIdx.x;
    const int i0 = blockIdx.y * 64;
    if (j >= n) return;
    double s0 = 0.0, s1 = 0.0;
    const int i1 = min(i0 + 64, m);
    for (int i = i0; i + 1 < i1; i += 2) {
        s0 = fma(A[(long)i * lda + j], x[i], s0);
        s1 = fma(A[(long)(i + 1) * lda + j], x[i + 1], s1);
    }
    if ((i1 - i0) & 1) s0 = fma(A[(long)(i1 - 1) * lda + j], x[i1 - 1], s0);
    work[(long)blockIdx.y * ldw + j] = s0 + s1;
}
int gemv_t_part_launch(const double* A, long lda, int m, int n, const double* x, double* work, long ldw, cudaStream_t s) {
    dim3 grid((n + 127) / 128, (m + 63) / 64);
    launch_k(false, gemv_t_part_ld_kernel, grid, 128, 0, s, A, lda, m, n, x, work, ldw);
    return count_launch();
}
__global__ void gemv_t_sum_kernel(const double* __restrict__ work, int nchunk, int n, double* __restrict__ y) {
    PDL_PROLOGUE();
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n) return;
    double s = 0.0;
    for (int c = 0; c < nchunk; ++c) s += work[(long)c * n + j];
    y[j] = s;
}

int gemv_t_launch(const double* A, long lda, int m, int n, const double* x, double* y, double* work, cudaStream_t s) {
    const int nchunk = (m + 63) / 64;
    dim3 grid((n + 127) / 128, nchunk);
    launch_k(true, gemv_t_part_kernel, grid, 128, 0, s, A, lda, m, n, x, work);
    launch_k(true, gemv_t_sum_kernel, (n + 255) / 256, 256, 0, s, work, nchunk, n, y);
    ++g_launches;
    return count_launch();
}

// =====================================================================================================================
// Diagonal 128x128 blocks: Cholesky (tf.linalg.cholesky at reference tsvgp.py:270,300 and util.py:377,382,388)
// and triangular inverse (used to turn tf.linalg.triangular_solve / cholesky_solve into tensor-core products).
// =====================================================================================================================
constexpr int DB = 128;

// ---------------------------------------------------------------------------------------------------------------------
// Cholesky of one 128x128 block AND X = L^-1, blocked: 4 x 4 sub-blocks of 32 x 32 in shared memory (row stride 36 doubles
// = 4 mod 16, so the DMMA fragment loads below are bank-conflict-free in both orientations).
// Per block step j:
//   (1) ONE warp factors the 32 x 32 diagonal sub-block with lane r owning row r in registers: per pivot one shuffle (the
//       pivot), rsqrt, the scaled column published through a double-buffered shared column (one __syncwarp, no CTA barrier),
//       FMAs only; the right-looking elimination of L X = I rides on the same pivot, so X_jj = L_jj^-1 comes out of the same loop;
//   (2) all 8 warps, DMMA: panel L_ij = A_ij X_jj^T (i > j) and the finished block row of the inverse X_jc = X_jj Xcur_jc (c < j);
//   (3) all 8 warps, DMMA: trailing A_ik -= L_ij L_kj^T (j < k <= i) and the inverse's elimination Xcur_ic -= L_ij X_jc (c <= j).
// 11 CTA barriers instead of 128, and the O(n^3) part runs on the FP64 tensor pipe.  A per-pivot register kernel with one CTA
// barrier per pivot was latency-bound on that barrier chain (77 us per block, 13 us of arithmetic: tools/diag_bench, r01).
// ---------------------------------------------------------------------------------------------------------------------
constexpr int QB = 32, QLD = 36, QBLK = QB * QLD, QNB = DB / QB;
__device__ __forceinline__ int qidx(int i, int j) { return (i * (i + 1) / 2 + j) * QBLK; }

// One warp: the (8 TM) x (8 TN) region at (r0, n0) of the 32 x 32 block C from the 32 x 32 blocks A ([r][k]) and B
// (NT: stored [n][k];  !NT: stored [k][n]).   mode 0: C = A B,  1: C -= A B,  2: C = -A B.   k runs over [klo, 32).
// TRI = 1: B is a lower-triangular block used as B^T (NT) with n0 = 0 — tile column j needs k < 8 (j + 1) only;
// TRI = 2: A is a lower-triangular block with r0 = 0 — tile row i needs k < 8 (i + 1) only.
// Every operand element is read before the warp stores (C may alias A when the region spans whole rows, or B when it spans
// whole columns).
template <int TM, int TN, bool NT, int TRI>
__device__ __forceinline__ void qblk_mma(double* C, const double* A, const double* B, int r0, int n0, int mode, int klo, int lane) {
    const int g = lane >> 2, t = lane & 3;
    double acc[TM][TN][2];
#pragma unroll
    for (int i = 0; i < TM; ++i)
#pragma unroll
        for (int j = 0; j < TN; ++j) acc[i][j][0] = acc[i][j][1] = 0.0;
#pragma unroll
    for (int ks = 0; ks < QB; ks += 4) {
        if (ks >= klo) {   // warp-uniform
            double a[TM], b[TN];
#pragma unroll
            for (int i = 0; i < TM; ++i) a[i] = (TRI == 2 && ks >= 8 * (i + 1)) ? 0.0 : A[(r0 + 8 * i + g) * QLD + ks + t];
#pragma unroll
            for (int j = 0; j < TN; ++j)
                b[j] = (TRI == 1 && ks >= 8 * (j + 1)) ? 0.0 : (NT ? B[(n0 + 8 * j + g) * QLD + ks + t] : B[(ks + t) * QLD + n0 + 8 * j + g]);
#pragma unroll
            for (int i = 0; i < TM; ++i)
#pragma unroll
                for (int j = 0; j < TN; ++j) {
                    if (TRI == 1 && ks >= 8 * (j + 1)) continue;
                    if (TRI == 2 && ks >= 8 * (i + 1)) continue;
                    dmma884(acc[i][j][0], acc[i][j][1], a[i], b[j]);
                }
        }
    }
    __syncwarp();
#pragma unroll
    for (int i = 0; i < TM; ++i)
#pragma unroll
        for (int j = 0; j < TN; ++j) {
            double2* dst = reinterpret_cast<double2*>(C + (r0 + 8 * i + g) * QLD + n0 + 8 * j + 2 * t);
            double2 v;
            if (mode == 1) {
                v = *dst;
                v.x -= acc[i][j][0];
                v.y -= acc[i][j][1];
            } else if (mode == 2) {
                v.x = -acc[i][j][0];
                v.y = -acc[i][j][1];
            } else {
                v.x = acc[i][j][0];
                v.y = acc[i][j][1];
            }
            *dst = v;
        }
}

// Warp 0: in-place Cholesky of the 32 x 32 block Ajj (lower; the upper part is written as zeros).  Lane r owns ROW r of A
// (a[c], c < r) and its diagonal element d.  Per pivot k the dependent chain is shuffle(d from lane k) -> rsqrt -> l = a[k] rs ->
// d -= l^2: the next pivot never waits on shared memory.  The scaled column k and 1 / L[k][k] are published in colbuf[k][.] /
// rsbuf[k] and signalled on mbarrier k, which is all warp 1 (below) needs to run the inverse one pivot behind on another scheduler.
// Returns 0, or k + 1 for the first non-positive (or NaN) pivot k.
// 1 / sqrt(m) for normal m > 0: hardware seed (MUFU.RSQ64H), two Newton steps — the pivot chain's longest link; CUDA's rsqrt()
// adds special-case handling the positive, normal pivots of a Cholesky never need.  (A non-positive pivot is caught before.)
__device__ __forceinline__ double rsqrt_pos(double m) {
    double y;
    asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(m));
    const double hm = 0.5 * m;
    y = y * fma(-hm * y, y, 1.5);
    y = y * fma(-hm * y, y, 1.5);
    return y;
}

// The next pivot's shuffle and reciprocal square root are issued BEFORE the bulk of the current rank-1 update (a warp issues in
// order: behind 30 DFMAs the chain would wait ~60 cycles per pivot for nothing), and the reciprocal square root is the bare
// Newton form above.
__device__ __forceinline__ int warp_potrf_32(double* Ajj, double* colbuf, double* rsbuf, uint64_t* bars, int lane) {
    double a[QB];
#pragma unroll
    for (int c = 0; c < QB; ++c) a[c] = c < lane ? Ajj[lane * QLD + c] : 0.0;
    double d = Ajj[lane * QLD + lane], dl = 0.0;
    int fail = 0;
    double piv = __shfl_sync(0xffffffffu, d, 0);
    if (!(piv > 0.0)) fail = 1;
    double rs = rsqrt_pos(fail ? 1.0 : piv);
#pragma unroll
    for (int k = 0; k < QB; ++k) {
        const double lk = lane > k ? a[k] * rs : 0.0;
        d = fma(-lk, lk, d);
        a[k] = lk;
        if (lane == k) dl = piv * rs;
        colbuf[k * QB + lane] = lk;
        if (lane == 0) rsbuf[k] = rs;
        mbar_arrive(bars + k);   // release: the column and rs are visible to whoever observes the completed phase
        __syncwarp();
        if (k + 1 < QB) {   // the chain first: next pivot and its reciprocal square root
            piv = __shfl_sync(0xffffffffu, d, k + 1);
            if (!(piv > 0.0) && fail == 0) fail = k + 2;   // uniform across the warp
            rs = rsqrt_pos(fail ? 1.0 : piv);
        }
#pragma unroll
        for (int c = k + 1; c < QB; ++c) a[c] = fma(-lk, colbuf[k * QB + c], a[c]);
    }
#pragma unroll
    for (int c = 0; c < QB; ++c) Ajj[lane * QLD + c] = c < lane ? a[c] : (c == lane ? dl : 0.0);
    return fail;
}
__device__ __forceinline__ void warp_trtri_32(double* Xjj, const double* colbuf, const double* rsbuf, uint64_t* bars, uint32_t parity,
                                              int lane) {
    double x[QB];
#pragma unroll
    for (int c = 0; c < QB; ++c) x[c] = c == lane ? 1.0 : 0.0;
#pragma unroll
    for (int k = 0; k < QB; ++k) {
        mbar_wait(bars + k, parity);
        const double xk = x[k] * rsbuf[k];   // X[k][lane], final
        x[k] = xk;
#pragma unroll
        for (int c = k + 1; c < QB; ++c) x[c] = fma(-colbuf[k * QB + c], xk, x[c]);
    }
#pragma unroll
    for (int c = 0; c < QB; ++c) Xjj[c * QLD + lane] = x[c];   // zero above the diagonal by construction
}

// ---------------------------------------------------------------------------------------------------------------------
// Look-ahead schedule of the blocked factorisation (36.9 us per block, 38.9 us with steps (1)-(3) in plain order: tools/diag_bench,
// r02).  The pivot chain of warps 0 / 1 (8 k cycles per 32 x 32 sub-block) is the critical path; everything else is arranged
// around it:
//   * the trailing update of step j is split: T_j^A = the blocks step j + 1 needs (block column j + 1 of A, block row j + 1 of the
//     inverse's work matrix) runs on all warps right after the panel; T_j^B = the rest is DEFERRED and runs on warps 2..7 while
//     warps 0 / 1 factor sub-block j + 1;
//   * the same six warps then write back what became final with panel j (block column j of L, block row j of X), so that only
//     the last column / row is left for the end.
// Dependencies: F_{j+1} touches A(j+1,j+1), X(j+1,j+1) only; T_j^B writes A(i,k), k >= j+2, and Xcur(i,c), i >= j+2, and reads block
// column j of L and block row j of X, which nobody writes any more.
// ---------------------------------------------------------------------------------------------------------------------
// rows [r0, r0 + nr) of the 32 x 32 sub-block (bi, bj) -> G (row stride ldg); zeros above the diagonal of a diagonal sub-block
__device__ __forceinline__ void qstore_rows(const double* blk, double* G, long ldg, int bi, int bj, int r0, int nr, int lane) {
    for (int r = r0; r < r0 + nr; ++r) {
        double v = blk[r * QLD + lane];
        if (bi == bj && lane > r) v = 0.0;
        G[(long)(QB * bi + r) * ldg + QB * bj + lane] = v;
    }
}

// trailing tasks of step j; part 0 = T_j^A (needed by step j + 1), part 1 = T_j^B (deferred).  Task t goes to worker (t % nw) + w0.
__device__ __forceinline__ void qtrailing(double* As, double* Xs, int j, int part, int w0, int nw, int warp, int lane) {
    int tsk = 0;
    for (int i = j + 1; i < QNB; ++i) {
        for (int k = j + 1; k <= i; ++k) {
            if ((k == j + 1 ? 0 : 1) != part) continue;
            for (int qd = 0; qd < 4; ++qd) {
                if (i == k && qd == 1) continue;   // strictly upper quarter of a diagonal block
                if ((tsk++ % nw) + w0 == warp)
                    qblk_mma<2, 2, true, 0>(As + qidx(i, k), As + qidx(i, j), As + qidx(k, j), 16 * (qd >> 1), 16 * (qd & 1), 1, 0, lane);
            }
        }
        if ((i == j + 1 ? 0 : 1) != part) continue;
        for (int c = 0; c <= j; ++c)
            for (int qd = 0; qd < 4; ++qd)
                if ((tsk++ % nw) + w0 == warp)
                    qblk_mma<2, 2, false, 0>(Xs + qidx(i, c), As + qidx(i, j), Xs + qidx(j, c), 16 * (qd >> 1), 16 * (qd & 1),
                                             c == j ? 2 : 1, c == j ? 16 * (qd & 1) : 0, lane);
    }
}

// write back block column j of L and block row j of X (final once panel j is done) in 16-row pieces; piece t -> worker (t % nw) + w0
__device__ __forceinline__ void qwriteback(const double* As, const double* Xs, double* A, long lda, double* Dinv, int j, int w0, int nw,
                                           int warp, int lane) {
    int tsk = 0;
    for (int i = j; i < QNB; ++i)
        for (int h = 0; h < 2; ++h)
            if ((tsk++ % nw) + w0 == warp) qstore_rows(As + qidx(i, j), A, lda, i, j, 16 * h, 16, lane);
    for (int c = 0; c <= j; ++c)
        for (int h = 0; h < 2; ++h)
            if ((tsk++ % nw) + w0 == warp) qstore_rows(Xs + qidx(j, c), Dinv, DB, j, c, 16 * h, 16, lane);
}

__global__ void __launch_bounds__(256) diag_potrf_inv_lookahead_kernel(double* A, long lda, double* Dinv, int blk, int* info) {
    PDL_PROLOGUE();
    extern __shared__ __align__(16) double S[];
    double* As = S;
    double* Xs = S + (QNB * (QNB + 1) / 2) * QBLK;
    __shared__ __align__(16) double colbuf[QB * QB];
    __shared__ __align__(16) double rsbuf[QB];
    __shared__ __align__(8) uint64_t bars[QB];
    __shared__ int sfail;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    if (tid == 0) sfail = 0;
    if (tid < QB) mbar_init(bars + tid, 32);
    const bool vec_ok = ((reinterpret_cast<uintptr_t>(A) | (uintptr_t)(lda * 8)) & 15) == 0;
    if (vec_ok) {
        for (int u = tid; u < DB * (DB / 2); u += 256) {
            const int r = u >> 6, c = (u & 63) * 2;
            if ((c >> 5) <= (r >> 5)) cp_async16(As + qidx(r >> 5, c >> 5) + (r & 31) * QLD + (c & 31), A + (long)r * lda + c);
        }
        cp_async_commit();
        cp_async_wait<0>();
    } else {
        for (int e = tid; e < DB * DB; e += 256) {
            const int r = e >> 7, c = e & 127;
            if ((c >> 5) <= (r >> 5)) As[qidx(r >> 5, c >> 5) + (r & 31) * QLD + (c & 31)] = A[(long)r * lda + c];
        }
    }
    __syncthreads();
#pragma unroll 1
    for (int j = 0; j < QNB; ++j) {
        if (warp == 0) {
            const int f = warp_potrf_32(As + qidx(j, j), colbuf, rsbuf, bars, lane);
            if (f && lane == 0) sfail = j * QB + f;
        } else if (warp == 1) {
            warp_trtri_32(Xs + qidx(j, j), colbuf, rsbuf, bars, (uint32_t)(j & 1), lane);
        } else if (j > 0) {   // deferred work of step j - 1, in the shadow of the pivot chain
            qtrailing(As, Xs, j - 1, 1, 2, 6, warp, lane);
            qwriteback(As, Xs, A, lda, Dinv, j - 1, 2, 6, warp, lane);
        }
        __syncthreads();
        if (sfail) break;   // uniform
        {   // panel rows below and the finished block row j of X
            int tsk = 0;
            for (int i = j + 1; i < QNB; ++i)
                for (int h = 0; h < 2; ++h)
                    if ((tsk++ & 7) == warp)
                        qblk_mma<2, 4, true, 1>(As + qidx(i, j), As + qidx(i, j), Xs + qidx(j, j), 16 * h, 0, 0, 0, lane);
            for (int c = 0; c < j; ++c)
                for (int h = 0; h < 2; ++h)
                    if ((tsk++ & 7) == warp)
                        qblk_mma<4, 2, false, 2>(Xs + qidx(j, c), Xs + qidx(j, j), Xs + qidx(j, c), 0, 16 * h, 0, 0, lane);
        }
        __syncthreads();
        if (j + 1 < QNB) {
            qtrailing(As, Xs, j, 0, 0, 8, warp, lane);   // what step j + 1 needs
            __syncthreads();
        }
    }
    if (sfail) {
        if (tid == 0) atomicCAS(info, 0, blk * DB + sfail);
        return;
    }
    qwriteback(As, Xs, A, lda, Dinv, QNB - 1, 0, 8, warp, lane);
}

constexpr int DIAG_BLOCKED_SMEM = 2 * (QNB * (QNB + 1) / 2) * QBLK * 8;

// opt in to the large dynamic shared memory of the diagonal-block kernel on the CURRENT device (call once per context)
int diag_init() {
    return (int)cudaFuncSetAttribute(diag_potrf_inv_lookahead_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, DIAG_BLOCKED_SMEM);
}

int diag_potrf_inv_launch(double* A, long lda, double* Dinv, int blk_index, int* info, cudaStream_t s) {
    launch_k(true, diag_potrf_inv_lookahead_kernel, 1, 256, DIAG_BLOCKED_SMEM, s, A, lda, Dinv, blk_index, info);
    return count_launch();
}

// =====================================================================================================================
// Elementwise M x M utilities
// =====================================================================================================================
#define EW_GRID(n) dim3(((n) + 31) / 32, ((n) + 7) / 8), dim3(32, 8)
#define EW_IJ const int j = blockIdx.x * 32 + threadIdx.x, i = blockIdx.y * 8 + threadIdx.y; if (i >= n || j >= n) return;

__global__ void add_diag_kernel(double* A, long lda, int n, double v) {
    PDL_PROLOGUE();
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) A[(long)i * lda + i] += v;
}
int add_diag_launch(double* A, long lda, int n, double v, cudaStream_t s) {
    launch_k(true, add_diag_kernel, (n + 255) / 256, 256, 0, s, A, lda, n, v);
    return count_launch();
}
__global__ void copy_add_diag_kernel(const double* A, double* B, long ld, int n, double v) {
    PDL_PROLOGUE();
    EW_IJ;
    B[(long)i * ld + j] = A[(long)i * ld + j] + (i == j ? v : 0.0);
}
int copy_add_diag_launch(const double* A, double* B, long ld, int n, double v, cudaStream_t s) {
    launch_k(true, copy_add_diag_kernel, EW_GRID(n), 0, s, A, B, ld, n, v);
    return count_launch();
}
__global__ void mirror_lower_kernel(double* A, long lda, int n) {
    PDL_PROLOGUE();
    __shared__ double tile[32][33];
    // block (bx, by) with by >= bx : read lower tile (by, bx), write transposed into (bx, by)
    const int bx = blockIdx.x, by = blockIdx.y;
    if (bx > by) return;
    for (int r = threadIdx.y; r < 32; r += 8) tile[r][threadIdx.x] = A[(long)(by * 32 + r) * lda + bx * 32 + threadIdx.x];
    __syncthreads();
    for (int r = threadIdx.y; r < 32; r += 8) {
        const int i = bx * 32 + r, j = by * 32 + threadIdx.x;   // upper element (i, j), i <= j region
        if (j > i) A[(long)i * lda + j] = tile[threadIdx.x][r];
    }
}
int mirror_lower_launch(double* A, long lda, int n, cudaStream_t s) {
    launch_k(true, mirror_lower_kernel, dim3(n / 32, n / 32), dim3(32, 8), 0, s, A, lda, n);
    return count_launch();
}
__global__ void flip_sym_kernel(const double* W, double* Wf, long ld, int n) {
    PDL_PROLOGUE();
    EW_IJ;
    if (j > i) { Wf[(long)i * ld + j] = 0.0; return; }
    const int a = n - 1 - i, b = n - 1 - j;   // a <= b : take the lower element W[b][a]
    Wf[(long)i * ld + j] = W[(long)b * ld + a];
}
int flip_sym_launch(const double* W, double* Wf, long ld, int n, cudaStream_t s) {
    launch_k(true, flip_sym_kernel, EW_GRID(n), 0, s, W, Wf, ld, n);
    return count_launch();
}
__global__ void antitranspose_kernel(const double* Linv, double* V, long ld, int n) {
    PDL_PROLOGUE();
    EW_IJ;
    V[(long)i * ld + j] = j <= i ? Linv[(long)(n - 1 - j) * ld + (n - 1 - i)] : 0.0;
}
int antitranspose_launch(const double* Linv, double* V, long ld, int n, cudaStream_t s) {
    launch_k(true, antitranspose_kernel, EW_GRID(n), 0, s, Linv, V, ld, n);
    return count_launch();
}
__global__ void zero_upper_kernel(double* A, long lda, int n) {
    PDL_PROLOGUE();
    EW_IJ;
    if (j > i) A[(long)i * lda + j] = 0.0;
}
int zero_upper_launch(double* A, long lda, int n, cudaStream_t s) {
    launch_k(true, zero_upper_kernel, EW_GRID(n), 0, s, A, lda, n);
    return count_launch();
}
__global__ void finalize_sites_kernel(const double* P, double* L2, long ld, int M, int n, const double* bad, const int* info) {
    PDL_PROLOGUE();
    EW_IJ;
    if ((bad && bad[0] != 0.0) || (info && (info[0] | info[1] | info[2] | info[3]))) return;   // failed step: the sites stay as they were
    L2[(long)i * ld + j] = (j <= i && i < M) ? -P[(long)i * ld + j] : 0.0;
}
int finalize_sites_launch(const double* P, double* L2, long ld, int M, int Mp, const double* bad, const int* info, cudaStream_t s) {
    const int n = Mp;
    launch_k(true, finalize_sites_kernel, EW_GRID(n), 0, s, P, L2, ld, M, Mp, bad, info);
    return count_launch();
}
// Linv = blockdiag(dinv[0], dinv[1], ...) with zeros elsewhere: the seed of the bottom-up triangular inverse, one launch
__global__ void trtri_seed_kernel(const double* dinv, double* Linv, long ld, int n) {
    PDL_PROLOGUE();
    EW_IJ;
    const int bi = i >> 7, bj = j >> 7;
    Linv[(long)i * ld + j] = bi == bj ? dinv[(long)bi * DB * DB + (i & 127) * DB + (j & 127)] : 0.0;
}
int trtri_seed_launch(const double* dinv, double* Linv, long ld, int n, cudaStream_t s) {
    launch_k(true, trtri_seed_kernel, EW_GRID(n), 0, s, dinv, Linv, ld, n);
    return count_launch();
}

// deterministic block reductions: fixed grid of 128 partial blocks, then one finishing block ------------------------
constexpr int RED_BLOCKS = 128;
__device__ __forceinline__ double block_sum_256(double v, double* sred) {
    v = warp_sum(v);
    if ((threadIdx.x & 31) == 0) sred[threadIdx.x >> 5] = v;
    __syncthreads();
    double s = 0.0;
    if (threadIdx.x == 0)
        for (int w = 0; w < 8; ++w) s += sred[w];
    __syncthreads();
    return s;   // valid on thread 0
}
__global__ void __launch_bounds__(256) dot_kernel(const double* x, const double* y, int n, double* out) {
    PDL_PROLOGUE();
    __shared__ double sred[8];
    double s = 0.0;
    for (int i = threadIdx.x; i < n; i += 256) s = fma(x[i], y[i], s);
    s = block_sum_256(s, sred);
    if (threadIdx.x == 0) out[0] = s;
}
int dot_launch(const double* x, const double* y, int n, double* out, cudaStream_t s) {
    launch_k(true, dot_kernel, 1, 256, 0, s, x, y, n, out);
    return count_launch();
}
__global__ void update_lambda1_kernel(double* l1, const double* G1, const double* G2mZ, int n, double lr, double scale,
                                      const double* bad, const int* info) {
    PDL_PROLOGUE();
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if ((bad && bad[0] != 0.0) || (info && (info[0] | info[1] | info[2] | info[3]))) return;
    if (i < n) l1[i] = (1.0 - lr) * l1[i] + lr * scale * (G1[i] - 2.0 * G2mZ[i]);
}
int update_lambda1_launch(double* l1, const double* G1, const double* G2mZ, int n, double lr, double scale, const double* bad,
                          const int* info, cudaStream_t s) {
    launch_k(true, update_lambda1_kernel, (n + 255) / 256, 256, 0, s, l1, G1, G2mZ, n, lr, scale, bad, info);
    return count_launch();
}
__global__ void lincomb_kernel(double* y, double a, const double* x1, double b, const double* x2, int n) {
    PDL_PROLOGUE();
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) y[i] = a * x1[i] + b * x2[i];
}
int lincomb_launch(double* y, double a, const double* x1, double b, const double* x2, int n, cudaStream_t s) {
    launch_k(true, lincomb_kernel, (n + 255) / 256, 256, 0, s, y, a, x1, b, x2, n);
    return count_launch();
}
__global__ void axpby_vec_guarded_kernel(double* y, const double* x, int n, double a, double b, const double* bad, const int* info) {
    PDL_PROLOGUE();
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if ((bad && bad[0] != 0.0) || (info && (info[0] | info[1] | info[2] | info[3]))) return;
    if (i < n) y[i] = a * y[i] + b * x[i];
}
int axpby_vec_guarded_launch(double* y, const double* x, int n, double a, double b, const double* bad, const int* info, cudaStream_t s) {
    launch_k(true, axpby_vec_guarded_kernel, (n + 255) / 256, 256, 0, s, y, x, n, a, b, bad, info);
    return count_launch();
}
__global__ void vsub_kernel(const double* a, const double* b, double* y, int n) {
    PDL_PROLOGUE();
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) y[i] = a[i] - b[i];
}
int vsub_launch(const double* a, const double* b, double* y, int n, cudaStream_t s) {
    launch_k(true, vsub_kernel, (n + 255) / 256, 256, 0, s, a, b, y, n);
    return count_launch();
}


// out[0] = sum_ij A[i][j] * B[i][j] over the n x n leading block (deterministic two-stage)
__global__ void __launch_bounds__(256) matdot_part_kernel(const double* A, const double* B, long ld, int n, double* part) {
    PDL_PROLOGUE();
    __shared__ double sred[8];
    double s = 0.0;
    const long total = (long)n * n;
    for (long e = (long)blockIdx.x * 256 + threadIdx.x; e < total; e += (long)RED_BLOCKS * 256) {
        const long o = (e / n) * ld + (e % n);
        s = fma(A[o], B[o], s);
    }
    s = block_sum_256(s, sred);
    if (threadIdx.x == 0) part[blockIdx.x] = s;
}
__global__ void __launch_bounds__(256) sum_parts_kernel(const double* part, double* out) {
    PDL_PROLOGUE();
    __shared__ double sred[8];
    double s = threadIdx.x < RED_BLOCKS ? part[threadIdx.x] : 0.0;
    s = block_sum_256(s, sred);
    if (threadIdx.x == 0) out[0] = s;
}
int matdot_launch(const double* A, const double* B, long ld, int n, double* out, double* part, cudaStream_t s) {
    if (!part) return -1;
    launch_k(true, matdot_part_kernel, RED_BLOCKS, 256, 0, s, A, B, ld, n, part);
    launch_k(true, sum_parts_kernel, 1, 256, 0, s, part, out);
    ++g_launches;
    return count_launch();
}
__global__ void __launch_bounds__(256) logdiag_kernel(const double* A, long lda, int n, double* out) {
    PDL_PROLOGUE();
    __shared__ double sred[8];
    double l = 0.0;
    for (int i = threadIdx.x; i < n; i += 256) l += log(A[(long)i * lda + i]);
    l = block_sum_256(l, sred);
    if (threadIdx.x == 0) out[0] = l;
}
int logdiag_launch(const double* A, long lda, int n, double* out, cudaStream_t s) {
    launch_k(true, logdiag_kernel, 1, 256, 0, s, A, lda, n, out);
    return count_launch();
}
// P = coef * G on [0,M)^2 plus jitter on its diagonal; identity on the padding block [M,n)
__global__ void init_update_kernel(const double* G, double* P, long ld, int M, int n, double coef, double jitter) {
    PDL_PROLOGUE();
    EW_IJ;
    double v;
    if (i < M && j < M) v = coef * G[(long)i * ld + j] + (i == j ? jitter : 0.0);
    else v = i == j ? 1.0 : 0.0;
    P[(long)i * ld + j] = v;
}
int init_update_launch(const double* G, double* P, long ld, int M, int Mp, double coef, double jitter, cudaStream_t s) {
    const int n = Mp;
    launch_k(true, init_update_kernel, EW_GRID(n), 0, s, G, P, ld, M, Mp, coef, jitter);
    return count_launch();
}
__global__ void set_scaled_identity_kernel(double* A, long ld, int M, int n, double v, double vpad) {
    PDL_PROLOGUE();
    EW_IJ;
    A[(long)i * ld + j] = i == j ? (i < M ? v : vpad) : 0.0;
}
int set_scaled_identity_launch(double* A, long ld, int M, int Mp, double v, double vpad, cudaStream_t s) {
    const int n = Mp;
    launch_k(true, set_scaled_identity_kernel, EW_GRID(n), 0, s, A, ld, M, Mp, v, vpad);
    return count_launch();
}
__global__ void axpby_guarded_kernel(double* P, const double* X, long ld, int n, double a, double b, const double* bad, const int* info) {
    PDL_PROLOGUE();
    EW_IJ;
    if ((bad && bad[0] != 0.0) || (info && (info[0] | info[1] | info[2] | info[3]))) return;
    P[(long)i * ld + j] = a * P[(long)i * ld + j] + b * X[(long)i * ld + j];
}
int axpby_guarded_launch(double* P, const double* X, long ld, int M, double a, double b, const double* bad, const int* info, cudaStream_t s) {
    const int n = M;
    launch_k(true, axpby_guarded_kernel, EW_GRID(n), 0, s, P, X, ld, n, a, b, bad, info);
    return count_launch();
}
__global__ void vadd_inplace_kernel(double* dst, const double* src, long n) {
    PDL_PROLOGUE();
    const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) dst[i] += src[i];
}
int vadd_inplace_launch(double* dst, const double* src, long n, cudaStream_t s) {
    launch_k(true, vadd_inplace_kernel, (unsigned)((n + 255) / 256), 256, 0, s, dst, src, n);
    return count_launch();
}
// v[i] = 1 + 0.5 sin(1.7 i) for i < M, 0 on the padding: deterministic start vector of the conditioning probe
__global__ void probe_vector_kernel(double* v, int M, int n) {
    PDL_PROLOGUE();
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) v[i] = i < M ? 1.0 + 0.5 * sin(1.7 * (double)i) : 0.0;
}
int probe_vector_launch(double* v, int M, int Mp, cudaStream_t s) {
    launch_k(true, probe_vector_kernel, (Mp + 255) / 256, 256, 0, s, v, M, Mp);
    return count_launch();
}
// stats tail: out[0] = sum of ve partials, out[1] = flags[0] as a double
__global__ void __launch_bounds__(256) stats_tail_kernel(const double* ve_blocks, long nblocks, const int* flags, const double* aux,
                                                         double* out) {
    __shared__ double sred[8];
    double s = 0.0;
    for (long i = threadIdx.x; i < nblocks; i += 256) s += ve_blocks[i];
    s = block_sum_256(s, sred);
    if (threadIdx.x == 0) { out[0] = s; out[1] = flags[0] ? 1.0 : 0.0; }
    double s2 = 0.0, s3 = 0.0;
    if (aux)
        for (long i = threadIdx.x; i < nblocks; i += 256) { s2 += aux[2 * i]; s3 += aux[2 * i + 1]; }
    s2 = block_sum_256(s2, sred);
    s3 = block_sum_256(s3, sred);
    if (threadIdx.x == 0) { out[2] = s2; out[3] = s3; }
}
int stats_tail_launch(const double* ve_blocks, long nblocks, const int* flags, const double* aux, double* out, cudaStream_t s) {
    stats_tail_kernel<<<1, 256, 0, s>>>(ve_blocks, nblocks, flags, aux, out);
    return count_launch();
}
// q = tr[0] * inv_c = sum_n |T^T k_n|^2 ;  out[0] += half_inv_s2 * q ;  out[1] = 1 unless sum_n v_n = sum_kdiag - q is finite and > 0
__global__ void variance_term_kernel(const double* tr, double inv_c, double sum_kdiag, double half_inv_s2, double* out) {
    const double q = tr[0] * inv_c;
    const double v = sum_kdiag - q;
    out[0] += half_inv_s2 * q;
    if (!isfinite(v) || (sum_kdiag > 0.0 && !(v > 0.0))) out[1] = 1.0;   // (a rank without rows has sum_kdiag = q = 0)
}
int variance_term_launch(const double* tr, double inv_c, double sum_kdiag, double half_inv_s2, double* out, cudaStream_t s) {
    variance_term_kernel<<<1, 1, 0, s>>>(tr, inv_c, sum_kdiag, half_inv_s2, out);
    return count_launch();
}

// ---- M-step gradient helpers ------------------------------------------------------------------------------------
// E[i][c] = scale * (alpha[i] g[c] - 2 h[c] U[i][c]) * Kp[i][c]   in place on U   (dELBO/dKuf times dk/dr2)
// ACC: added to E instead (the latents of a coupled likelihood share Kuf, so their dELBO/dKuf add up before the F product)
template <bool ACC>
__global__ void egrad_uf_kernel(double* __restrict__ U, const double* __restrict__ Kp, long ld, int Mp, int ncols,
                                const double* __restrict__ alpha, const double* __restrict__ g, const double* __restrict__ h, double scale,
                                double* __restrict__ E) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    const int i0 = blockIdx.y * 16;
    if (c >= ncols) return;
    const double gc = g[c], hc2 = 2.0 * h[c];
    for (int i = i0; i < i0 + 16 && i < Mp; ++i) {
        const long o = (long)i * ld + c;
        if (ACC) E[o] += scale * (alpha[i] * gc - hc2 * U[o]) * Kp[o];
        else U[o] = scale * (alpha[i] * gc - hc2 * U[o]) * Kp[o];
    }
}
int egrad_uf_launch(double* U, const double* Kp, long ld, int Mp, int ncols, const double* alpha, const double* g, const double* h,
                    double scale, cudaStream_t s, double* E) {
    const dim3 grid((ncols + 255) / 256, (Mp + 15) / 16);
    if (E) egrad_uf_kernel<true><<<grid, 256, 0, s>>>(U, Kp, ld, Mp, ncols, alpha, g, h, scale, E);
    else egrad_uf_kernel<false><<<grid, 256, 0, s>>>(U, Kp, ld, Mp, ncols, alpha, g, h, scale, nullptr);
    return count_launch();
}
// Xa[c][j] (row-major [ncols][W], W = aug_width(D)) = xs_j | 1 | xs_j^2 | 0 ... of point n0 + c (zero rows for c >= nvalid)
__global__ void xaug_kernel(const double* __restrict__ XsT, long ldx, long n0, long nvalid, int ncols, int D, double* __restrict__ Xa,
                            const double* __restrict__ origin, int W) {
    __shared__ double tile[32][33];
    // block: 32 points x W aug columns, 32 at a time; transposes through shared memory so both sides stay coalesced
    const int c0 = blockIdx.x * 32, tx = threadIdx.x & 31, ty = threadIdx.x >> 5;   // 256 threads = 8 rows of 32
    for (int jb = 0; jb < W; jb += 32) {
        for (int r = ty; r < 32; r += 8) {   // r = aug column within the 32-block, tx = point
            const int j = jb + r;
            const long c = c0 + tx;
            double v = 0.0;
            if (c < nvalid) {
                // coordinates relative to a common origin (the centroid of the inducing inputs): the host expands
                // sum E (z - x)^2 = z^2 S1 - 2 z EX + C2, which cancels catastrophically for inputs far from 0 (time stamps ...)
                if (j < D) v = XsT[(long)j * ldx + n0 + c] - (origin ? origin[j] : 0.0);
                else if (j == D) v = 1.0;
                else if (j <= 2 * D) { const double x = XsT[(long)(j - D - 1) * ldx + n0 + c] - (origin ? origin[j - D - 1] : 0.0); v = x * x; }
            }
            tile[r][tx] = v;
        }
        __syncthreads();
        for (int r = ty; r < 32; r += 8) {   // r = point, tx = aug column
            if (c0 + r < ncols) Xa[(long)(c0 + r) * W + jb + tx] = tile[tx][r];
        }
        __syncthreads();
    }
}
int xaug_launch(const double* XsT, long ldx, long n0, long nvalid, int ncols, int D, double* Xa, cudaStream_t s, const double* origin) {
    xaug_kernel<<<(ncols + 31) / 32, 256, 0, s>>>(XsT, ldx, n0, nvalid, ncols, D, Xa, origin, aug_width(D));
    return count_launch();
}
// Gamma[i][j] = scale (QBQ_ij - (qb_i a_j + qb_j a_i)/2) - (a_i a_j - (qm_i a_j + qm_j a_i) + QKQ_ij)/2   (dELBO/dKuu, symmetric)
// E[i][j] = Gamma[i][j] * Kp[i][j] off the diagonal, 0 on it
__global__ void gamma_uu_kernel(const double* QBQ, const double* QKQ, const double* qb, const double* qm, const double* al,
                                const double* Kp, double* Gamma, double* E, long ld, int n, double scale) {
    EW_IJ;
    const long o = (long)i * ld + j;
    const double ai = al[i], aj = al[j];
    const double gmm = scale * (0.5 * (QBQ[o] + QBQ[(long)j * ld + i]) - 0.5 * (qb[i] * aj + qb[j] * ai)) -
                       0.5 * (ai * aj - (qm[i] * aj + qm[j] * ai) + 0.5 * (QKQ[o] + QKQ[(long)j * ld + i]));
    Gamma[o] = gmm;
    E[o] = i == j ? 0.0 : gmm * Kp[o];
}
int gamma_uu_launch(const double* QBQ, const double* QKQ, const double* qb, const double* qm, const double* al, const double* Kp,
                    double* Gamma, double* E, long ld, int n, double scale, cudaStream_t s) {
    gamma_uu_kernel<<<EW_GRID(n), 0, s>>>(QBQ, QKQ, qb, qm, al, Kp, Gamma, E, ld, n, scale);
    return count_launch();
}
// The whitened sibling's dELBO/dKuu (DESIGN §10), symmetric; D = A^-1 B A^-1 - R^-1 B R^-1, W = R0^-1 A R0^-1, rb = R^-1 b,
// al = R^-1 lambda_1, a0 = R0^-1 lambda_1, w = R0^-1 A a0:
// Gamma[i][j] = scale (D_ij - (rb_i al_j + rb_j al_i)/2) - (2 R0inv_ij - Ainv_ij - W_ij + a0_i a0_j - (w_i a0_j + w_j a0_i))/2
// E[i][j] = Gamma[i][j] * Kp[i][j] off the diagonal, 0 on it
__global__ void gamma_uu_white_kernel(const double* D, const double* W, const double* R0inv, const double* Ainv, const double* rb,
                                      const double* al, const double* a0, const double* w, const double* Kp, double* Gamma, double* E,
                                      long ld, int n, double scale) {
    EW_IJ;
    const long o = (long)i * ld + j, t = (long)j * ld + i;
    const double a0i = a0[i], a0j = a0[j];
    const double gmm = scale * (0.5 * (D[o] + D[t]) - 0.5 * (rb[i] * al[j] + rb[j] * al[i])) -
                       0.5 * (2.0 * R0inv[o] - Ainv[o] - 0.5 * (W[o] + W[t]) + a0i * a0j - (w[i] * a0j + w[j] * a0i));
    Gamma[o] = gmm;
    E[o] = i == j ? 0.0 : gmm * Kp[o];
}
int gamma_uu_white_launch(const double* D, const double* W, const double* R0inv, const double* Ainv, const double* rb, const double* al,
                          const double* a0, const double* w, const double* Kp, double* Gamma, double* E, long ld, int n, double scale,
                          cudaStream_t s) {
    gamma_uu_white_kernel<<<EW_GRID(n), 0, s>>>(D, W, R0inv, Ainv, rb, al, a0, w, Kp, Gamma, E, ld, n, scale);
    return count_launch();
}

}  // namespace tsvgp
