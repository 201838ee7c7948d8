// FP64 DMMA GEMM engine (see gemm.cuh).  sm_100a only.
#include "gemm.cuh"
#include "common.cuh"
#include <math.h>
#include <map>
#include <queue>
#include <functional>
#include <mutex>
#include <type_traits>
#include <utility>
#include <vector>

namespace tsvgp {

namespace {

constexpr int BM = 128, BN = 128, BK = 16, NTHREADS = 256;
constexpr int KC_LD = BK + 4;    // [128][20] : rows 160 B apart -> the 4 rows of a half-warp fragment read hit distinct banks
constexpr int MC_LD = BM + 4;    // [16][132]
constexpr int KC_ELEMS = BM * KC_LD;
constexpr int MC_ELEMS = BK * MC_LD;

template <bool A_KC, bool B_KC, bool SCALE>
struct Smem {
    static constexpr int A_ELEMS = A_KC ? KC_ELEMS : MC_ELEMS;
    static constexpr int B_ELEMS = B_KC ? KC_ELEMS : MC_ELEMS;
    static constexpr int STAGE = A_ELEMS + B_ELEMS + (SCALE ? 2 * BK : 0);   // + per-k scale and mat-vec vectors
};

template <bool KC>
__device__ __forceinline__ void load_tile(double* s, const double* __restrict__ g, long ld, int row0, int k0, int tid) {
    if (KC) {
        // 128 rows x 16 k  = 1024 16-byte chunks
#pragma unroll
        for (int c = 0; c < 4; ++c) {
            int idx = tid + c * NTHREADS;
            int r = idx >> 3, cc = (idx & 7) * 2;
            cp_async16(s + r * KC_LD + cc, g + (long)(row0 + r) * ld + k0 + cc);
        }
    } else {
        // 16 k-rows x 128
#pragma unroll
        for (int c = 0; c < 4; ++c) {
            int idx = tid + c * NTHREADS;
            int r = idx >> 6, cc = (idx & 63) * 2;
            cp_async16(s + r * MC_LD + cc, g + (long)(k0 + r) * ld + row0 + cc);
        }
    }
}

template <int EPI>
__device__ __forceinline__ void gemm_epilogue(const GemmP& p, double (&acc)[8][4][2], double* smem, int ti, int tj, int bz, int ks,
                                              int tid, int g, int t, int wm, int wn) {
    if (EPI == EPI_STORE || EPI == EPI_STORE_COLNORM) {
        const bool split = p.ksplit > 1;
        double* Cg = split ? p.part + (long)ks * p.part_stride + (long)bz * (p.part_sC ? p.part_sC : p.sC)
                           : ((p.C2 != nullptr && ks == 1) ? p.C2 : p.C) + (long)bz * p.sC;
        const long ldo = (split && p.part_ld) ? p.part_ld : p.ldc;
        const double alpha = p.alpha, beta = split ? 0.0 : p.beta;
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const long row = ti * BM + wm + 8 * i + g;
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const int col = tj * BN + wn + 8 * j + 2 * t;
                double2* ptr = reinterpret_cast<double2*>(Cg + row * ldo + col);
                double2 o;
                o.x = alpha * acc[i][j][0];
                o.y = alpha * acc[i][j][1];
                if (beta != 0.0) {
                    const double2 old = *ptr;
                    o.x += beta * old.x;
                    o.y += beta * old.y;
                }
                *ptr = o;
            }
        }
    }
    if (EPI == EPI_COLNORM || EPI == EPI_STORE_COLNORM) {
        // column sums of squares over this tile's 128 rows -> norm_out[ti][col]
        double cs[4][2];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            cs[j][0] = 0.0; cs[j][1] = 0.0;
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                cs[j][0] = fma(acc[i][j][0], acc[i][j][0], cs[j][0]);
                cs[j][1] = fma(acc[i][j][1], acc[i][j][1], cs[j][1]);
            }
#pragma unroll
            for (int e = 0; e < 2; ++e) {
                double v = cs[j][e];
                v += __shfl_xor_sync(0xffffffffu, v, 4);
                v += __shfl_xor_sync(0xffffffffu, v, 8);
                v += __shfl_xor_sync(0xffffffffu, v, 16);
                cs[j][e] = v;
            }
        }
        double* red = smem;   // [2][128]; pipeline buffers are idle now
        if (g == 0) {
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                red[(wm >> 6) * BN + wn + 8 * j + 2 * t] = cs[j][0];
                red[(wm >> 6) * BN + wn + 8 * j + 2 * t + 1] = cs[j][1];
            }
        }
        __syncthreads();
        if (tid < BN) p.norm_out[(long)bz * p.sC + (long)ti * p.ldn + tj * BN + tid] = red[tid] + red[BN + tid];
    }
}

// ---- mainloop ---------------------------------------------------------------------------------------------------------
// Stage hand-over goes through mbarriers instead of a CTA-wide barrier per k-tile: every thread's cp.async group arrives on
// full[stage] when it lands; a warp that has consumed a stage arrives on empty[stage]; a stage is refilled two tiles after it was
// consumed, so warps may drift up to two k-tiles apart and the DMMA pipe of an SM sub-partition is not drained at every tile
// boundary (ncu r01: 84 % DMMA-pipe active with a CTA barrier per k-tile).
constexpr int PSTAGES = 5;

template <bool A_KC, bool B_KC, bool SCALE, int EPI>
__global__ void __launch_bounds__(NTHREADS, 1) gemm_kernel_mb(GemmP p, int order) {
    PDL_PROLOGUE();   // no-op unless launched with the programmatic-serialisation attribute (GemmP::pdl)
    using S = Smem<A_KC, B_KC, SCALE>;
    extern __shared__ __align__(16) double smem[];
    uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + S::STAGE * PSTAGES);
    uint64_t* empty = full_bar + PSTAGES;

    // Launch order = longest tiles first.  CTAs are dispatched in linear block order (x fastest); with a triangular operand the
    // contraction length of a tile depends on its row or column, and the default order (tile rows ascending) can put the longest
    // tiles LAST.  order: bit 0 = the tile COLUMN is the slow index, bit 1 = the slow index runs backwards (host: tile_order()).
    int tj = blockIdx.x, ti = blockIdx.y;
    if (order & 1) { const int lin = blockIdx.y * gridDim.x + blockIdx.x; tj = lin / (int)gridDim.y; ti = lin % (int)gridDim.y; }
    if (order & 2) { if (order & 1) tj = (int)gridDim.x - 1 - tj; else ti = (int)gridDim.y - 1 - ti; }
    if (p.lower_out && tj > ti) return;
    if (p.row_mod > 1 && ti % p.row_mod != p.row_rem) return;
    const int zdiv = p.C2 != nullptr ? 2 : p.ksplit;
    const int bz = blockIdx.z / zdiv, ks = blockIdx.z % zdiv;
    const double* Ag = p.A + (long)bz * p.sA;
    const double* Bg = p.B + (long)bz * p.sB;

    int kb = 0, ke = p.k;
    if (p.a_tri == 1) ke = min(ke, (ti + 1) * BM);
    if (p.a_tri == 2) kb = max(kb, ti * BM);
    if (p.b_tri == 1) ke = min(ke, (tj + 1) * BN);
    if (p.b_tri == 2) kb = max(kb, tj * BN);
    if (p.ksplit > 1) {
        int nkt = max(ke - kb, 0) / BK;
        int per = (nkt + p.ksplit - 1) / p.ksplit;
        kb += ks * per * BK;
        ke = min(ke, kb + per * BK);
    }
    const bool piece2 = p.C2 != nullptr && ks == 1;
    if (p.C2 != nullptr) { if (piece2) kb = max(kb, p.ksp); else ke = min(ke, p.ksp); }
    const int KT = max(ke - kb, 0) / BK;

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, g = lane >> 2, t = lane & 3;
    const bool plain = p.a_tri == 0 && p.b_tri == 0;
    const bool diag_tile = p.lower_out && ti == tj && plain;
    // Warps w and w + 4 share an SM sub-partition, i.e. one DMMA pipe.  The 8x8 blocks skipped below (zero blocks of a triangular
    // operand inside its diagonal k-block; the strictly upper blocks of a diagonal output tile) must be spread EVENLY over the four
    // pipes, or the tile runs at the speed of the fullest one:
    //  * general mapping: the two warps of a sub-partition sit in different row halves (wm 0 / 64), so inside the diagonal k-block of
    //    an upper-triangular A^T — where row block i is non-zero only from k-tile i/2 on — every pipe sees the same mix;
    //  * diagonal tile of a symmetric product (needed blocks per warp: 32, 32, 26, 26, 10, 10, 0, 0): the pairs (64,0)+(0,64),
    //    (64,32)+(0,96), (0,0)+(64,96), (64,64)+(0,32) give 32 / 32 / 36 / 36 DMMAs per k-step and pipe instead of up to 64.
    // one nibble per warp: bit 2 = row half (wm / 64), bits 0-1 = column quarter (wn / 32); see g_wmap / g_wmap_diag below
    const unsigned nib = ((diag_tile ? p.wmap_diag : p.wmap) >> (4 * warp)) & 15u;
    const int wm = (int)(nib >> 2) * 64, wn = (int)(nib & 3u) * 32;
    const int dj = diag_tile ? (wm - wn) / 8 : 64;   // diagonal tile of a symmetric product: (i, j) needed iff j <= i + dj
    const int dj_pat = dj >= 3 ? 0 : (dj == 0 ? 1 : (dj == -4 ? 2 : 3));
    const bool tri_a2 = p.a_tri == 2 && p.b_tri == 0 && !p.lower_out;

    if (tid == 0) {
#pragma unroll
        for (int s = 0; s < PSTAGES; ++s) { mbar_init(&full_bar[s], NTHREADS); mbar_init(&empty[s], NTHREADS / 32); }
    }
    __syncthreads();

    double acc[8][4][2];
#pragma unroll
    for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) { acc[i][j][0] = 0.0; acc[i][j][1] = 0.0; }
    // Fused mat-vec b += A g, carried by the first tile column: its two warps with wn == 0 cover all 128 rows of the tile.
    const bool matvec = SCALE && p.gvec != nullptr && wn == 0 && tj == 0;
    const bool use_scale = SCALE && p.kscale != nullptr;
    double bacc[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) bacc[i] = 0.0;

    int ps = 0, pround = 0, L = 0;          // producer cursor: tile L goes to stage ps, the pround-th use of that stage
    auto produce = [&]() {
        if (L < KT) {
            if (pround > 0) mbar_wait(&empty[ps], (pround - 1) & 1);
            double* sa = smem + ps * S::STAGE;
            double* sb = sa + S::A_ELEMS;
            const int k0 = kb + L * BK;
            load_tile<A_KC>(sa, Ag, p.lda, ti * BM, k0, tid);
            load_tile<B_KC>(sb, Bg, p.ldb, tj * BN, k0, tid);
            if (SCALE && tid < BK / 2 && p.kscale) cp_async16(sb + S::B_ELEMS + tid * 2, p.kscale + k0 + tid * 2);
            if (SCALE && tid >= 32 && tid < 32 + BK / 2 && p.gvec) cp_async16(sb + S::B_ELEMS + BK + (tid - 32) * 2, p.gvec + k0 + (tid - 32) * 2);
            cp_async_mbar_arrive(&full_bar[ps]);
        }
        ++L;
        if (++ps == PSTAGES) { ps = 0; ++pround; }
    };
#pragma unroll
    for (int s = 0; s < PSTAGES - 2; ++s) produce();

    int cs = 0, cph = 0;
    for (int kt = 0; kt < KT; ++kt) {
        produce();
        // which 8x8 blocks of this warp's 64x32 tile are identically zero / not needed in this k-tile (compile-time patterns only:
        // run-time predicates around single DMMAs cost more than the DMMAs they save)
        //   IHI < 8 : A(i,k) = 0 for row blocks i >= IHI (upper-triangular A^T, k-tile inside the diagonal k-block)
        //   DJ      : diagonal tile of a symmetric (lower_out) product: block (i, j) needed iff j <= i + DJ
        int ihi = 8;
        if (tri_a2) ihi = min(8, max(0, ((kb + kt * BK - ti * BM - wm + BK - 1) >> 3) + 1));
        mbar_wait(&full_bar[cs], cph);
        const double* sa = smem + cs * S::STAGE;
        const double* sb = sa + S::A_ELEMS;
        const double* ssc = sb + S::B_ELEMS;
        auto k_tile = [&](auto ihi_tag, auto dj_tag, auto mv_tag, auto sc_tag) {
            constexpr int IHI = decltype(ihi_tag)::value, DJ = decltype(dj_tag)::value;
            constexpr bool MV = decltype(mv_tag)::value, SC = decltype(sc_tag)::value;
#pragma unroll
            for (int kk = 0; kk < BK; kk += 4) {
                double a[8], b[4];
#pragma unroll
                for (int i = 0; i < 8; ++i)
                    a[i] = A_KC ? sa[(wm + 8 * i + g) * KC_LD + kk + t] : sa[(kk + t) * MC_LD + wm + 8 * i + g];
#pragma unroll
                for (int j = 0; j < 4; ++j)
                    b[j] = B_KC ? sb[(wn + 8 * j + g) * KC_LD + kk + t] : sb[(kk + t) * MC_LD + wn + 8 * j + g];
                if (SCALE) {
                    if (SC) {
                        const double h = ssc[kk + t];
#pragma unroll
                        for (int j = 0; j < 4; ++j) b[j] *= h;
                    }
                    if (MV) {
                        const double gk = ssc[BK + kk + t];
#pragma unroll
                        for (int i = 0; i < 8; ++i) bacc[i] = fma(a[i], gk, bacc[i]);
                    }
                }
#pragma unroll
                for (int i = 0; i < 8; ++i)
#pragma unroll
                    for (int j = 0; j < 4; ++j)
                        if (i < IHI && j <= i + DJ) dmma884(acc[i][j][0], acc[i][j][1], a[i], b[j]);
            }
        };
        using I8 = std::integral_constant<int, 8>;
        using FULLJ = std::integral_constant<int, 64>;
        using J0 = std::integral_constant<int, 0>;
        using Jm4 = std::integral_constant<int, -4>;
        using Yes = std::true_type;
        using No = std::false_type;
        if (SCALE) {   // statistics products: optional per-k weights (absent when the weights are one constant, Gaussian likelihood)
            if (matvec) {   // the two warps of the first tile column that also carry b += A g
                if (use_scale) { if (dj_pat == 1) k_tile(I8{}, J0{}, Yes{}, Yes{}); else k_tile(I8{}, FULLJ{}, Yes{}, Yes{}); }
                else { if (dj_pat == 1) k_tile(I8{}, J0{}, Yes{}, No{}); else k_tile(I8{}, FULLJ{}, Yes{}, No{}); }
            } else if (use_scale) {
                if (dj_pat == 0) k_tile(I8{}, FULLJ{}, No{}, Yes{});
                else if (dj_pat == 1) k_tile(I8{}, J0{}, No{}, Yes{});
                else if (dj_pat == 2) k_tile(I8{}, Jm4{}, No{}, Yes{});
            } else {
                if (dj_pat == 0) k_tile(I8{}, FULLJ{}, No{}, No{});
                else if (dj_pat == 1) k_tile(I8{}, J0{}, No{}, No{});
                else if (dj_pat == 2) k_tile(I8{}, Jm4{}, No{}, No{});
            }
        }
        else if (dj_pat == 0 && ihi == 8) k_tile(I8{}, FULLJ{}, No{}, No{});                      // the common case
        else if (dj_pat == 1) k_tile(I8{}, J0{}, No{}, No{});                                    // j <= i
        else if (dj_pat == 2) k_tile(I8{}, Jm4{}, No{}, No{});                                   // j <= i - 4
        else if (dj_pat == 3) {}                                                                  // nothing needed
        else if (ihi >= 6) k_tile(std::integral_constant<int, 6>{}, FULLJ{}, No{}, No{});
        else if (ihi >= 4) k_tile(std::integral_constant<int, 4>{}, FULLJ{}, No{}, No{});
        else if (ihi >= 2) k_tile(std::integral_constant<int, 2>{}, FULLJ{}, No{}, No{});
        // ihi == 0 : every A block of this warp is zero in this k-tile
        __syncwarp();
        if (lane == 0) mbar_arrive(&empty[cs]);
        if (++cs == PSTAGES) { cs = 0; cph ^= 1; }
    }
    __syncthreads();   // every global read of this CTA has landed and every warp is out of the pipeline buffers

    if (SCALE && matvec) {   // rows wm + 8 i + g : sum the 4 lanes that split k, then one lane adds into the (CTA-private) rows of b
        double* bo = (p.C2 != nullptr && ks == 1) ? p.bout2 : p.bout;
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            double v = bacc[i];
            v += __shfl_xor_sync(0xffffffffu, v, 1);
            v += __shfl_xor_sync(0xffffffffu, v, 2);
            if (t == 0) bo[ti * BM + wm + 8 * i + g] += v;
        }
    }
    gemm_epilogue<EPI>(p, acc, smem, ti, tj, bz, ks, tid, g, t, wm, wn);
}

constexpr int RED_SLICES = 8;   // row slices per 128 x 128 tile: the reduction is bandwidth work, spread it over 8x the CTAs
__global__ void __launch_bounds__(256) splitk_reduce_kernel(GemmP p) {
    PDL_PROLOGUE();   // no-op unless launched with the programmatic-serialisation attribute (GemmP::pdl)
    const int tj = blockIdx.x, ti = blockIdx.y;
    if (p.lower_out && tj > ti) return;
    if (p.row_mod > 1 && ti % p.row_mod != p.row_rem) return;
    const int bz = blockIdx.z / RED_SLICES, sl = blockIdx.z % RED_SLICES;
    const long pld = p.part_ld ? p.part_ld : p.ldc;
    const double* part = p.part + (long)bz * (p.part_sC ? p.part_sC : p.sC);
    double* C = p.C + (long)bz * p.sC;
    constexpr int ROWS = BM / RED_SLICES;
    // 256 threads over a 16 x 128 strip, two doubles each
    for (int e = threadIdx.x; e < ROWS * BN / 2; e += blockDim.x) {
        const int r = sl * ROWS + e / (BN / 2), c = (e % (BN / 2)) * 2;
        const long poff = (long)(ti * BM + r) * pld + tj * BN + c;
        double2 s = make_double2(0.0, 0.0);
#pragma unroll 4
        for (int k = 0; k < p.ksplit; ++k) {
            const double2 v = *reinterpret_cast<const double2*>(part + (long)k * p.part_stride + poff);
            s.x += v.x; s.y += v.y;
        }
        double2* ptr = reinterpret_cast<double2*>(C + (long)(ti * BM + r) * p.ldc + tj * BN + c);
        if (p.beta != 0.0) {
            const double2 old = *ptr;
            s.x += p.beta * old.x; s.y += p.beta * old.y;
        }
        *ptr = s;
    }
}

// warp -> (row half, column quarter) of the 128 x 128 CTA tile, one nibble per warp (warp 0 in the low nibble), used where
// GemmP::wmap / wmap_diag are 0 (tools/gemm_bench sets them to compare maps).
// Measured on B200 (tools/gemm_bench, profiles/gemm_bench_r02.txt):
//  * general tiles: any map whose sub-partition partners (warps w, w + 4) sit in the SAME row half is fastest for the triangular
//    variance product (1.056 ms per 8192-point slab at M = 2048); partners in different row halves cost 5 % (1.107 - 1.111 ms):
//    inside the diagonal k-block a warp that runs alone on its sub-partition drives the DMMA pipe at only ~64 % of its rate.
//  * diagonal tile of a symmetric product: its needed 8x8 blocks per 64 x 32 warp tile are 32, 32, 26, 26, 10, 10, 0, 0.  The
//    default map puts 32 + 26 on one pipe (1.09 x the time of a FULL tile); pairing (64,0)+(0,64), (64,32)+(0,96), (0,0)+(64,96),
//    (64,64)+(0,32) — 32 / 32 / 36 / 36 per pipe — brings a diagonal tile to 0.78 x a full tile.
unsigned g_wmap = 0x73625140u, g_wmap_diag = 0x17326054u;

// longest contraction first (see gemm_kernel_mb): which tile index bounds the k range, and in which direction it shrinks
static int tile_order(const GemmP& p) {
    if (p.a_tri && p.b_tri) return 0;                       // k range depends on both indices: keep the default
    if (p.a_tri == 2) return 0;                             // k >= ti * 128: row 0 is longest and already first
    if (p.a_tri == 1) return 2;                             // k <  (ti + 1) * 128: last row longest -> rows backwards
    if (p.b_tri == 2) return 1;                             // k >= tj * 128: column 0 longest -> columns are the slow index
    if (p.b_tri == 1) return 3;                             // k <  (tj + 1) * 128: last column longest
    return 0;
}

template <bool A_KC, bool B_KC, bool SCALE>
constexpr int mb_bytes() { return Smem<A_KC, B_KC, SCALE>::STAGE * PSTAGES * 8 + 2 * PSTAGES * 8; }

template <bool A_KC, bool B_KC, bool SCALE, int EPI>
int launch_inst(const GemmP& p, cudaStream_t stream) {
    dim3 grid(p.n / BN, p.m / BM, p.batch * (p.C2 ? 2 : p.ksplit));
    GemmP q = p;
    if (!q.wmap) q.wmap = g_wmap;
    if (!q.wmap_diag) q.wmap_diag = g_wmap_diag;
    launch_k(p.pdl != 0, gemm_kernel_mb<A_KC, B_KC, SCALE, EPI>, grid, NTHREADS, mb_bytes<A_KC, B_KC, SCALE>(), stream, q, tile_order(q));
    return count_launch();
}

template <bool A_KC, bool B_KC, bool SCALE, int EPI>
int init_inst() {
    return (int)cudaFuncSetAttribute(gemm_kernel_mb<A_KC, B_KC, SCALE, EPI>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                     mb_bytes<A_KC, B_KC, SCALE>());
}

}  // namespace

int gemm_init() {
    int e = 0;
    e |= init_inst<true, true, false, EPI_STORE>();
    e |= init_inst<true, true, true, EPI_STORE>();
    e |= init_inst<false, false, false, EPI_STORE>();
    e |= init_inst<false, false, false, EPI_COLNORM>();
    e |= init_inst<false, false, false, EPI_STORE_COLNORM>();
    e |= init_inst<true, false, false, EPI_STORE>();
    e |= init_inst<true, false, false, EPI_COLNORM>();
    e |= init_inst<true, false, false, EPI_STORE_COLNORM>();
    return e;
}

// Greedy in-order dispatch of the lower tiles of an nt x nt symmetric product onto `sms` single-CTA SMs, first every tile's big
// piece (kt1 k-tiles), then every tile's small piece (kt2), in launch order (tile rows, diagonal tile last in its row).  A diagonal
// tile needs only its lower 8x8 blocks and runs at DIAG_COST of a full tile (see the warp mapping in gemm_kernel_mb); every piece
// also pays `ovh` k-tiles of prologue / epilogue (pipeline fill, C tile read-modify-write).
constexpr double DIAG_COST = 0.78;   // measured: one diagonal tile / one full tile of the same k (tools/gemm_bench)
static double dispatch_makespan(int nt, int sms, int kt1, int kt2, double ovh) {
    std::priority_queue<double, std::vector<double>, std::greater<double>> free_at;   // earliest-free SM first
    for (int s = 0; s < sms; ++s) free_at.push(0.0);
    double last = 0.0;
    auto run = [&](double kt) {
        for (int ti = 0; ti < nt; ++ti)
            for (int tj = 0; tj <= ti; ++tj) {
                const double t = free_at.top() + (tj == ti ? DIAG_COST : 1.0) * kt + ovh;
                free_at.pop();
                free_at.push(t);
                last = t > last ? t : last;
            }
    };
    run(kt1);
    if (kt2 > 0) run(kt2);
    return last;
}

int balanced_ksplit(int tiles, int k) {
    static int sms = 0;
    if (!sms) {
        int dev = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
        if (sms <= 0) sms = 148;
    }
    static std::map<std::pair<int, int>, int> cache;
    static std::mutex cache_mutex;   // contexts of different host threads share this table
    std::lock_guard<std::mutex> lock(cache_mutex);
    const auto key = std::make_pair(tiles, k);
    auto it = cache.find(key);
    if (it != cache.end()) return it->second;
    int nt = 1;
    while (nt * (nt + 1) / 2 < tiles) ++nt;   // tiles = nt (nt + 1) / 2 lower tiles
    const int kt = k / BK;
    const double ovh = 3.0;   // measured: a split-off piece costs about 3 k-tiles beyond its DMMA work (tools/gemm_bench)
    int best = k;
    double best_t = dispatch_makespan(nt, sms, kt, 0, ovh);
    // every split point on a k-tile grid; the makespan falls off a cliff just below the optimum (one more round of small pieces)
    // and rises only slowly above it, so the chosen point sits a little above the model's optimum
    const int step = kt >= 1024 ? kt / 512 : 1;
    int best_kt1 = kt;
    for (int kt1 = kt / 2; kt1 <= kt - 4; kt1 += step) {
        const double t = dispatch_makespan(nt, sms, kt1, kt - kt1, ovh);
        if (t < best_t) { best_t = t; best_kt1 = kt1; }
    }
    if (best_kt1 < kt) {
        const int safe = best_kt1 + (kt + 63) / 64;
        if (safe <= kt - 4 && dispatch_makespan(nt, sms, safe, kt - safe, ovh) < 0.985 * dispatch_makespan(nt, sms, kt, 0, ovh))
            best = safe * BK;
        else if (best_t < 0.985 * dispatch_makespan(nt, sms, kt, 0, ovh)) best = best_kt1 * BK;
    }
    cache[key] = best;
    return best;
}

int gemm_launch(const GemmP& p, cudaStream_t stream) {
    if (p.gvec && (!p.bout || (p.C2 && !p.bout2) || p.ksplit != 1 || !p.lower_out)) return -1;
    if (p.C2 && (p.ksplit != 1 || p.epilogue != EPI_STORE || p.ksp % BK || p.ksp <= 0 || p.ksp >= p.k)) return -1;
    if (p.m % BM || p.n % BN || p.k % BK || p.m <= 0 || p.n <= 0) return -1;
    const bool scale = p.kscale != nullptr || p.gvec != nullptr;   // the variant that stages per-k vectors
    if (p.a_kc && p.b_kc) {
        if (p.epilogue != EPI_STORE) return -1;
        return scale ? launch_inst<true, true, true, EPI_STORE>(p, stream) : launch_inst<true, true, false, EPI_STORE>(p, stream);
    }
    if (scale) return -1;
    if (!p.a_kc && !p.b_kc) {
        if (p.epilogue == EPI_COLNORM) return p.ksplit == 1 ? launch_inst<false, false, false, EPI_COLNORM>(p, stream) : -1;
        if (p.epilogue == EPI_STORE_COLNORM) return p.ksplit == 1 && !p.C2 ? launch_inst<false, false, false, EPI_STORE_COLNORM>(p, stream) : -1;
        return launch_inst<false, false, false, EPI_STORE>(p, stream);
    }
    if (p.a_kc && !p.b_kc) {
        if (p.epilogue == EPI_COLNORM) return p.ksplit == 1 && !p.C2 ? launch_inst<true, false, false, EPI_COLNORM>(p, stream) : -1;
        if (p.epilogue == EPI_STORE_COLNORM) return p.ksplit == 1 && !p.C2 ? launch_inst<true, false, false, EPI_STORE_COLNORM>(p, stream) : -1;
        if (p.epilogue != EPI_STORE) return -1;
        return launch_inst<true, false, false, EPI_STORE>(p, stream);
    }
    return -1;
}

int splitk_reduce_launch(const GemmP& p, cudaStream_t stream) {
    dim3 grid(p.n / BN, p.m / BM, p.batch * RED_SLICES);
    launch_k(p.pdl != 0, splitk_reduce_kernel, grid, 256, 0, stream, p);
    return count_launch();
}

int gemm_launch_auto(GemmP p, cudaStream_t stream, double* ws, size_t ws_doubles) {
    static int sms = 0;
    if (!sms) {
        int dev = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
        if (sms <= 0) sms = 148;
    }
    p.pdl = 1;   // the M x M chains: programmatic dependent launch (see common.cuh)
    const bool eligible = ws && p.ksplit == 1 && !p.C2 && !p.gvec && !p.kscale && p.epilogue == EPI_STORE && p.m % BM == 0 && p.n % BN == 0;
    if (eligible) {
        const long nti = p.m / BM, ntj = p.n / BN;
        long tiles = p.lower_out ? (ntj >= nti ? nti * (nti + 1) / 2 : nti * ntj - ntj * (ntj - 1) / 2) : nti * ntj;   // tiles with tj <= ti
        if (p.row_mod > 1) tiles = (tiles + p.row_mod - 1) / p.row_mod;
        tiles *= p.batch;
        // contraction length a typical tile sees (triangular operands skip about half of their k-blocks)
        long keff = p.k;
        if (p.a_tri || p.b_tri) keff = keff / 2 > BM ? keff / 2 : (keff < BM ? keff : BM);
        const long kt = keff / BK;
        long ks = tiles > 0 ? sms / tiles : 1;
        if (ks > kt / 2) ks = kt / 2;                       // at least two k-tiles per piece
        const size_t slab = (size_t)p.batch * p.m * p.n;    // compact partial image of C
        if (slab > 0 && ks > (long)(ws_doubles / slab)) ks = (long)(ws_doubles / slab);
        if (ks > 16) ks = 16;
        if (ks >= 2) {
            p.ksplit = (int)ks; p.part = ws; p.part_stride = (long)slab; p.part_ld = p.n; p.part_sC = (long)p.m * p.n;
            int e = gemm_launch(p, stream);
            if (e) return e;
            return splitk_reduce_launch(p, stream);
        }
    }
    return gemm_launch(p, stream);
}

}  // namespace tsvgp
