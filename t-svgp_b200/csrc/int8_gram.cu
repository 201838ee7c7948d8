// Exact fixed-point Gram product on the INT8 tensor cores (tcgen05.mma kind::i8, SASS UTCIMMA): see int8_gram.cuh and DESIGN §2.
//   i8_residue_kernel : K (FP64 slab) -> A = rint(K 2^52 / v) -> 64-bit integer -> three 18-bit limbs -> 16 int8 residue planes
//                       (integer arithmetic: one multiply-high per modulus), written as the shared-memory image the MMA descriptors
//                       describe (128-row x 128-byte k-blocks of K-major core matrices, 128-byte swizzle)
//   i8_gram_kernel    : persistent CTA pairs, warp-specialised: in each CTA one producer thread streams k-blocks into a 6-stage
//                       mbarrier ring with cp.async.bulk; the pair's leader issues 256 x 256 x 32 MMAs (cta_group::2) into a
//                       double-buffered TMEM accumulator; four epilogue warps per CTA reduce the int32 tiles modulo p_i into
//                       residue tiles.  Modulus-major schedule: the lower 256 x 256 blocks of modulus i, then i + 1 (one modulus's
//                       planes stay in L2 while its blocks run)
//   i8_crt_kernel     : Garner's mixed-radix digits (one reduction per digit) + Horner in 128-bit integers -> the exact integer ->
//                       one rounding -> C += alpha ...
#include "int8_gram.cuh"
#include "common.cuh"

namespace tsvgp {

namespace i8 {

constexpr int KB_BYTES = 16384;                 // one 128-row x 128-byte k-block
constexpr int BN = 256;                         // accumulator columns: two 128-tiles of one tile row per CTA
constexpr int STAGES = 6;
constexpr int STAGE_BYTES = 2 * KB_BYTES;       // one CTA's A and B row blocks of one k-block
constexpr int GEMM_SMEM = STAGES * STAGE_BYTES + 1024;
constexpr int GEMM_THREADS = 192;               // warp 0 producer, warp 1 MMA issuer (rank 0) or stage forwarder (rank 1), warps 2..5 epilogue

__host__ __device__ constexpr int modulus(int i) {
    constexpr int p[I8_NMOD] = {256, 255, 253, 251, 247, 241, 239, 233, 229, 227, 223, 217, 211, 199, 197, 193};
    return p[i];
}
__host__ __device__ constexpr int inv_mod(int a, int m) {   // a^-1 mod m (a, m coprime)
    int t = 0, nt = 1, r = m, nr = a % m;
    while (nr) { const int q = r / nr, t2 = t - q * nt, r2 = r - q * nr; t = nt; nt = t2; r = nr; nr = r2; }
    return t < 0 ? t + m : t;
}
__host__ __device__ constexpr unsigned __int128 prod_moduli() {
    unsigned __int128 P = 1;
    for (int i = 0; i < I8_NMOD; ++i) P *= (unsigned)modulus(i);
    return P;
}

// byte offset of (row r, byte k) inside a k-block: 8-row x 128-byte swizzle atoms, 16-byte chunk c of row r at c ^ (r & 7)
__device__ __forceinline__ uint32_t kblock_off(int r, int k) {
    return (r >> 3) * 1024 + (r & 7) * 128 + ((((k >> 4) ^ (r & 7)) << 4) | (k & 15));
}

// lower 128 x 256 blocks of one modulus: tile row i holds ceil((i + 1) / 2) blocks of two tiles.  The product kernel takes this count
// (its `nblk`) for the tile count it names; it schedules 256 x 256 pair blocks
__host__ __device__ inline int blocks_per_modulus(int nt) {
    int n = 0;
    for (int i = 0; i < nt; ++i) n += (i + 2) / 2;
    return n;
}

// ---- tcgen05 -------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t saddr(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
// shared-memory matrix descriptor: start >> 4, stride between 8-row groups 1024 B, version 1 (bit 46), 128-byte swizzle (mode 2)
__device__ __forceinline__ uint64_t sdesc(uint32_t a) {
    return (uint64_t)((a >> 4) & 0x3FFF) | (uint64_t)(1024 >> 4) << 32 | 1ull << 46 | 2ull << 61;
}
// instruction descriptor: D s32, A and B signed 8-bit, both K-major, M = 256 (a CTA pair), N = BN
constexpr uint32_t IDESC = 2u << 4 | 1u << 7 | 1u << 10 | (uint32_t)(BN >> 3) << 17 | (256u >> 4) << 24;
__device__ __forceinline__ void fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&v)[32]) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,"
                 "%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];\n"
                 "tcgen05.wait::ld.sync.aligned;\n"
                 : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]), "=r"(v[9]),
                   "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]), "=r"(v[17]), "=r"(v[18]),
                   "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]),
                   "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
                 : "r"(taddr)
                 : "memory");
}

// ---- residues --------------------------------------------------------------------------------------------------------------
// x mod p for x <= MOD_X_MAX by one multiply-high: q = floor(x m / 2^36) with m = ceil(2^36 / p) is floor(x / p) while x (m p - 2^36)
// < 2^36 (the error x (m p - 2^36) / (p 2^36) stays below 1 / p); both callers' bounds are checked at compile time below
constexpr uint32_t MOD_X_MAX = (1u << 28) - 1;
__host__ __device__ constexpr uint32_t mod_magic(int p) { return (uint32_t)(((1ull << 36) + p - 1) / p); }
__host__ __device__ constexpr bool mod_magic_exact(int i) {
    return i == I8_NMOD || ((uint64_t)MOD_X_MAX * ((uint64_t)mod_magic(modulus(i)) * modulus(i) - (1ull << 36)) < (1ull << 36) &&
                            mod_magic_exact(i + 1));
}
static_assert(mod_magic_exact(0), "mod_small: the multiply-high quotient is exact for x <= MOD_X_MAX");
template <int P>
__device__ __forceinline__ uint32_t mod_small(uint32_t x) {   // x mod P, x <= MOD_X_MAX
    return x - (__umulhi(x, mod_magic(P)) >> 4) * P;
}

// The grid integer t (|t| < 2^53) enters as u = t + 2^53 in [1, 2^54), split into 18-bit limbs u = l2 2^36 + l1 2^18 + l0.  For an
// odd modulus p with h = (p - 1) / 2,  x = l2 (2^36 mod p) + l1 (2^18 mod p) + l0 + ((h - 2^53) mod p)  is t + h (mod p) and below
// 2^27, so  (x mod p) - h  is t's residue in the symmetric range [-h, h].  Modulus 256 is t's low byte (2^53 = 0 mod 256), the
// two's complement of its residue in [-128, 127].
struct Limbs { uint32_t l0, l1, l2; };
__device__ __forceinline__ Limbs limbs_of(double t) {
    const uint64_t u = (uint64_t)(__double2ll_rn(t) + (1ll << 53));
    const uint32_t lo = (uint32_t)u, hi = (uint32_t)(u >> 32);
    return {lo & 0x3FFFF, __funnelshift_r(lo, hi, 18) & 0x3FFFF, hi >> 4};
}
template <int M>
__device__ __forceinline__ uint32_t residue_byte(const Limbs& a) {   // symmetric residue mod p_M; only the low byte counts
    constexpr int p = modulus(M), h = (p - 1) / 2;
    constexpr uint32_t c18 = (1u << 18) % p, c36 = (uint32_t)((1ull << 36) % p);
    constexpr uint32_t off = (uint32_t)((h + p - (int)((1ull << 53) % p)) % p);
    if constexpr (M == 0) {
        return a.l0;
    } else {
        const uint32_t x = a.l2 * c36 + a.l1 * c18 + a.l0 + off;
        return mod_small<p>(x) - h;
    }
}
template <int M>
__device__ __forceinline__ uint32_t residue4(const Limbs* a) {   // 4 residue bytes, packed
    return __byte_perm(__byte_perm(residue_byte<M>(a[0]), residue_byte<M>(a[1]), 0x0040),
                       __byte_perm(residue_byte<M>(a[2]), residue_byte<M>(a[3]), 0x0040), 0x5410);
}
template <int M>
__device__ __forceinline__ void store_residues(const Limbs* a, int8_t* dst, size_t pstride) {
    if constexpr (M < I8_NMOD) {
        uint4 w;
        w.x = residue4<M>(a); w.y = residue4<M>(a + 4); w.z = residue4<M>(a + 8); w.w = residue4<M>(a + 12);
        *reinterpret_cast<uint4*>(dst + M * pstride) = w;
        store_residues<M + 1>(a, dst, pstride);
    }
}

// block (kb, rb): one 128-row x 128-column k-block of every plane; a thread takes 16 consecutive columns of a row (one chunk)
__global__ void __launch_bounds__(256) i8_residue_kernel(const double* __restrict__ K, long ldk, double scale, int8_t* __restrict__ planes,
                                                         size_t pstride, int nrb) {
    const int kb = blockIdx.x, rb = blockIdx.y;
#pragma unroll 1
    for (int it = 0; it < 4; ++it) {
        const int c = threadIdx.x + 256 * it, row = c >> 3, kc = c & 7;
        const double2* src = reinterpret_cast<const double2*>(K + (size_t)(rb * 128 + row) * ldk + kb * 128 + kc * 16);
        double k[16];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const double2 v = __ldg(src + j);
            k[2 * j] = v.x; k[2 * j + 1] = v.y;
        }
        Limbs a[16];
#pragma unroll
        for (int j = 0; j < 16; ++j) {
            const double t = rint(k[j] * scale);
            a[j] = limbs_of(fabs(t) < 9007199254740992.0 ? t : 0.0);   // off the grid (non-finite): 0; the point kernel flags such a step
        }
        store_residues<0>(a, planes + (size_t)(kb * nrb + rb) * KB_BYTES + kblock_off(row, kc * 16), pstride);
    }
}

// ---- products --------------------------------------------------------------------------------------------------------------
// CTA pairs (cluster of 2): pair unit (m, I, J <= I) is the 256 x 256 block of pair row I and pair column J of modulus m.  CTA rank r
// loads A = row block 2I + r and B = row block 2J + r (16 KB each per k-block, one copy when I == J); the leader (rank 0) issues
// 256 x 256 x 32 MMAs (cta_group::2), which read A's 256 rows and B's 256 rows from both CTAs' shared memory and leave rank r's 128
// rows, tiles (2I + r, 2J) and (2I + r, 2J + 1), in rank r's TMEM.  Stages are released to both producers by a multicast commit.
// Rank 1's copies complete on its own `full` barrier (a bulk copy signals a barrier of the CTA it writes to); one thread of rank 1
// forwards each completed stage to the leader's `full`, which therefore counts two arrivals.  Pairs depend on no other pair.
__device__ __forceinline__ uint32_t cluster_rank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ uint32_t leader_addr(const void* p) {   // the same shared-memory object in rank 0 of the cluster
    uint32_t a;
    asm volatile("mapa.shared::cluster.u32 %0, %1, 0;" : "=r"(a) : "r"(saddr(p)));
    return a;
}
// An arrival on a barrier of the other CTA.  Its default CTA-scope release is enough: what it orders is data the async proxy wrote
// (a stage a bulk copy completed) or read (TMEM after tcgen05.wait::ld and a tcgen05 fence).  A cluster-scope release would put a
// GPU-wide memory barrier in front of every forwarded stage: measured, that halves the product rate.
__device__ __forceinline__ void mbar_arrive_remote(uint32_t cluster_addr) {
    asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
__device__ __forceinline__ void cluster_sync() {
    asm volatile("barrier.cluster.arrive.release;\nbarrier.cluster.wait.acquire;" ::: "memory");
}
__device__ __forceinline__ void mma_i8_pair(uint32_t d, uint64_t a, uint64_t b, uint32_t acc) {
    asm volatile("{\n.reg .pred p;\nsetp.ne.b32 p, %4, 0;\ntcgen05.mma.cta_group::2.kind::i8 [%0], %1, %2, %3, p;\n}\n" ::"r"(d), "l"(a), "l"(b),
                 "r"(IDESC), "r"(acc));
}
__device__ __forceinline__ void mma_commit_pair(uint64_t* bar) {   // arrive on `bar` in both CTAs once the MMAs issued so far are done
    asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(saddr(bar)),
                 "h"((uint16_t)3) : "memory");
}
__device__ __forceinline__ void pair_coords(int u, int& I, int& J) {
    I = 0;
    while (u > I) { u -= I + 1; ++I; }
    J = u;
}

__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(GEMM_THREADS, 1)
    i8_gram_kernel(const int8_t* __restrict__ planes, size_t pstride, int nrb, int nkb, int nblk, uint8_t* __restrict__ tiles, size_t tstride) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = smem_raw + ((1024 - (saddr(smem_raw) & 1023)) & 1023);   // swizzle atoms on 1 KB boundaries
    __shared__ uint64_t full[STAGES], empty[STAGES], tfull[2], tempty[2];
    __shared__ uint32_t tslot;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t rank = cluster_rank();
    int nt = 0;   // blocks_per_modulus is strictly increasing: nblk names the tile count
    for (int n = 0; n < nblk; ++nt) n += (nt + 2) / 2;
    const int per_mod = (nrb / 2) * (nrb / 2 + 1) / 2, units = I8_NMOD * per_mod;
    const int pair = blockIdx.x >> 1, npairs = gridDim.x >> 1;   // a 1-D grid of clusters of 2: ranks are blockIdx.x & 1
    if (threadIdx.x == 0) {
        for (int s = 0; s < STAGES; ++s) { mbar_init(&full[s], rank == 0 ? 2 : 1); mbar_init(&empty[s], 1); }
        for (int b = 0; b < 2; ++b) { mbar_init(&tfull[b], 1); mbar_init(&tempty[b], 8); }   // the epilogue warps of both CTAs
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) {   // one warp of each CTA: the same 512 columns in both
        asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], 512;" ::"r"(saddr(&tslot)));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;");
    }
    fence_before();
    cluster_sync();
    fence_after();
    const uint32_t tmem = tslot;

    if (warp == 0) {
        if (lane == 0) {   // producer (both CTAs)
            int k = 0;
            for (int u = pair; u < units; u += npairs) {
                const int m = u / per_mod;
                int I, J;
                pair_coords(u - m * per_mod, I, J);
                const int8_t* pa = planes + m * pstride + (size_t)(2 * I + rank) * KB_BYTES;
                const int8_t* pb = planes + m * pstride + (size_t)(2 * J + rank) * KB_BYTES;
                for (int kb = 0; kb < nkb; ++kb, ++k) {
                    const int s = k % STAGES;
                    if (k >= STAGES) mbar_wait(&empty[s], ((k / STAGES) - 1) & 1);
                    uint8_t* st = smem + s * STAGE_BYTES;
                    mbar_expect_tx(&full[s], I == J ? KB_BYTES : 2 * KB_BYTES);
                    tma_bulk_g2s(st, pa + (size_t)kb * nrb * KB_BYTES, KB_BYTES, &full[s]);
                    if (I != J) tma_bulk_g2s(st + KB_BYTES, pb + (size_t)kb * nrb * KB_BYTES, KB_BYTES, &full[s]);
                }
            }
        }
    } else if (warp == 1) {
        if (lane == 0 && rank != 0) {   // forwards rank 1's completed stages to the leader
            int k = 0;
            for (int u = pair; u < units; u += npairs)
                for (int kb = 0; kb < nkb; ++kb, ++k) {
                    const int s = k % STAGES;
                    mbar_wait(&full[s], (k / STAGES) & 1);
                    mbar_arrive_remote(leader_addr(&full[s]));
                }
        } else if (lane == 0) {   // MMA issuer (leader)
            int k = 0, t = 0;
            for (int u = pair; u < units; u += npairs, ++t) {
                int I, J;
                pair_coords(u % per_mod, I, J);
                const int buf = t & 1;
                if (t >= 2) mbar_wait(&tempty[buf], ((t >> 1) - 1) & 1);
                fence_after();
                const uint32_t d = tmem + buf * BN;
                for (int kb = 0; kb < nkb; ++kb, ++k) {
                    const int s = k % STAGES;
                    mbar_wait(&full[s], (k / STAGES) & 1);
                    fence_after();
                    const uint32_t a = saddr(smem + s * STAGE_BYTES), b = I == J ? a : a + KB_BYTES;
#pragma unroll
                    for (int kk = 0; kk < 4; ++kk) mma_i8_pair(d, sdesc(a + 32 * kk), sdesc(b + 32 * kk), (kb | kk) != 0);
                    mma_commit_pair(&empty[s]);
                }
                mma_commit_pair(&tfull[buf]);
            }
        }
    } else {   // epilogue (both CTAs): TMEM lanes 32 (warp % 4) .. + 31 are rows of this CTA's row block
        const int row = (warp & 3) * 32 + lane;
        const uint32_t lane_base = tmem + ((uint32_t)((warp & 3) * 32) << 16);
        int t = 0;
        for (int u = pair; u < units; u += npairs, ++t) {
            const int m = u / per_mod;
            int I, J;
            pair_coords(u - m * per_mod, I, J);
            const int i = 2 * I + rank;   // tile row; i == nt is the padding block of an odd tile count
            const int buf = t & 1;
            mbar_wait(&tfull[buf], (t >> 1) & 1);
            __syncwarp();
            fence_after();
            int pm = 0;
#pragma unroll
            for (int q = 0; q < I8_NMOD; ++q) pm = m == q ? modulus(q) : pm;
            const double ipm = 1.0 / pm;
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                const int j = 2 * J + h;
                if (j > i || i >= nt) break;
                uint8_t* dst = tiles + m * tstride + ((size_t)(i * (i + 1) / 2 + j) * KB_BYTES) + row * 128;
#pragma unroll 1
                for (int c0 = 0; c0 < 128; c0 += 32) {
                    uint32_t v[32];
                    tmem_ld32(lane_base + buf * BN + h * 128 + c0, v);
                    uint32_t w[8];
#pragma unroll
                    for (int e = 0; e < 32; ++e) {
                        const int x = (int)v[e];
                        int r = x - (int)floor((double)x * ipm) * pm;
                        r = r < 0 ? r + pm : (r >= pm ? r - pm : r);
                        if ((e & 3) == 0) w[e >> 2] = 0;
                        w[e >> 2] |= (uint32_t)r << (8 * (e & 3));
                    }
                    uint4* d4 = reinterpret_cast<uint4*>(dst + c0);
                    d4[0] = make_uint4(w[0], w[1], w[2], w[3]);
                    d4[1] = make_uint4(w[4], w[5], w[6], w[7]);
                }
            }
            fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive_remote(leader_addr(&tempty[buf]));
        }
    }
    __syncwarp();
    fence_before();
    cluster_sync();   // every MMA has completed and no CTA of the pair still signals the other's barriers
    fence_after();
    if (warp == 1) {
        __syncwarp();
        asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, 512;" ::"r"(tmem));
    }
}

// ---- reconstruction ----------------------------------------------------------------------------------------------------------
// Garner's digits with one reduction each: x = sum_J v_J prod_{K<J} p_K with 0 <= v_J < p_J, so
//   v_I = (r_I - sum_{J<I} v_J c_IJ) inv_I mod p_I = (r_I inv_I + sum_{J<I} v_J c'_IJ) mod p_I,
// c_IJ = (prod_{K<J} p_K) mod p_I, inv_I = (prod_{K<I} p_K)^-1 mod p_I and c'_IJ = -c_IJ inv_I mod p_I, all compile-time constants.
// The sum is below 16 * 255 * 255 < MOD_X_MAX: one exact reduction per digit.
__host__ __device__ constexpr int prefix_mod(int J, int I) {   // (prod_{K<J} p_K) mod p_I
    int c = 1;
    for (int K = 0; K < J; ++K) c = c * modulus(K) % modulus(I);
    return c;
}
__host__ __device__ constexpr int garner_inv(int I) { return inv_mod(prefix_mod(I, I), modulus(I)); }
__host__ __device__ constexpr int garner_coef(int I, int J) {   // c'_IJ
    return (modulus(I) - prefix_mod(J, I) * garner_inv(I) % modulus(I)) % modulus(I);
}
template <int I, int J>
__device__ __forceinline__ uint32_t garner_sum(uint32_t s, const uint32_t* v) {
    if constexpr (J == I) {
        return s;
    } else {
        constexpr uint32_t c = garner_coef(I, J);
        return garner_sum<I, J + 1>(s + v[J] * c, v);
    }
}
template <int I>
__device__ __forceinline__ void garner(const uint32_t* r, uint32_t* v) {
    if constexpr (I == 0) {
        v[0] = r[0];
        garner<1>(r, v);
    } else if constexpr (I < I8_NMOD) {
        constexpr uint32_t inv = garner_inv(I);
        const uint32_t s = garner_sum<I, 0>(r[I] * inv, v);
        v[I] = mod_small<modulus(I)>(s);
        garner<I + 1>(r, v);
    }
}

__host__ __device__ inline int clz64(uint64_t x) {
#ifdef __CUDA_ARCH__
    return __clzll((long long)x);
#else
    return __builtin_clzll(x);
#endif
}
__host__ __device__ inline double u128_to_double(unsigned __int128 u) {   // correctly rounded (to nearest even)
    const uint64_t hi = (uint64_t)(u >> 64), lo = (uint64_t)u;
    if (hi == 0) return (double)lo;
    const int sh = 64 - clz64(hi);                 // 1 .. 62: the value has 64 + sh significant bits
    uint64_t m = (uint64_t)(u >> sh);              // top 64 bits; what is shifted out only matters as a sticky bit
    if (lo & ((1ull << sh) - 1)) m |= 1;
    return scalbn((double)m, sh);
}

__global__ void __launch_bounds__(256) i8_crt_kernel(const uint8_t* __restrict__ tiles, size_t tstride, double* __restrict__ C, long ldc,
                                                     double scale) {
    constexpr unsigned __int128 P = prod_moduli();
    const int tile = blockIdx.x >> 4;
    int ti = 0;
    while ((ti + 1) * (ti + 2) / 2 <= tile) ++ti;
    const int tj = tile - ti * (ti + 1) / 2;
    const int e = (blockIdx.x & 15) * 1024 + threadIdx.x * 4, row = e >> 7, col = e & 127;
    uint32_t w[I8_NMOD];
#pragma unroll
    for (int m = 0; m < I8_NMOD; ++m) w[m] = __ldg(reinterpret_cast<const uint32_t*>(tiles + m * tstride + (size_t)tile * KB_BYTES + e));
    double out[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        uint32_t r[I8_NMOD], v[I8_NMOD];
#pragma unroll
        for (int m = 0; m < I8_NMOD; ++m) r[m] = (w[m] >> (8 * q)) & 0xFF;
        garner<0>(r, v);
        unsigned __int128 x = v[I8_NMOD - 1];
#pragma unroll
        for (int m = I8_NMOD - 2; m >= 0; --m) x = x * (unsigned)modulus(m) + v[m];
        const bool neg = x > P / 2;   // symmetric range: the exact integer is x - P
        const double d = u128_to_double(neg ? P - x : x);
        out[q] = neg ? -d : d;
    }
    // C + fl(B') scale with one rounding (fma), written out so that it does not rest on the compiler's contraction
    double2* c = reinterpret_cast<double2*>(C + (size_t)(ti * 128 + row) * ldc + tj * 128 + col);
    double2 a = c[0], b = c[1];
    a.x = fma(out[0], scale, a.x); a.y = fma(out[1], scale, a.y); b.x = fma(out[2], scale, b.x); b.y = fma(out[3], scale, b.y);
    c[0] = a; c[1] = b;
}

}  // namespace i8

using namespace i8;

static int plane_row_blocks(int Mp) { return (Mp / 128 + 1) & ~1; }   // even: the last block of an odd tile row reads one past it

size_t i8_plane_bytes(int Mp, long nc) { return (size_t)I8_NMOD * (nc / 128) * plane_row_blocks(Mp) * KB_BYTES; }
size_t i8_tile_bytes(int Mp) {
    const size_t nt = Mp / 128;
    return (size_t)I8_NMOD * nt * (nt + 1) / 2 * KB_BYTES;
}

int i8_planes_init(int8_t* planes, int Mp, long nc_alloc, cudaStream_t s) {
    return (int)cudaMemsetAsync(planes, 0, i8_plane_bytes(Mp, nc_alloc), s);
}

// CTAs of the product launch: two per cluster that can be resident at once (queried once per device and host thread), so that
// every pair runs in the first wave, and at most two per pair unit
static int i8_gram_grid(int nrb, int& grid) {
    thread_local int cached_dev = -1, clusters = 0;
    int dev = 0;
    if (cudaError_t e = cudaGetDevice(&dev)) return (int)e;
    if (dev != cached_dev) {
        if (cudaError_t e = cudaFuncSetAttribute(i8_gram_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, GEMM_SMEM)) return (int)e;
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3(2); cfg.blockDim = dim3(GEMM_THREADS); cfg.dynamicSmemBytes = GEMM_SMEM;
        if (cudaError_t e = cudaOccupancyMaxActiveClusters(&clusters, i8_gram_kernel, &cfg)) return (int)e;
        if (clusters < 1) return (int)cudaErrorInvalidConfiguration;
        cached_dev = dev;
    }
    const int pairs = I8_NMOD * (nrb / 2) * (nrb / 2 + 1) / 2;
    grid = 2 * (pairs < clusters ? pairs : clusters);
    return 0;
}

int i8_syrk_launch(const double* K, long ldk, int Mp, int ncols, double var, double alpha, int8_t* planes, long nc_alloc, uint8_t* tiles,
                   double* C, long ldc, cudaStream_t s) {
    if (ncols <= 0 || ncols % 128 || ncols > I8_MAX_COLS || ncols > nc_alloc || Mp % 128 || ldk % 2 || ldc % 2)
        return (int)cudaErrorInvalidValue;
    const int nt = Mp / 128, nrb = plane_row_blocks(Mp), nkb = ncols / 128;
    const size_t pstride = (size_t)(nc_alloc / 128) * nrb * KB_BYTES;
    const size_t tstride = (size_t)nt * (nt + 1) / 2 * KB_BYTES;
    i8_residue_kernel<<<dim3(nkb, nt), 256, 0, s>>>(K, ldk, 4503599627370496.0 / var, planes, pstride, nrb);
    if (int e = count_launch()) return e;
    int grid = 0;
    if (int e = i8_gram_grid(nrb, grid)) return e;
    i8_gram_kernel<<<grid, GEMM_THREADS, GEMM_SMEM, s>>>(planes, pstride, nrb, nkb, blocks_per_modulus(nt), tiles, tstride);
    if (int e = count_launch()) return e;
    i8_crt_kernel<<<(unsigned)(tstride / KB_BYTES) * 16, 256, 0, s>>>(tiles, tstride, C, ldc, alpha * var * var * 0x1p-104);
    return count_launch();
}

}  // namespace tsvgp
