// INT8 tensor-core peak probe for B200 (sm_100a): the sustained rate of tcgen05.mma.kind::i8 (SASS UTCIMMA), s8 x s8 -> s32 in
// tensor memory, from one persistent CTA per SM.
//   resident : operands stay in shared memory, one thread issues 128 x N x 32 MMAs back to back
//   streamed : a 4-stage mbarrier ring fed by cp.async.bulk (one 128-row x 128-byte A k-block + one N-row B k-block per stage)
//              from a 32 MB operand image laid out as the Gram product's residue planes ([k-block][128-row block][16 KB])
//   pair     : the same stream into CTA pairs (clusters of 2): 256 x 256 x 32 MMAs (cta_group::2) issued by the leader, each CTA
//              loading one 128-row A and one 128-row B k-block per stage (32 KB), 6 stages; as many pairs as can be resident
// Both operand layouts are checked bit-exactly against the host first: K-major core matrices without swizzle, and 128-byte swizzle.
// Tooling only (not part of the product library). Build: see tools/Makefile.
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>
#include <cuda_runtime.h>

#define CK(x) do { cudaError_t e = (x); if (e != cudaSuccess) { printf("CUDA error %s at %s:%d\n", cudaGetErrorString(e), __FILE__, __LINE__); exit(1);} } while (0)

__device__ __forceinline__ uint32_t sa(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* b, uint32_t n) { asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(sa(b)), "r"(n)); }
__device__ __forceinline__ void mbar_wait(uint64_t* b, uint32_t parity) {
    asm volatile("{\n.reg .pred P1;\nW1:\nmbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n@P1 bra D1;\nbra W1;\nD1:\n}\n" ::"r"(sa(b)),
                 "r"(parity) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* b, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(sa(b)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* b) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(sa(dst)), "l"(src), "r"(bytes),
                 "r"(sa(b)) : "memory");
}
// shared-memory matrix descriptor (tcgen05): start, leading / stride byte offsets, version 1, swizzle mode (0 none, 2 = 128 B)
__device__ __forceinline__ uint64_t sdesc(uint32_t saddr, uint32_t lbo, uint32_t sbo, uint32_t swz) {
    return (uint64_t)((saddr >> 4) & 0x3FFF) | (uint64_t)((lbo >> 4) & 0x3FFF) << 16 | (uint64_t)((sbo >> 4) & 0x3FFF) << 32 | 1ull << 46 |
           (uint64_t)swz << 61;
}
// instruction descriptor: D s32, A and B signed 8-bit, both K-major, M = 128
__host__ __device__ constexpr uint32_t idesc_i8(int n) { return 2u << 4 | 1u << 7 | 1u << 10 | (uint32_t)(n >> 3) << 17 | (128u >> 4) << 24; }
__device__ __forceinline__ void mma_i8(uint32_t d, uint64_t a, uint64_t b, uint32_t idesc, uint32_t acc) {
    asm volatile("{\n.reg .pred p;\nsetp.ne.b32 p, %4, 0;\ntcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, p;\n}\n" ::"r"(d), "l"(a), "l"(b),
                 "r"(idesc), "r"(acc));
}
__device__ __forceinline__ void mma_commit(uint64_t* b) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(sa(b)) : "memory");
}
__device__ __forceinline__ void tmem_alloc(uint32_t* slot, uint32_t cols) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(sa(slot)), "r"(cols));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t t, uint32_t cols) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(t), "r"(cols));
}

// operand k-block layout: byte (row r, k) of a tile of R rows x 128 bytes
__host__ __device__ inline uint32_t kblock_off(int r, int k, int swz) {
    if (swz) return (r >> 3) * 1024 + (r & 7) * 128 + ((((k >> 4) ^ (r & 7)) << 4) | (k & 15));
    return (r >> 3) * 1024 + (k >> 4) * 128 + (r & 7) * 16 + (k & 15);
}

// one 128 x N x 128 product of k-block images A (16 KB) and B (N x 128 B), D written row-major s32 [128][N]
template <int N>
__global__ void __launch_bounds__(128, 1) k_verify(const int8_t* gA, const int8_t* gB, int32_t* D, int swz) {
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    uint8_t* smem = smem_raw + ((1024 - (sa(smem_raw) & 1023)) & 1023);   // 128-byte swizzle atoms sit on 1 KB boundaries
    __shared__ uint64_t bar[2];
    __shared__ uint32_t tslot;
    uint8_t* sA = smem; uint8_t* sB = smem + 16384;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (warp == 0) tmem_alloc(&tslot, 256 < N ? 512 : 256);
    if (threadIdx.x == 0) { mbar_init(&bar[0], 1); mbar_init(&bar[1], 1); asm volatile("fence.mbarrier_init.release.cluster;"); }
    asm volatile("tcgen05.fence::before_thread_sync;");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;");
    const uint32_t tm = tslot;
    if (threadIdx.x == 0) {
        mbar_expect_tx(&bar[0], 16384 + N * 128);
        bulk_g2s(sA, gA, 16384, &bar[0]);
        bulk_g2s(sB, gB, N * 128, &bar[0]);
        mbar_wait(&bar[0], 0);
        asm volatile("tcgen05.fence::after_thread_sync;");
        for (int kk = 0; kk < 4; ++kk) {
            const uint32_t step = swz ? 32 * kk : 256 * kk;
            mma_i8(tm, sdesc(sa(sA) + step, 128, 1024, swz ? 2 : 0), sdesc(sa(sB) + step, 128, 1024, swz ? 2 : 0), idesc_i8(N), kk > 0);
        }
        mma_commit(&bar[1]);
    }
    mbar_wait(&bar[1], 0);
    __syncwarp();
    asm volatile("tcgen05.fence::after_thread_sync;");
    const int row = warp * 32 + lane;
    for (int c0 = 0; c0 < N; c0 += 8) {
        uint32_t v[8];
        asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];\n"
                     : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7])
                     : "r"(tm + ((uint32_t)(warp * 32) << 16) + c0));
        asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
        for (int j = 0; j < 8; ++j) D[row * N + c0 + j] = (int32_t)v[j];
    }
    asm volatile("tcgen05.fence::before_thread_sync;");
    __syncthreads();
    if (warp == 0) tmem_dealloc(tm, 256 < N ? 512 : 256);
}

// resident operands: `iters` x 4 MMAs (one 128-byte k-block) into two alternating accumulators
template <int N>
__global__ void __launch_bounds__(128, 1) k_resident(int iters, int swz, int32_t* sink) {
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    uint8_t* smem = smem_raw + ((1024 - (sa(smem_raw) & 1023)) & 1023);   // 128-byte swizzle atoms sit on 1 KB boundaries
    __shared__ uint64_t bar;
    __shared__ uint32_t tslot;
    uint8_t* sA = smem; uint8_t* sB = smem + 16384;
    for (int i = threadIdx.x; i < (16384 + N * 128) / 4; i += blockDim.x) ((uint32_t*)smem)[i] = 0x01020304u * (i % 7);
    asm volatile("fence.proxy.async.shared::cta;");
    if (threadIdx.x < 32) tmem_alloc(&tslot, 2 * N);
    if (threadIdx.x == 0) { mbar_init(&bar, 1); asm volatile("fence.mbarrier_init.release.cluster;"); }
    asm volatile("tcgen05.fence::before_thread_sync;");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;");
    const uint32_t tm = tslot;
    if (threadIdx.x == 0) {
        const uint32_t sw = swz ? 2 : 0;
        for (int it = 0; it < iters; ++it)
#pragma unroll
            for (int kk = 0; kk < 4; ++kk) {
                const uint32_t step = swz ? 32 * kk : 256 * kk;
                mma_i8(tm + (it & 1) * N, sdesc(sa(sA) + step, 128, 1024, sw), sdesc(sa(sB) + step, 128, 1024, sw), idesc_i8(N), kk > 0);
            }
        mma_commit(&bar);
    }
    mbar_wait(&bar, 0);
    __syncwarp();
    asm volatile("tcgen05.fence::after_thread_sync;");
    uint32_t v;
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x1.b32 {%0}, [%1];\ntcgen05.wait::ld.sync.aligned;" : "=r"(v) : "r"(tm + ((uint32_t)((threadIdx.x >> 5) * 32) << 16)));
    if (v == 0x7fffffffu) sink[blockIdx.x] = v;
    asm volatile("tcgen05.fence::before_thread_sync;");
    __syncthreads();
    if (threadIdx.x < 32) tmem_dealloc(tm, 2 * N);
}

// streamed operands: warp 0 feeds a STAGES-deep ring with bulk copies, warp 1 issues the MMAs and releases each stage by commit.
// Work unit u (strided over the CTAs): A = 128-row block u % nrb, B = the N/128 row blocks from (u / nrb) * N/128, all nkb k-blocks.
template <int N, int STAGES>
__global__ void __launch_bounds__(128, 1) k_stream(const int8_t* img, int nrb, int nkb, int units, int swz, int32_t* sink) {
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    uint8_t* smem = smem_raw + ((1024 - (sa(smem_raw) & 1023)) & 1023);   // 128-byte swizzle atoms sit on 1 KB boundaries
    __shared__ uint64_t full[STAGES], empty[STAGES], done;
    __shared__ uint32_t tslot;
    constexpr uint32_t SA = 16384, SB = N * 128, SS = SA + SB;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (warp == 0) tmem_alloc(&tslot, 2 * N);
    if (threadIdx.x == 0) {
        for (int s = 0; s < STAGES; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); }
        mbar_init(&done, 1);
        asm volatile("fence.mbarrier_init.release.cluster;");
    }
    asm volatile("tcgen05.fence::before_thread_sync;");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;");
    const uint32_t tm = tslot;
    const int nb = N / 128;
    if (warp == 0 && lane == 0) {
        int k = 0;
        for (int u = blockIdx.x; u < units; u += gridDim.x) {
            const int ra = u % nrb, rb = ((u / nrb) * nb) % nrb;
            for (int kb = 0; kb < nkb; ++kb, ++k) {
                const int s = k % STAGES;
                if (k >= STAGES) mbar_wait(&empty[s], ((k / STAGES) - 1) & 1);
                uint8_t* st = smem + s * SS;
                mbar_expect_tx(&full[s], SS);
                bulk_g2s(st, img + ((size_t)kb * nrb + ra) * 16384, SA, &full[s]);
                bulk_g2s(st + SA, img + ((size_t)kb * nrb + rb) * 16384, SB, &full[s]);
            }
        }
    } else if (warp == 1 && lane == 0) {
        int k = 0, t = 0;
        const uint32_t sw = swz ? 2 : 0;
        for (int u = blockIdx.x; u < units; u += gridDim.x, ++t) {
            for (int kb = 0; kb < nkb; ++kb, ++k) {
                const int s = k % STAGES;
                mbar_wait(&full[s], (k / STAGES) & 1);
                asm volatile("tcgen05.fence::after_thread_sync;");
                const uint32_t a = sa(smem + s * SS), b = a + SA;
#pragma unroll
                for (int kk = 0; kk < 4; ++kk) {
                    const uint32_t step = swz ? 32 * kk : 256 * kk;
                    mma_i8(tm + (t & 1) * N, sdesc(a + step, 128, 1024, sw), sdesc(b + step, 128, 1024, sw), idesc_i8(N), kb > 0 || kk > 0);
                }
                mma_commit(&empty[s]);
            }
        }
        mma_commit(&done);
    }
    __syncwarp();
    mbar_wait(&done, 0);
    __syncwarp();
    asm volatile("tcgen05.fence::after_thread_sync;");
    uint32_t v;
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x1.b32 {%0}, [%1];\ntcgen05.wait::ld.sync.aligned;" : "=r"(v) : "r"(tm + ((uint32_t)(warp * 32) << 16)));
    if (v == 0x7fffffffu) sink[blockIdx.x] = v;
    asm volatile("tcgen05.fence::before_thread_sync;");
    __syncthreads();
    if (warp == 0) tmem_dealloc(tm, 2 * N);
}

// streamed CTA pairs: pair unit u has A = pair row u % (nrb / 2), B = pair row (u / (nrb / 2)) % (nrb / 2); rank r loads row 2I + r
// of each.  Rank 1's copies complete on its own barrier and one thread forwards them to the leader's (as the Gram product does).
template <int STAGES>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(128, 1) k_stream_pair(const int8_t* img, int nrb, int nkb, int units, int32_t* sink) {
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    uint8_t* smem = smem_raw + ((1024 - (sa(smem_raw) & 1023)) & 1023);
    __shared__ uint64_t full[STAGES], empty[STAGES], done;
    __shared__ uint32_t tslot;
    constexpr uint32_t SA = 16384, SS = 2 * SA;
    constexpr uint32_t IDESC2 = 2u << 4 | 1u << 7 | 1u << 10 | (256u >> 3) << 17 | (256u >> 4) << 24;   // M = 256, N = 256
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    uint32_t rank;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(rank));
    const int pr = nrb / 2, pair = blockIdx.x >> 1, npairs = gridDim.x >> 1;
    if (threadIdx.x == 0) {
        for (int s = 0; s < STAGES; ++s) { mbar_init(&full[s], rank == 0 ? 2 : 1); mbar_init(&empty[s], 1); }
        mbar_init(&done, 1);
        asm volatile("fence.mbarrier_init.release.cluster;");
    }
    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], 512;" ::"r"(sa(&tslot)));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;");
    }
    asm volatile("tcgen05.fence::before_thread_sync;");
    asm volatile("barrier.cluster.arrive.release;\nbarrier.cluster.wait.acquire;" ::: "memory");
    asm volatile("tcgen05.fence::after_thread_sync;");
    const uint32_t tm = tslot;
    if (warp == 0 && lane == 0) {   // producer
        int k = 0;
        for (int u = pair; u < units; u += npairs) {
            const int ra = 2 * (u % pr) + rank, rb = 2 * ((u / pr) % pr) + rank;
            for (int kb = 0; kb < nkb; ++kb, ++k) {
                const int s = k % STAGES;
                if (k >= STAGES) mbar_wait(&empty[s], ((k / STAGES) - 1) & 1);
                uint8_t* st = smem + s * SS;
                mbar_expect_tx(&full[s], SS);
                bulk_g2s(st, img + ((size_t)kb * nrb + ra) * 16384, SA, &full[s]);
                bulk_g2s(st + SA, img + ((size_t)kb * nrb + rb) * 16384, SA, &full[s]);
            }
        }
    } else if (warp == 1 && lane == 0 && rank != 0) {   // forward rank 1's stages to the leader
        int k = 0;
        for (int u = pair; u < units; u += npairs)
            for (int kb = 0; kb < nkb; ++kb, ++k) {
                const int s = k % STAGES;
                mbar_wait(&full[s], (k / STAGES) & 1);
                uint32_t ra;
                asm volatile("mapa.shared::cluster.u32 %0, %1, 0;" : "=r"(ra) : "r"(sa(&full[s])));
                asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(ra) : "memory");
            }
    } else if (warp == 1 && lane == 0) {   // MMA issuer (leader)
        int k = 0, t = 0;
        for (int u = pair; u < units; u += npairs, ++t) {
            for (int kb = 0; kb < nkb; ++kb, ++k) {
                const int s = k % STAGES;
                asm volatile("{\n.reg .pred P1;\nWC:\nmbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n@P1 bra DC;\n"
                             "bra WC;\nDC:\n}\n" ::"r"(sa(&full[s])), "r"((k / STAGES) & 1) : "memory");
                asm volatile("tcgen05.fence::after_thread_sync;");
                const uint32_t a = sa(smem + s * SS), b = a + SA;
#pragma unroll
                for (int kk = 0; kk < 4; ++kk)
                    asm volatile("{\n.reg .pred p;\nsetp.ne.b32 p, %4, 0;\ntcgen05.mma.cta_group::2.kind::i8 [%0], %1, %2, %3, p;\n}\n"
                                 ::"r"(tm + (t & 1) * 256), "l"(sdesc(a + 32 * kk, 128, 1024, 2)), "l"(sdesc(b + 32 * kk, 128, 1024, 2)),
                                 "r"(IDESC2), "r"((uint32_t)(kb > 0 || kk > 0)));
                asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
                             ::"r"(sa(&empty[s])), "h"((uint16_t)3) : "memory");
            }
        }
        asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
                     ::"r"(sa(&done)), "h"((uint16_t)3) : "memory");
    }
    __syncwarp();
    if (pair < units) mbar_wait(&done, 0);   // a pair without units issues no commit
    __syncwarp();
    asm volatile("tcgen05.fence::after_thread_sync;");
    uint32_t v;
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x1.b32 {%0}, [%1];\ntcgen05.wait::ld.sync.aligned;" : "=r"(v) : "r"(tm + ((uint32_t)(warp * 32) << 16)));
    if (v == 0x7fffffffu) sink[blockIdx.x] = v;
    asm volatile("tcgen05.fence::before_thread_sync;");
    asm volatile("barrier.cluster.arrive.release;\nbarrier.cluster.wait.acquire;" ::: "memory");
    asm volatile("tcgen05.fence::after_thread_sync;");
    if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, 512;" ::"r"(tm));
}

static float time_ms(cudaEvent_t a, cudaEvent_t b) { float ms; cudaEventElapsedTime(&ms, a, b); return ms; }

static void smi(const char* tag) {
    FILE* f = popen("nvidia-smi --query-gpu=name,power.limit,power.draw,clocks.sm,clocks.max.sm --format=csv,noheader -i 0", "r");
    char line[512] = {0};
    if (f) { if (!fgets(line, sizeof line, f)) line[0] = 0; pclose(f); }
    printf("nvidia-smi [%s]: %s", tag, line[0] ? line : "(unavailable)\n");
}

template <int N>
static bool verify(int swz) {
    std::vector<int8_t> a(128 * 128), b(N * 128), ia(16384), ib(N * 128);
    uint32_t st = 12345u + N + swz;
    auto rnd = [&]() { st = st * 1664525u + 1013904223u; return (int8_t)(st >> 24); };
    for (auto& x : a) x = rnd();
    for (auto& x : b) x = rnd();
    for (int r = 0; r < 128; ++r) for (int k = 0; k < 128; ++k) ia[kblock_off(r, k, swz)] = a[r * 128 + k];
    for (int r = 0; r < N; ++r) for (int k = 0; k < 128; ++k) ib[kblock_off(r, k, swz)] = b[r * 128 + k];
    int8_t *dA, *dB; int32_t* dD;
    CK(cudaMalloc(&dA, ia.size())); CK(cudaMalloc(&dB, ib.size())); CK(cudaMalloc(&dD, 4 * 128 * N));
    CK(cudaMemcpy(dA, ia.data(), ia.size(), cudaMemcpyHostToDevice));
    CK(cudaMemcpy(dB, ib.data(), ib.size(), cudaMemcpyHostToDevice));
    CK(cudaMemset(dD, 0, 4 * 128 * N));
    const int sm_bytes = 16384 + N * 128 + 1024;
    CK(cudaFuncSetAttribute(k_verify<N>, cudaFuncAttributeMaxDynamicSharedMemorySize, sm_bytes));
    k_verify<N><<<1, 128, sm_bytes>>>(dA, dB, dD, swz);
    CK(cudaDeviceSynchronize());
    std::vector<int32_t> d(128 * N);
    CK(cudaMemcpy(d.data(), dD, 4 * d.size(), cudaMemcpyDeviceToHost));
    long bad = 0;
    for (int i = 0; i < 128; ++i)
        for (int j = 0; j < N; ++j) {
            int32_t ref = 0;
            for (int k = 0; k < 128; ++k) ref += (int32_t)a[i * 128 + k] * (int32_t)b[j * 128 + k];
            if (ref != d[i * N + j] && bad++ < 4) printf("  mismatch (%d,%d): got %d want %d\n", i, j, d[i * N + j], ref);
        }
    printf("verify 128x%dx128 %s: %s (%ld of %d entries differ)\n", N, swz ? "swizzle-128B" : "no-swizzle", bad ? "FAIL" : "exact", bad, 128 * N);
    cudaFree(dA); cudaFree(dB); cudaFree(dD);
    return bad == 0;
}

template <int N>
static void resident(int sms, int32_t* sink, cudaEvent_t e0, cudaEvent_t e1, int swz, int iters) {
    const int sm_bytes = 16384 + N * 128 + 1024;
    CK(cudaFuncSetAttribute(k_resident<N>, cudaFuncAttributeMaxDynamicSharedMemorySize, sm_bytes));
    k_resident<N><<<sms, 128, sm_bytes>>>(iters / 8, swz, sink);
    CK(cudaDeviceSynchronize());
    cudaEventRecord(e0);
    k_resident<N><<<sms, 128, sm_bytes>>>(iters, swz, sink);
    cudaEventRecord(e1); CK(cudaDeviceSynchronize());
    const float ms = time_ms(e0, e1);
    const double ops = 2.0 * sms * iters * 4.0 * 128 * N * 32;
    printf("resident 128x%dx32 %s: %8.3f ms  %7.1f TOP/s\n", N, swz ? "sw128" : "noswz", ms, ops / ms * 1e-9);
}

template <int N, int STAGES>
static double stream(int sms, const int8_t* img, int nrb, int nkb, int units, int32_t* sink, cudaEvent_t e0, cudaEvent_t e1, int swz, int reps,
                     bool print = true) {
    const int sm_bytes = STAGES * (16384 + N * 128) + 1024;
    CK(cudaFuncSetAttribute(k_stream<N, STAGES>, cudaFuncAttributeMaxDynamicSharedMemorySize, sm_bytes));
    k_stream<N, STAGES><<<sms, 128, sm_bytes>>>(img, nrb, nkb, units, swz, sink);
    CK(cudaDeviceSynchronize());
    cudaEventRecord(e0);
    for (int r = 0; r < reps; ++r) k_stream<N, STAGES><<<sms, 128, sm_bytes>>>(img, nrb, nkb, units, swz, sink);
    cudaEventRecord(e1); CK(cudaDeviceSynchronize());
    const float ms = time_ms(e0, e1) / reps;
    const double ops = 2.0 * units * 128.0 * N * 128.0 * nkb;
    const double bytes = (double)units * nkb * (16384 + N * 128);
    if (print)
        printf("streamed 128x%d %d stages %s, %d units x %d k-blocks: %8.3f ms  %7.1f TOP/s  (smem fill %.1f TB/s)\n", N, STAGES,
               swz ? "sw128" : "noswz", units, nkb, ms, ops / ms * 1e-9, bytes / ms * 1e-9);
    return ops / ms * 1e-9;
}

template <int STAGES>
static void stream_pair(const int8_t* img, int nrb, int nkb, int units, int32_t* sink, cudaEvent_t e0, cudaEvent_t e1, int reps) {
    const int sm_bytes = STAGES * 32768 + 1024;
    CK(cudaFuncSetAttribute(k_stream_pair<STAGES>, cudaFuncAttributeMaxDynamicSharedMemorySize, sm_bytes));
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(2); cfg.blockDim = dim3(128); cfg.dynamicSmemBytes = sm_bytes;
    int clusters = 0;
    CK(cudaOccupancyMaxActiveClusters(&clusters, k_stream_pair<STAGES>, &cfg));
    const int grid = 2 * clusters;
    k_stream_pair<STAGES><<<grid, 128, sm_bytes>>>(img, nrb, nkb, units, sink);
    CK(cudaDeviceSynchronize());
    cudaEventRecord(e0);
    for (int r = 0; r < reps; ++r) k_stream_pair<STAGES><<<grid, 128, sm_bytes>>>(img, nrb, nkb, units, sink);
    cudaEventRecord(e1); CK(cudaDeviceSynchronize());
    const float ms = time_ms(e0, e1) / reps;
    const double ops = 2.0 * units * 256.0 * 256 * 128.0 * nkb;
    const double bytes = (double)units * nkb * 2 * 32768;
    printf("streamed pairs 256x256 %d stages sw128, %d pair units x %d k-blocks, %d CTAs (%d resident clusters): %8.3f ms  %7.1f TOP/s  "
           "(smem fill %.1f TB/s)\n", STAGES, units, nkb, grid, clusters, ms, ops / ms * 1e-9, bytes / ms * 1e-9);
}

int main() {
    cudaDeviceProp p; CK(cudaGetDeviceProperties(&p, 0));
    const int sms = p.multiProcessorCount;
    int clk_khz = 0; cudaDeviceGetAttribute(&clk_khz, cudaDevAttrClockRate, 0);
    printf("device %s sms %d cc %d.%d clockRate(attr) %d kHz\n", p.name, sms, p.major, p.minor, clk_khz);
    smi("idle");
    bool ok = true;
    ok &= verify<128>(0); ok &= verify<128>(1); ok &= verify<256>(0); ok &= verify<256>(1);
    if (!ok) { printf("layout check failed: no rates reported\n"); return 1; }
    int32_t* sink; CK(cudaMalloc(&sink, 4 * sms));
    cudaEvent_t e0, e1; cudaEventCreate(&e0); cudaEventCreate(&e1);
    for (int swz = 0; swz < 2; ++swz) { resident<128>(sms, sink, e0, e1, swz, 200000); resident<256>(sms, sink, e0, e1, swz, 100000); }
    // the Gram product's operand image at M = 2048, a 16 384-point slab: 16 row blocks x 128 k-blocks x 16 KB = 32 MB (one modulus)
    const int nrb = 16, nkb = 128;
    int8_t* img; CK(cudaMalloc(&img, (size_t)nrb * nkb * 16384));
    CK(cudaMemset(img, 3, (size_t)nrb * nkb * 16384));
    // 72 lower 128 x 256 blocks per modulus, 16 moduli: 1152 units per slab
    for (int swz = 0; swz < 2; ++swz) {
        stream<128, 6>(sms, img, nrb, nkb, 1152 * 2, sink, e0, e1, swz, 5);
        stream<256, 4>(sms, img, nrb, nkb, 1152, sink, e0, e1, swz, 5);
    }
    // the same work in 576 pair units of 256 x 256
    stream_pair<6>(img, nrb, nkb, 576, sink, e0, e1, 5);
    // sustained: ~2 s of the streamed 128 x 256 loop, clocks sampled while it runs
    {
        const int reps = 60;
        const int sm_bytes = 4 * (16384 + 256 * 128) + 1024;
        cudaEventRecord(e0);
        for (int r = 0; r < reps; ++r) k_stream<256, 4><<<sms, 128, sm_bytes>>>(img, nrb, nkb, 1152, 1, sink);
        cudaEventRecord(e1);
        for (int i = 0; i < 3; ++i) smi("under load");
        CK(cudaDeviceSynchronize());
        const float ms = time_ms(e0, e1);
        const double ops = reps * 2.0 * 1152 * 128.0 * 256 * 128.0 * nkb;
        printf("streamed 128x256 sw128 sustained (%.0f ms): %.1f TOP/s\n", ms, ops / ms * 1e-9);
    }
    smi("after");
    cudaFree(img); cudaFree(sink);
    return 0;
}
