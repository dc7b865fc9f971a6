// actor_tc.cuh -- the actor's forward pass on the 5th-generation tensor cores (tcgen05, accumulators in TMEM),
// as building blocks shared by the acting kernel (policy_mlp.cu) and the closed-loop rollout kernel (rollout.cu).
// Both kernels run the same warp roles on the same shared-memory map: 8 epilogue warps in two groups of four
// (warp w: TMEM lanes 32 (w % 4) .. + 31, the hardware's lane window of a warp; group w / 4), and warp 8 issues
// the MMAs.  Both kernels run the pass through the functions below (actor_prologue .. actor_normal_draw), so the
// rollout's actions are bit-identical to boatagent_policy_act's.
#pragma once
#include <cstdint>
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <mutex>

#include "../../include/boatenv.h"
#include "common.cuh"

namespace boatenv {

constexpr int kHidden = 256, kTileM = 128, kK1 = 16, kN3 = 16;
constexpr int kEpiThreads = 256, kThreads = kEpiThreads + 32, kMmaWarp = kEpiThreads / 32;
// shared-memory map (bytes).  Operand layout: element (row, k) of an R-row operand sits at
// (k / 8) * (R * 16) + row * 16 + (k % 8) * 2  -- 8x8 core matrices, K-adjacent cores R*16 bytes apart (LBO),
// row groups 128 bytes apart (SBO).
constexpr int kOffW1 = 0;                                   // [256 rows][16]
constexpr int kOffW2 = kOffW1 + kHidden * kK1 * 2;          // [256 rows][256]
constexpr int kOffW3 = kOffW2 + kHidden * kHidden * 2;      // fp32 [16 rows][256], row-major: the heads stay in fp32
constexpr int kOffB1 = kOffW3 + kN3 * kHidden * 4;          // fp32[256]
constexpr int kOffB2 = kOffB1 + kHidden * 4;
constexpr int kOffB3 = kOffB2 + kHidden * 4;                // fp32[16]
constexpr int kBlobBytes = kOffB3 + kN3 * 4;                // what the host packs (BOATAGENT_POLICY_BLOB_BYTES)
static_assert(kBlobBytes == BOATAGENT_POLICY_BLOB_BYTES, "header and kernel disagree on the weight blob");

// UMMA shared-memory descriptor, K-major, no swizzle (cute::UMMA::SmemDescriptor: start >> 4 at [0,14), LBO >> 4 at
// [16,30), SBO >> 4 at [32,46), version 1 at [46,48), layout type 0 at [61,64)).
__device__ __forceinline__ uint64_t umma_desc(uint32_t addr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
    return (uint64_t)((addr >> 4) & 0x3fffu) | ((uint64_t)((lbo_bytes >> 4) & 0x3fffu) << 16) |
           ((uint64_t)((sbo_bytes >> 4) & 0x3fffu) << 32) | (1ull << 46);
}
// Instruction descriptor of tcgen05.mma.kind::f16 (cute::UMMA::InstrDescriptor): D = f32, A = B = bf16, both K-major.
__host__ __device__ constexpr uint32_t umma_idesc(int m, int n) {
    return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(m >> 4) << 24);
}
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
        "}" ::"r"(tmem_d), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void umma_commit(uint64_t *bar) {   // arrives on `bar` when every MMA issued so far is done
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
// 32 consecutive fp32 accumulator columns of this thread's TMEM lane: asynchronous load (the registers are valid after
// tmem_ld_wait()), so the next chunk can be in flight while the current one is processed
__device__ __forceinline__ void tmem_ld32_issue(uint32_t taddr, uint32_t (&r)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
          "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
          "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr));
}
// The registers are tied to the wait as in/out operands: nothing that reads them can be scheduled above it.
__device__ __forceinline__ void tmem_ld_wait(uint32_t (&r)[32]) {
    asm volatile("tcgen05.wait::ld.sync.aligned;"
                 : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7]), "+r"(r[8]),
                   "+r"(r[9]), "+r"(r[10]), "+r"(r[11]), "+r"(r[12]), "+r"(r[13]), "+r"(r[14]), "+r"(r[15]), "+r"(r[16]),
                   "+r"(r[17]), "+r"(r[18]), "+r"(r[19]), "+r"(r[20]), "+r"(r[21]), "+r"(r[22]), "+r"(r[23]), "+r"(r[24]),
                   "+r"(r[25]), "+r"(r[26]), "+r"(r[27]), "+r"(r[28]), "+r"(r[29]), "+r"(r[30]), "+r"(r[31])
                 :
                 : "memory");
}
__device__ __forceinline__ uint32_t pack_bf16(float lo, float hi) {
    const __nv_bfloat162 p = __floats2bfloat162_rn(lo, hi);
    return *reinterpret_cast<const uint32_t *>(&p);
}

// Two tiles in flight per CTA.  Epilogue group g (warps 4g .. 4g + 3, one env row = one TMEM lane per thread) owns
// the TMEM columns 256 g .. 256 g + 255 and every other tile of the CTA.  The layer-1 activations never go to
// shared memory: the epilogue packs them to bf16 pairs and stores them back into TMEM (tcgen05.st, in place over
// the accumulator columns it has already read), and layer 2 takes its A operand from TMEM.  Layer 2 runs as two
// N = 128 halves into the upper 128 columns of the region, so while one group is in an epilogue the tensor pipe
// works for the other.  Hand-offs are mbarriers (no CTA-wide barrier in the loop); the MMA warp polls them.
constexpr int kOffA0 = (kBlobBytes + 127) / 128 * 128;      // two [128 rows][16] tiles
constexpr int kOffBar = kOffA0 + 2 * kTileM * kK1 * 2;      // 2 groups x {a0_ready, d1_ready, h1_ready, d2_ready, d2_free}
constexpr int kSmemBytes = kOffBar + 2 * 5 * 8;
static_assert(kSmemBytes <= 227 * 1024, "shared memory budget");
enum { B_A0 = 0, B_D1 = 1, B_H1 = 2, B_D2 = 3, B_FREE = 4 };

__device__ __forceinline__ void mbar_arrive(uint64_t *bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_test(uint64_t *bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "mbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t"
        "}" : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity) : "memory");
    return ok != 0;
}
// D[tmem] (+)= A[tmem, bf16 pairs per column] . B[smem]^T
__device__ __forceinline__ void umma_bf16_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, {%5, %5, %5, %5}, p;\n\t"
        "}" ::"r"(tmem_d), "r"(tmem_a), "l"(b_desc), "r"(idesc), "r"(accumulate), "r"(0u) : "memory");
}
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const uint32_t (&r)[16]) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
        "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};" ::"r"(taddr), "r"(r[0]), "r"(r[1]),
        "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]), "r"(r[10]), "r"(r[11]),
        "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15])
        : "memory");
}

// Prologue of every CTA: the weight blob into shared memory, the 2 x 5 mbarriers, 512 TMEM columns.  Returns the
// TMEM base address.
__device__ __forceinline__ uint32_t actor_prologue(const unsigned char *__restrict__ blob, unsigned char *smem,
                                                   uint32_t *tmem_base_slot) {
    const int tid = threadIdx.x, warp = tid >> 5;
    uint64_t *bars = reinterpret_cast<uint64_t *>(smem + kOffBar);
    for (int i = tid; i < kBlobBytes / 16; i += kThreads)
        reinterpret_cast<uint4 *>(smem)[i] = __ldg(reinterpret_cast<const uint4 *>(blob) + i);
    if (tid == 0) {
        for (int g = 0; g < 2; ++g) {
            mbar_init(bars + 5 * g + B_A0, 128);
            mbar_init(bars + 5 * g + B_D1, 1);
            mbar_init(bars + 5 * g + B_H1, 128);
            mbar_init(bars + 5 * g + B_D2, 1);
            mbar_init(bars + 5 * g + B_FREE, 128);
        }
        mbar_fence_init();
    }
    if (warp == kMmaWarp) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 512;" ::"r"(smem_u32(tmem_base_slot)) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    fence_proxy_async_smem();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    return *tmem_base_slot;
}

// One poll of group g's MMA state machine (lane 0 of the MMA warp): issues whatever the group's barriers allow.
// `state` 0: waiting for the observations (A0), 1: for h1 in TMEM, 2: for the first layer-2 half to be read.
// Returns true when the group's pass through the network is fully issued (the caller advances its parity).
__device__ __forceinline__ bool actor_mma_poll(uint64_t *b, int &state, uint32_t par, uint32_t region, uint32_t sbase, int g) {
    if (state == 0) {          // observations staged -> layer 1: D1[128][256] = A0 . W1^T
        if (!mbar_test(b + B_A0, par)) return false;
        tc_fence_after();
        umma_bf16(region, umma_desc(sbase + kOffA0 + g * (kTileM * kK1 * 2), kTileM * 16, 128),
                  umma_desc(sbase + kOffW1, kHidden * 16, 128), umma_idesc(kTileM, kHidden), 0u);
        umma_commit(b + B_D1);
        state = 1;
        return false;
    }
    // h1 is in TMEM (state 1) / the first half has been read (state 2)
    if (!mbar_test(b + (state == 1 ? B_H1 : B_FREE), par)) return false;
    tc_fence_after();
    const int half = state - 1;   // output columns 128 half .. + 127 of layer 2
#pragma unroll 1
    for (int k = 0; k < kHidden / 16; ++k)
        umma_bf16_ts(region + 128u, region + 8u * k,
                     umma_desc(sbase + kOffW2 + half * (128 * 16) + k * 2 * (kHidden * 16), kHidden * 16, 128),
                     umma_idesc(kTileM, 128), k > 0 ? 1u : 0u);
    umma_commit(b + B_D2);
    if (state == 1) { state = 2; return false; }
    state = 0;
    return true;
}

// Epilogue: this thread's row of observations -> bf16 A operand of layer 1, then signals a0_ready.  The previous
// pass's epilogue, i.e. every read of this group's TMEM region, is behind the caller.
__device__ __forceinline__ void actor_stage_a0(uint64_t *b, unsigned char *a0, int row, const float (&o)[kK1]) {
#pragma unroll
    for (int j = 0; j < 2; ++j) {
        uint4 out;
        out.x = pack_bf16(o[j * 8 + 0], o[j * 8 + 1]);
        out.y = pack_bf16(o[j * 8 + 2], o[j * 8 + 3]);
        out.z = pack_bf16(o[j * 8 + 4], o[j * 8 + 5]);
        out.w = pack_bf16(o[j * 8 + 6], o[j * 8 + 7]);
        *reinterpret_cast<uint4 *>(a0 + j * (kTileM * 16) + row * 16) = out;
    }
    fence_proxy_async_smem();
    tc_fence_before();
    mbar_arrive(b + B_A0);
}

// Layer-1 epilogue: accumulator -> + bias -> ReLU -> bf16 pairs, back into TMEM in place; then signals h1_ready.
__device__ __forceinline__ void actor_layer1_epilogue(uint64_t *b, uint32_t par, uint32_t region, const float *b1) {
    mbar_wait(b + B_D1, par);
    tc_fence_after();
    {
        uint32_t ra[32], rb[32];
        auto chunk = [&](const uint32_t (&r)[32], int c) {
            uint32_t packed[16];
#pragma unroll
            for (int q = 0; q < 8; ++q) {
                const float4 bb = *reinterpret_cast<const float4 *>(b1 + c * 32 + 4 * q);
                packed[2 * q] = pack_bf16(fmaxf(__uint_as_float(r[4 * q + 0]) + bb.x, 0.f),
                                          fmaxf(__uint_as_float(r[4 * q + 1]) + bb.y, 0.f));
                packed[2 * q + 1] = pack_bf16(fmaxf(__uint_as_float(r[4 * q + 2]) + bb.z, 0.f),
                                              fmaxf(__uint_as_float(r[4 * q + 3]) + bb.w, 0.f));
            }
            tmem_st16(region + 16u * c, packed);   // columns 16 c .. 16 c + 15 <= what has been read so far
        };
        tmem_ld32_issue(region, ra);
#pragma unroll
        for (int c = 0; c < 8; c += 2) {
            tmem_ld_wait(ra); tmem_ld32_issue(region + 32u * (c + 1), rb); chunk(ra, c);
            tmem_ld_wait(rb);
            if (c + 2 < 8) tmem_ld32_issue(region + 32u * (c + 2), ra);
            chunk(rb, c + 1);
        }
    }
    asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
    tc_fence_before();
    mbar_arrive(b + B_H1);
}

// Layer-2 epilogue (two halves of 128 columns) fused with the fp32 heads: acc[j] = relu(h2) . w3[j] (bias not added).
template <int NH>
__device__ __forceinline__ void actor_layer2_heads(uint64_t *b, uint32_t region, const float *b2, const float *w3,
                                                   float (&acc)[NH]) {
#pragma unroll
    for (int j = 0; j < NH; ++j) acc[j] = 0.f;
#pragma unroll 1
    for (int half = 0; half < 2; ++half) {
        mbar_wait(b + B_D2, (uint32_t)half);   // two completions per pass: parities 0, 1
        tc_fence_after();
        uint32_t ra[32], rb[32];
        auto chunk = [&](const uint32_t (&r)[32], int c) {   // c: 32-column chunk of the 256 layer-2 outputs
            float v[32];
#pragma unroll
            for (int q = 0; q < 8; ++q) {
                const float4 bb = *reinterpret_cast<const float4 *>(b2 + c * 32 + 4 * q);
                v[4 * q + 0] = fmaxf(__uint_as_float(r[4 * q + 0]) + bb.x, 0.f);
                v[4 * q + 1] = fmaxf(__uint_as_float(r[4 * q + 1]) + bb.y, 0.f);
                v[4 * q + 2] = fmaxf(__uint_as_float(r[4 * q + 2]) + bb.z, 0.f);
                v[4 * q + 3] = fmaxf(__uint_as_float(r[4 * q + 3]) + bb.w, 0.f);
            }
#pragma unroll
            for (int j = 0; j < NH; ++j) {
                const float4 *w = reinterpret_cast<const float4 *>(w3 + j * kHidden + c * 32);
#pragma unroll
                for (int q = 0; q < 8; ++q) {
                    const float4 ww = w[q];
                    acc[j] = fmaf(v[4 * q + 0], ww.x, acc[j]);
                    acc[j] = fmaf(v[4 * q + 1], ww.y, acc[j]);
                    acc[j] = fmaf(v[4 * q + 2], ww.z, acc[j]);
                    acc[j] = fmaf(v[4 * q + 3], ww.w, acc[j]);
                }
            }
        };
        const uint32_t d2 = region + 128u;
        tmem_ld32_issue(d2, ra);
        tmem_ld_wait(ra); tmem_ld32_issue(d2 + 32u, rb); chunk(ra, half * 4 + 0);
        tmem_ld_wait(rb); tmem_ld32_issue(d2 + 64u, ra); chunk(rb, half * 4 + 1);
        tmem_ld_wait(ra); tmem_ld32_issue(d2 + 96u, rb); chunk(ra, half * 4 + 2);
        tmem_ld_wait(rb); chunk(rb, half * 4 + 3);
        if (half == 0) {   // the columns may be overwritten by the second half now
            tc_fence_before();
            mbar_arrive(b + B_FREE);
        }
    }
}

// Standard-normal draw of (env row, step, action) for the tanh-squashed action: Box-Muller on
// Philox(seed; env, step, action).
__device__ __forceinline__ float actor_normal_draw(long long env, unsigned long long step, int a, unsigned long long seed) {
    const Philox4 r = philox4x32_10(
        (uint32_t)env, (uint32_t)((unsigned long long)env >> 32), (uint32_t)step,
        0xD0000000u | ((uint32_t)a << 16) | (uint32_t)((step >> 32) & 0xffffu), (uint32_t)seed,
        (uint32_t)(seed >> 32));
    const float u1 = ((float)(r.x >> 8) + 0.5f) * (1.0f / 16777216.0f);
    const float u2 = ((float)(r.y >> 8) + 0.5f) * (1.0f / 16777216.0f);
    return sqrtf(-2.0f * logf(u1)) * cospif(2.0f * u2);
}

// Launch set-up of a family of kernels built on this pass, on the current device: raises their dynamic shared-memory
// limit to kSmemBytes and returns the SM count in n_sm.  Done once per device and family (the statics belong to the
// instantiation) under a mutex, so that alternating devices or host threads neither thrash nor race.
template <auto... Kernels>
cudaError_t actor_kernels_setup(int &n_sm) {
    static std::mutex mu;
    static int n_sm_of[64] = {0};
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    if (dev < 0 || dev >= 64) return cudaErrorInvalidDevice;
    std::lock_guard<std::mutex> lock(mu);
    if (n_sm_of[dev] == 0) {
        for (const void *k : {(const void *)Kernels...}) {
            e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBytes);
            if (e != cudaSuccess) return e;
        }
        int v = 0;
        e = cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev);
        if (e != cudaSuccess) return e;
        n_sm_of[dev] = v;
    }
    n_sm = n_sm_of[dev];
    return cudaSuccess;
}

}  // namespace boatenv
