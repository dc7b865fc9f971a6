// policy_mlp.cu -- the actor's forward pass for acting (ActorNetwork.forward + sample_normal without
// gradients, networks/networks.py:38-70; choose_action, agent/continuous_agent.py:57-61) over N envs as ONE
// persistent kernel on the 5th-generation tensor cores (tcgen05, accumulators in TMEM).
//
//   obs[N][obs_dim] -> relu(fc1) -> relu(fc2) -> (mean, std heads) -> tanh-squashed draw -> action[N][A]
//
// The three dense layers are 256 wide.  Through cuBLAS every layer writes its [N][256] activations to HBM
// and the next one reads them back (1 GB per layer for a million envs); here a CTA keeps a 128-env tile
// on chip from the observations to the actions:
//   * all weights (bf16 layers 144 kB + fp32 heads 16 kB) live in shared memory for the life of the CTA, the
//     bf16 ones in the K-major no-swizzle core-matrix layout the UMMA descriptors address directly;
//   * the two hidden layers are tcgen05.mma (M = 128 envs, K steps of 16) into TMEM.  An epilogue thread owns
//     one env row (= one TMEM lane): after layer 1 it reads the accumulator back (tcgen05.ld), adds the bias,
//     applies ReLU, rounds to bf16 and stores the pairs back into TMEM (tcgen05.st) as the A operand of
//     layer 2; after layer 2 the fp32 activations go straight from registers into the dot products of the two
//     heads (fp32 weights), the draw and the squash;
//   * two tiles are in flight per CTA (two epilogue groups, two TMEM regions), so one tile's epilogue runs
//     under the other's MMAs; observations are fetched one tile ahead;
//   * HBM traffic is the input and the output: 4 * obs_dim + 4 * A bytes per env.
// Inputs are rounded to bf16 (fp32 accumulation): acting only, the learner never sees this kernel.
// The rollout kernel (rollout.cu) runs the same pass through the copies of these steps in actor_tc.cuh
// (actor_prologue .. actor_normal_draw), which must stay statement for statement equal to the code below: a change
// here is made there too (tests/test_gpu_rollout.py checks the two kernels' actions bit for bit).
#include <mutex>

#include "actor_tc.cuh"
#include "launch.h"

namespace {

using namespace boatenv;

template <int NA>
__global__ void __launch_bounds__(kThreads, 1)
policy_mlp_kernel(const unsigned char *__restrict__ blob, const float *__restrict__ obs, const float *__restrict__ eps,
                   const float *__restrict__ max_action, unsigned long long seed, unsigned long long step, long long n,
                   int obs_dim, float *__restrict__ action_out) {
    extern __shared__ __align__(128) unsigned char smem[];
    __shared__ uint32_t tmem_base_slot;
    constexpr int NH = 2 * NA;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    uint64_t *bars = reinterpret_cast<uint64_t *>(smem + kOffBar);

    for (int i = tid; i < kBlobBytes / 16; i += kThreads)
        reinterpret_cast<uint4 *>(smem)[i] = __ldg(reinterpret_cast<const uint4 *>(blob) + i);
    if (tid == 0) {
        for (int g = 0; g < 2; ++g) {
            asm volatile("mbarrier.init.shared::cta.b64 [%0], 128;" ::"r"(smem_addr(bars + 5 * g + B_A0)) : "memory");
            asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(smem_addr(bars + 5 * g + B_D1)) : "memory");
            asm volatile("mbarrier.init.shared::cta.b64 [%0], 128;" ::"r"(smem_addr(bars + 5 * g + B_H1)) : "memory");
            asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(smem_addr(bars + 5 * g + B_D2)) : "memory");
            asm volatile("mbarrier.init.shared::cta.b64 [%0], 128;" ::"r"(smem_addr(bars + 5 * g + B_FREE)) : "memory");
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == kMmaWarp) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 512;" ::"r"(smem_addr(&tmem_base_slot)) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    proxy_fence();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = tmem_base_slot;
    const uint32_t sbase = smem_addr(smem);
    const long long n_tiles = (n + kTileM - 1) / kTileM;
    const long long G = gridDim.x;
    // local tile j of this CTA is global tile blockIdx.x + j * G; group g takes the local tiles j = 2 i + g
    const long long my_tiles = n_tiles > (long long)blockIdx.x ? (n_tiles - blockIdx.x + G - 1) / G : 0;

    if (warp == kMmaWarp) {
        if (lane == 0) {
            // ===== MMA issuer: a small state machine per group, served in whatever order the barriers complete =====
            int state[2] = {0, 0};
            long long it[2] = {0, 0};
            const long long cnt[2] = {(my_tiles + 1) / 2, my_tiles / 2};
            while (it[0] < cnt[0] || it[1] < cnt[1]) {
#pragma unroll
                for (int g = 0; g < 2; ++g) {
                    if (it[g] >= cnt[g]) continue;
                    uint64_t *b = bars + 5 * g;
                    const uint32_t par = (uint32_t)(it[g] & 1);
                    const uint32_t region = tmem + 256u * g;
                    if (state[g] == 0) {          // observations staged -> layer 1: D1[128][256] = A0 . W1^T
                        if (!bar_test(b + B_A0, par)) continue;
                        tc_fence_after();
                        umma_bf16(region, umma_desc(sbase + kOffA0 + g * (kTileM * kK1 * 2), kTileM * 16, 128),
                                  umma_desc(sbase + kOffW1, kHidden * 16, 128), umma_idesc(kTileM, kHidden), 0u);
                        umma_commit(b + B_D1);
                        state[g] = 1;
                    } else {                      // h1 is in TMEM (state 1) / the first half has been read (state 2)
                        if (!bar_test(b + (state[g] == 1 ? B_H1 : B_FREE), par)) continue;
                        tc_fence_after();
                        const int half = state[g] - 1;   // output columns 128 half .. + 127 of layer 2
#pragma unroll 1
                        for (int k = 0; k < kHidden / 16; ++k)
                            umma_bf16_ts(region + 128u, region + 8u * k,
                                         umma_desc(sbase + kOffW2 + half * (128 * 16) + k * 2 * (kHidden * 16), kHidden * 16, 128),
                                         umma_idesc(kTileM, 128), k > 0 ? 1u : 0u);
                        umma_commit(b + B_D2);
                        if (state[g] == 1) state[g] = 2;
                        else { state[g] = 0; ++it[g]; }
                    }
                }
            }
        }
    } else {
        // ===== epilogue group g: one env row per thread =====
        const int g = warp >> 2, row = (warp & 3) * 32 + lane;
        uint64_t *b = bars + 5 * g;
        const uint32_t region = tmem + 256u * g + ((uint32_t)(warp & 3) * 32u << 16);
        const float *b1 = reinterpret_cast<const float *>(smem + kOffB1), *b2 = reinterpret_cast<const float *>(smem + kOffB2),
                    *b3 = reinterpret_cast<const float *>(smem + kOffB3), *w3 = reinterpret_cast<const float *>(smem + kOffW3);
        unsigned char *a0 = smem + kOffA0 + g * (kTileM * kK1 * 2);
        const long long cnt = g == 0 ? (my_tiles + 1) / 2 : my_tiles / 2;
        float o[kK1];
        auto fetch_obs = [&](long long i) {
            const long long e = ((long long)blockIdx.x + (2 * i + g) * G) * kTileM + row;
#pragma unroll
            for (int q = 0; q < kK1; ++q) o[q] = (q < obs_dim && i < cnt && e < n) ? __ldg(obs + e * obs_dim + q) : 0.f;
        };
        fetch_obs(0);
        for (long long i = 0; i < cnt; ++i) {
            const long long env = ((long long)blockIdx.x + (2 * i + g) * G) * kTileM + row;
            const uint32_t par = (uint32_t)(i & 1);
            // ---- observations -> bf16 A0 (the previous tile's epilogue, i.e. every read of this region, is behind us) ----
#pragma unroll
            for (int j = 0; j < 2; ++j) {
                uint4 out;
                out.x = pack_bf16(o[j * 8 + 0], o[j * 8 + 1]);
                out.y = pack_bf16(o[j * 8 + 2], o[j * 8 + 3]);
                out.z = pack_bf16(o[j * 8 + 4], o[j * 8 + 5]);
                out.w = pack_bf16(o[j * 8 + 6], o[j * 8 + 7]);
                *reinterpret_cast<uint4 *>(a0 + j * (kTileM * 16) + row * 16) = out;
            }
            proxy_fence();
            tc_fence_before();
            bar_arrive(b + B_A0);
            fetch_obs(i + 1);
            // ---- layer-1 epilogue: accumulator -> + bias -> ReLU -> bf16 pairs, back into TMEM in place ----
            bar_wait(b + B_D1, par);
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
            bar_arrive(b + B_H1);
            // ---- layer-2 epilogue (two halves of 128 columns) fused with the fp32 heads ----
            float acc[NH];
#pragma unroll
            for (int j = 0; j < NH; ++j) acc[j] = 0.f;
#pragma unroll 1
            for (int half = 0; half < 2; ++half) {
                bar_wait(b + B_D2, (uint32_t)half);   // two completions per tile: parities 0, 1
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
                    bar_arrive(b + B_FREE);
                }
            }
            if (env < n) {
#pragma unroll
                for (int a = 0; a < NA; ++a) {   // sample_normal, networks.py:47-65
                    const float mean = acc[a] + b3[a];
                    const float log_std = -5.0f + 3.5f * (tanhf(acc[NA + a] + b3[NA + a]) + 1.0f);
                    float e;
                    if (eps) {
                        e = __ldg(eps + env * NA + a);
                    } else {   // Box-Muller on Philox(seed; env, step, action)
                        const boatenv::Philox4 r = boatenv::philox4x32_10(
                            (uint32_t)env, (uint32_t)((unsigned long long)env >> 32), (uint32_t)step,
                            0xD0000000u | ((uint32_t)a << 16) | (uint32_t)((step >> 32) & 0xffffu), (uint32_t)seed,
                            (uint32_t)(seed >> 32));
                        const float u1 = ((float)(r.x >> 8) + 0.5f) * (1.0f / 16777216.0f);
                        const float u2 = ((float)(r.y >> 8) + 0.5f) * (1.0f / 16777216.0f);
                        e = sqrtf(-2.0f * logf(u1)) * cospif(2.0f * u2);
                    }
                    action_out[env * NA + a] = tanhf(mean + e * expf(log_std)) * __ldg(max_action + a);
                }
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == kMmaWarp) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 512;" ::"r"(tmem) : "memory");
}

}  // namespace

extern "C" int boatagent_policy_act(const void *weight_blob, const float *obs, const float *eps, const float *max_action,
                                    uint64_t seed, uint64_t step, int64_t n, int32_t obs_dim, int32_t n_actions,
                                    float *action_out, void *stream) {
    if (!weight_blob || !obs || !max_action || !action_out || n <= 0) return BOATENV_EINVAL;
    if (obs_dim < 1 || obs_dim > kK1) return BOATENV_EUNSUPPORTED;
    if ((reinterpret_cast<uintptr_t>(weight_blob) & 15u) != 0) return BOATENV_EALIGN;
    using kern_t = void (*)(const unsigned char *, const float *, const float *, const float *, unsigned long long,
                            unsigned long long, long long, int, float *);
    kern_t kern = nullptr;
    switch (n_actions) {   // the head count is a template parameter (its dot products live in registers)
    case 1: kern = policy_mlp_kernel<1>; break;
    case 2: kern = policy_mlp_kernel<2>; break;
    case 4: kern = policy_mlp_kernel<4>; break;
    case 8: kern = policy_mlp_kernel<8>; break;
    default: return BOATENV_EUNSUPPORTED;
    }
    // per-device configuration (max dynamic shared memory of the four instantiations, SM count): done once per
    // device under a mutex, so that alternating devices or host threads neither thrash nor race
    static std::mutex mu;
    static int n_sm_of[64] = {0};
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return (int)e;
    if (dev < 0 || dev >= 64) return (int)cudaErrorInvalidDevice;
    int n_sm = 0;
    {
        std::lock_guard<std::mutex> lock(mu);
        if (n_sm_of[dev] == 0) {
            for (kern_t k : {(kern_t)policy_mlp_kernel<1>, (kern_t)policy_mlp_kernel<2>, (kern_t)policy_mlp_kernel<4>,
                             (kern_t)policy_mlp_kernel<8>}) {
                e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBytes);
                if (e != cudaSuccess) return (int)e;
            }
            int v = 0;
            e = cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev);
            if (e != cudaSuccess) return (int)e;
            n_sm_of[dev] = v;
        }
        n_sm = n_sm_of[dev];
    }
    const long long tiles = (n + kTileM - 1) / kTileM;
    const unsigned grid = (unsigned)(tiles < n_sm ? tiles : n_sm);
    kern<<<grid, kThreads, kSmemBytes, (cudaStream_t)stream>>>((const unsigned char *)weight_blob, obs, eps, max_action, seed,
                                                              step, n, obs_dim, action_out);
    boatenv::count_launch();
    return (int)cudaGetLastError();
}
