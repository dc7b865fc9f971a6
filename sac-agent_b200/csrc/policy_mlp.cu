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
// The pass is the building blocks of actor_tc.cuh (actor_prologue .. actor_normal_draw), which the rollout kernel
// (rollout.cu) runs too: the two kernels' actions agree bit for bit (tests/test_gpu_rollout.py).
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
    const uint32_t tmem = actor_prologue(blob, smem, &tmem_base_slot);
    const uint32_t sbase = smem_u32(smem);
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
                for (int g = 0; g < 2; ++g)
                    if (it[g] < cnt[g] && actor_mma_poll(bars + 5 * g, state[g], (uint32_t)(it[g] & 1), tmem + 256u * g, sbase, g))
                        ++it[g];
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
            actor_stage_a0(b, a0, row, o);
            fetch_obs(i + 1);   // the next tile's observations load under this tile's MMAs
            actor_layer1_epilogue(b, (uint32_t)(i & 1), region, b1);
            float acc[NH];
            actor_layer2_heads<NH>(b, region, b2, w3, acc);
            if (env < n) {
#pragma unroll
                for (int a = 0; a < NA; ++a) {   // sample_normal, networks.py:47-65
                    const float mean = acc[a] + b3[a];
                    const float log_std = -5.0f + 3.5f * (tanhf(acc[NA + a] + b3[NA + a]) + 1.0f);
                    const float e = eps ? __ldg(eps + env * NA + a) : actor_normal_draw(env, step, a, seed);
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
    int n_sm = 0;
    const cudaError_t e = actor_kernels_setup<policy_mlp_kernel<1>, policy_mlp_kernel<2>, policy_mlp_kernel<4>,
                                              policy_mlp_kernel<8>>(n_sm);
    if (e != cudaSuccess) return (int)e;
    const long long tiles = (n + kTileM - 1) / kTileM;
    const unsigned grid = (unsigned)(tiles < n_sm ? tiles : n_sm);
    kern<<<grid, kThreads, kSmemBytes, (cudaStream_t)stream>>>((const unsigned char *)weight_blob, obs, eps, max_action, seed,
                                                              step, n, obs_dim, action_out);
    boatenv::count_launch();
    return (int)cudaGetLastError();
}
