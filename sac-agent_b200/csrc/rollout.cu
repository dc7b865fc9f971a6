// rollout.cu -- closed-loop evaluation of the tcgen05 policy on a BoatEnv handle (main.py -r, render_model:
// main.py:137-172, without the rendering) as ONE persistent kernel: the actor's forward pass (actor_tc.cuh, the
// warp roles of policy_mlp.cu) and the env step (boat_step.cuh, the K = 1 sub-step) fused, so an env never leaves
// the SM while its episode runs.
//
//   * an epilogue group owns a 128-env tile (four 32-env state blocks); warp w % 4 of the group loads block
//     4 tile + w % 4 into registers once and keeps it there for up to max_steps steps;
//   * per step the epilogue thread of an env runs the heads, draws the action (exactly boatagent_policy_act's
//     for row i and step step0 + t), takes one substep<WK, true> and stages the next observation straight into
//     its row of the group's bf16 A0 tile; the MMA warp loops within the tile;
//   * an env whose episode ends is frozen (no auto-reset, no further steps): counters updated once as the step
//     kernel does, terminal state kept, terminal observation out;
//   * a tile ends when all its rows are frozen or max_steps is reached; its state goes back to its blocks (dyn
//     slots, index word, the wind coefficients if a piece change replaced them) and the group takes its next tile;
//   * a piece change (wind[index] of the next step in the next spline piece) is served in the env's own lane by
//     wind_setup_lane_any: the envs of a freshly reset tile cross piece boundaries at the same step, so it runs
//     converged.
// fp32 handles and one action only.  Design notes and measurements: DESIGN.md sections 4 and 8.
#include "actor_tc.cuh"
#include "boat_step.cuh"
#include "launch.h"

using namespace boatenv;

namespace {

struct RolloutArgs {
    const unsigned char *blob;
    const float *max_action;
    unsigned long long seed, step0;
    int max_steps, deterministic;
    const float *obs_in;
    float *obs_out, *return_out;
    int32_t *steps_out;
    uint8_t *term_out;
};

// OR of `v` over the 128 threads of epilogue group g (named barrier 1 + g; the MMA warp never joins it).
__device__ __forceinline__ bool group_any(bool v, int g) {
    uint32_t r;
    asm volatile(
        "{\n\t"
        ".reg .pred p, q;\n\t"
        "setp.ne.u32 p, %1, 0;\n\t"
        "bar.red.or.pred q, %2, 128, p;\n\t"
        "selp.u32 %0, 1, 0, q;\n\t"
        "}" : "=r"(r) : "r"((uint32_t)v), "r"(1 + g) : "memory");
    return r != 0;
}

template <int WK>
__global__ void __launch_bounds__(kThreads, 1)
boat_rollout_kernel(const __grid_constant__ DevCfg c, const __grid_constant__ RolloutArgs a) {
    extern __shared__ __align__(128) unsigned char smem[];
    __shared__ uint32_t tmem_base_slot;
    __shared__ volatile int group_done[2];   // set by an epilogue group after its last pass: the MMA warp stops serving it
    constexpr bool kCurves = (WK == WIND_VEL_CURVE || WK == WIND_ANGLE_RECT || WK == WIND_BOTH);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    uint64_t *bars = reinterpret_cast<uint64_t *>(smem + kOffBar);
    if (tid < 2) group_done[tid] = 0;
    const uint32_t tmem = actor_prologue(a.blob, smem, &tmem_base_slot);   // its __syncthreads orders group_done
    const uint32_t sbase = smem_u32(smem);
    const long long n = c.n_envs;
    const long long n_tiles = (n + kTileM - 1) / kTileM;
    const long long G = gridDim.x;
    const long long my_tiles = n_tiles > (long long)blockIdx.x ? (n_tiles - blockIdx.x + G - 1) / G : 0;

    if (warp == kMmaWarp) {
        if (lane == 0) {
            // ===== MMA issuer: as in policy_mlp.cu, but a group makes as many passes as its tiles take steps =====
            int state[2] = {0, 0};
            long long it[2] = {0, 0};
            bool live[2] = {true, true};
            while (live[0] || live[1]) {
#pragma unroll
                for (int g = 0; g < 2; ++g) {
                    if (!live[g]) continue;
                    // a group raises its flag only after waiting for its last pass's layer 2, i.e. once every pass
                    // it asked for has been issued: state 0 and no A0 pending
                    if (state[g] == 0 && group_done[g] && !mbar_test(bars + 5 * g + B_A0, (uint32_t)(it[g] & 1))) {
                        live[g] = false;
                        continue;
                    }
                    if (actor_mma_poll(bars + 5 * g, state[g], (uint32_t)(it[g] & 1), tmem + 256u * g, sbase, g)) ++it[g];
                }
            }
        }
    } else {
        // ===== epilogue group g: one env per thread, state in registers for a whole tile =====
        const int g = warp >> 2, wq = warp & 3, row = wq * 32 + lane;
        uint64_t *b = bars + 5 * g;
        const uint32_t region = tmem + 256u * g + ((uint32_t)wq * 32u << 16);
        const float *b1 = reinterpret_cast<const float *>(smem + kOffB1), *b2 = reinterpret_cast<const float *>(smem + kOffB2),
                    *b3 = reinterpret_cast<const float *>(smem + kOffB3), *w3 = reinterpret_cast<const float *>(smem + kOffW3);
        unsigned char *a0 = smem + kOffA0 + g * (kTileM * kK1 * 2);
        const long long cnt = g == 0 ? (my_tiles + 1) / 2 : my_tiles / 2;
        const float max_a = __ldg(a.max_action);
        const float inv_Lm1 = c.f.inv_Lm1;
        long long pass = 0;   // passes through the network so far: the barriers' parity
        for (long long i = 0; i < cnt; ++i) {
            const long long tile = (long long)blockIdx.x + (2 * i + g) * G;
            const long long blk = tile * 4 + wq;
            const long long env = blk * 32 + lane;
            const bool active = env < n;
            // ---- the env's state and last observation -> registers ----
            float d[D_COUNT];
            float wa[4] = {0.f, 0.f, 0.f, 0.f}, wb[4] = {0.f, 0.f, 0.f, 0.f};
            float o[kK1];
            Fx<float> fx;
            int index = 0;
            uint32_t episode = 0u;
            char *gb = c.state + (size_t)blk * (size_t)c.block_bytes;
#pragma unroll
            for (int q = 0; q < D_COUNT; ++q) d[q] = 0.f;
            fx.rud = 0.0; fx.sx = 0; fx.sy = 0;
            if (active) {
                load_vecs<float, D_COUNT>(gb, lane, d);
                if (kCurves) load_vecs<float, 4>(gb + c.off_wa, lane, wa);
                if (WK == WIND_BOTH) load_vecs<float, 4>(gb + c.off_wb, lane, wb);
                fx.load(c, d, reinterpret_cast<const uint32_t *>(gb + c.off_idx)[lane], index);
                if (kCurves) episode = reinterpret_cast<const uint32_t *>(gb + c.off_epi)[lane];
            }
#pragma unroll
            for (int q = 0; q < kK1; ++q) o[q] = (q < kObsDim && active) ? __ldg(a.obs_in + env * kObsDim + q) : 0.f;
            bool alive = active, wind_dirty = false;
            int code = BOATENV_TERM_NONE, nsteps = 0;
            for (int t = 0;;) {
                actor_stage_a0(b, a0, row, o);
                actor_layer1_epilogue(b, (uint32_t)(pass & 1), region, b1);
                float acc[2];
                actor_layer2_heads<2>(b, region, b2, w3, acc);
                ++pass;
                if (alive) {
                    // ---- the action boatagent_policy_act gives row env at step step0 + t (sample_normal, networks.py:47-65) ----
                    const unsigned long long step = a.step0 + (unsigned long long)t;
                    const float mean = acc[0] + b3[0];
                    const float log_std = -5.0f + 3.5f * (tanhf(acc[1] + b3[1]) + 1.0f);
                    float e;
                    if (a.deterministic) {
                        e = 0.f;
                    } else {
                        e = actor_normal_draw(env, step, 0, a.seed);
                    }
                    const float action = tanhf(mean + e * expf(log_std)) * max_a;
                    // ---- one env sub-step, as the K = 1 step kernel takes it ----
                    float w, th;
                    int j, r;
                    wind_sample<float, WK>(c, index, wa, wb, inv_Lm1, w, th, j, r);
                    float rew, accel[3];
                    substep<WK, true>(c, d, fx, index, action, w, th, accel, rew, code);
                    ++nsteps;
                    index += 1;
                    stage_obs(c, o, d, fx, accel, index);
                    if (code != BOATENV_TERM_NONE) {
                        alive = false;   // statistics as the step kernel counts them
                        count_episode_end(c, blk, code, d[D_RET]);
                    } else if (kCurves && next_sample_in_next_piece(c, j, r)) {
                        double cf[8];
                        wind_setup_lane_any(c, env, episode, index, cf);
#pragma unroll
                        for (int m = 0; m < 4; ++m) {
                            wa[m] = (float)cf[m];
                            wb[m] = (float)cf[4 + m];
                        }
                        wind_dirty = true;
                    }
                }
                ++t;
                const bool any_alive = group_any(alive, g);
                if (!any_alive || t >= a.max_steps) break;
            }
            // ---- write-back: state (episode number untouched), outputs ----
            if (active) {
                float dd[D_COUNT];
#pragma unroll
                for (int q = 0; q < D_COUNT; ++q) dd[q] = d[q];
                const uint32_t index_word = fx.pack(dd, index);
                store_vecs<float, D_COUNT>(gb, lane, dd);
                reinterpret_cast<uint32_t *>(gb + c.off_idx)[lane] = index_word;
                if (kCurves && wind_dirty) {
                    store_vecs<float, 4>(gb + c.off_wa, lane, wa);
                    if (WK == WIND_BOTH) store_vecs<float, 4>(gb + c.off_wb, lane, wb);
                }
#pragma unroll
                for (int q = 0; q < kObsDim; ++q) a.obs_out[env * kObsDim + q] = o[q];
                a.return_out[env] = d[D_RET];
                a.steps_out[env] = nsteps;
                a.term_out[env] = (uint8_t)code;
            }
        }
        if (row == 0) group_done[g] = 1;
    }
    tc_fence_before();
    __syncthreads();
    if (warp == kMmaWarp) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 512;" ::"r"(tmem) : "memory");
}

using kern_t = void (*)(const DevCfg, const RolloutArgs);

kern_t kernel_for(int wind_kind) {
    switch (wind_kind) {
    case WIND_NONE: return boat_rollout_kernel<WIND_NONE>;
    case WIND_CONST: return boat_rollout_kernel<WIND_CONST>;
    case WIND_VEL_CURVE: return boat_rollout_kernel<WIND_VEL_CURVE>;
    case WIND_ANGLE_RECT: return boat_rollout_kernel<WIND_ANGLE_RECT>;
    case WIND_BOTH: return boat_rollout_kernel<WIND_BOTH>;
    default: return nullptr;
    }
}

}  // namespace

extern "C" int boatagent_rollout(boatenv_t h, const void *weight_blob, const float *max_action, uint64_t seed,
                                 uint64_t step0, int32_t max_steps, uint32_t flags, const float *obs_in, float *obs_out,
                                 float *return_out, int32_t *steps_out, uint8_t *term_out, void *stream) {
    if (!h || !weight_blob || !max_action || !obs_in || !obs_out || !return_out || !steps_out || !term_out ||
        max_steps < 1 || (flags & ~BOATAGENT_ROLLOUT_DETERMINISTIC) != 0)
        return BOATENV_EINVAL;
    if (handle_precision(h) != 32) return BOATENV_EUNSUPPORTED;
    if (!handle_was_reset(h)) return BOATENV_ESTATE;
    if ((reinterpret_cast<uintptr_t>(weight_blob) & 15u) != 0) return BOATENV_EALIGN;
    boatenv::DeviceGuard _guard(handle_device(h));
    if (!_guard.ok()) return (int)_guard.error();
    const DevCfg &c = *handle_cfg(h);
    const kern_t kern = kernel_for(c.wind_kind);
    if (!kern) return BOATENV_EINVAL;
    int n_sm = 0;
    const cudaError_t e = actor_kernels_setup<boat_rollout_kernel<WIND_NONE>, boat_rollout_kernel<WIND_CONST>,
                                              boat_rollout_kernel<WIND_VEL_CURVE>, boat_rollout_kernel<WIND_ANGLE_RECT>,
                                              boat_rollout_kernel<WIND_BOTH>>(n_sm);
    if (e != cudaSuccess) return (int)e;
    RolloutArgs a;
    a.blob = static_cast<const unsigned char *>(weight_blob);
    a.max_action = max_action;
    a.seed = seed;
    a.step0 = step0;
    a.max_steps = max_steps;
    a.deterministic = (flags & BOATAGENT_ROLLOUT_DETERMINISTIC) ? 1 : 0;
    a.obs_in = obs_in;
    a.obs_out = obs_out;
    a.return_out = return_out;
    a.steps_out = steps_out;
    a.term_out = term_out;
    // one CTA per SM at most: with fewer tiles than SMs every tile gets a CTA (and an SM) of its own rather than
    // sharing a CTA with a second tile -- a tile's steps are a dependent chain, a second group only helps once the
    // SMs run out (measured against pairing in profiles/rollout_eval.json, DESIGN.md section 8)
    const long long tiles = (c.n_envs + kTileM - 1) / kTileM;
#ifdef BOAT_ROLLOUT_PAIR_TILES   // measurement only (profiles/rollout_eval.py): two tiles per CTA also below n_sm tiles
    const long long ctas = (tiles + 1) / 2;
#else
    const long long ctas = tiles;
#endif
    const unsigned grid = (unsigned)(ctas < n_sm ? ctas : n_sm);
    kern<<<grid, kThreads, kSmemBytes, (cudaStream_t)stream>>>(c, a);
    count_launch();
    return (int)cudaGetLastError();
}
