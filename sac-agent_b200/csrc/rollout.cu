// rollout.cu -- the tcgen05 policy and the env step fused into ONE persistent kernel per call: the actor's forward
// pass (actor_tc.cuh, the warp roles of policy_mlp.cu) and the K = 1 sub-step (boat_step.cuh), so an env never leaves
// the SM between steps.  Two kernels share the building blocks below:
//   * boat_rollout_kernel: closed-loop evaluation (main.py -r, render_model: main.py:137-172, without the
//     rendering).  An env whose episode ends is frozen (no auto-reset, no further steps): counters updated once as
//     the step kernel does, terminal state kept, terminal observation out.  A tile ends when all its rows are frozen
//     or max_steps is reached.
//   * boat_collect_kernel: experience collection (the main.py:78-90 loop body: act, step, remember) over T steps.
//     Every step writes its transition into the replay ring, and an env whose episode ends is reset in its own lane
//     as BOATENV_AUTO_RESET does in the step kernel; every tile runs exactly T steps.  Its <WK, true>
//     instantiations (boatagent_collect_record) also write each step's recorder row of selected envs into a
//     boatenv_record_ring, as boatenv_record_rows would after every step.
// Common to both:
//   * an epilogue group owns a 128-env tile (four 32-env state blocks); warp w % 4 of the group loads block
//     4 tile + w % 4 into registers once and keeps it there for the whole call;
//   * per step the epilogue thread of an env runs the heads, draws the action (exactly boatagent_policy_act's
//     for row i and step step0 + t), takes one substep<WK, true> and stages the next observation straight into
//     its row of the group's bf16 A0 tile; the MMA warp loops within the tile;
//   * at the end of a tile its state goes back to its blocks (dyn slots, index word, the wind coefficients if they
//     were replaced) and the group takes its next tile;
//   * a piece change (wind[index] of the next step in the next spline piece) needs new wind coefficients.  The
//     rollout computes them in the env's own lane (wind_setup_lane_any): the envs of a freshly reset tile cross
//     piece boundaries at the same step, so it runs converged.  Collection resets envs at scattered steps, so its
//     requests (piece changes and new episodes) are sparse, and the whole warp serves one env at a time
//     (wind_setup_warp, as the step kernel does).
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

// MMA issuer (lane 0 of the MMA warp): as in policy_mlp.cu, but a group makes as many passes as its tiles take steps.
// Serves both groups until each has raised its flag in group_done.
__device__ __forceinline__ void mma_serve_groups(uint64_t *bars, uint32_t tmem, uint32_t sbase, volatile int *group_done) {
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

// One env as its epilogue thread holds it in registers for a whole tile.
struct TileEnv {
    float d[D_COUNT];
    float wa[4], wb[4];
    float o[kK1];      // the last observation; columns kObsDim.. stay 0 (the padded K of layer 1)
    Fx<float> fx;
    int index;
    uint32_t episode;  // loaded when the kernel needs it (kEpisode)
};

// The env's state (lane `lane` of state block `gb`) and its last observation -> registers; padding lanes of a ragged
// last tile (active = false) get zeros.
template <int WK, bool kEpisode>
__device__ __forceinline__ void tile_env_load(const DevCfg &c, const char *gb, int lane, long long env, bool active,
                                              const float *obs_in, TileEnv &s) {
    constexpr bool kCurves = (WK == WIND_VEL_CURVE || WK == WIND_ANGLE_RECT || WK == WIND_BOTH);
#pragma unroll
    for (int q = 0; q < D_COUNT; ++q) s.d[q] = 0.f;
#pragma unroll
    for (int m = 0; m < 4; ++m) { s.wa[m] = 0.f; s.wb[m] = 0.f; }
    s.fx.rud = 0.0; s.fx.sx = 0; s.fx.sy = 0;
    s.index = 0;
    s.episode = 0u;
    if (active) {
        load_vecs<float, D_COUNT>(gb, lane, s.d);
        if (kCurves) load_vecs<float, 4>(gb + c.off_wa, lane, s.wa);
        if (WK == WIND_BOTH) load_vecs<float, 4>(gb + c.off_wb, lane, s.wb);
        s.fx.load(c, s.d, reinterpret_cast<const uint32_t *>(gb + c.off_idx)[lane], s.index);
        if (kEpisode) s.episode = reinterpret_cast<const uint32_t *>(gb + c.off_epi)[lane];
    }
#pragma unroll
    for (int q = 0; q < kK1; ++q) s.o[q] = (q < kObsDim && active) ? __ldg(obs_in + env * kObsDim + q) : 0.f;
}

// One step of an env: the action boatagent_policy_act gives row `env` at step `step` from the heads' accumulators
// (sample_normal, networks.py:47-65; deterministic: e = 0), then one env sub-step as the K = 1 step kernel takes it.
// o[] becomes the next observation.  Returns the action; j, r: the spline piece of the wind sample
// (next_sample_in_next_piece).
template <int WK>
__device__ __forceinline__ float act_and_substep(const DevCfg &c, TileEnv &s, const float (&acc)[2], const float *b3,
                                                 float max_a, float inv_Lm1, long long env, unsigned long long step,
                                                 unsigned long long seed, bool deterministic, float &rew, int &code,
                                                 int &j, int &r) {
    const float mean = acc[0] + b3[0];
    const float log_std = -5.0f + 3.5f * (tanhf(acc[1] + b3[1]) + 1.0f);
    float e;
    if (deterministic) {
        e = 0.f;
    } else {
        e = actor_normal_draw(env, step, 0, seed);
    }
    const float action = tanhf(mean + e * expf(log_std)) * max_a;
    float w, th;
    wind_sample<float, WK>(c, s.index, s.wa, s.wb, inv_Lm1, w, th, j, r);
    float accel[3];
    substep<WK, true>(c, s.d, s.fx, s.index, action, w, th, accel, rew, code);
    s.index += 1;
    stage_obs(c, s.o, s.d, s.fx, accel, s.index);
    return action;
}

// The folded wind coefficients of the piece that holds sample `index_next` of the env's episode s.episode.
__device__ __forceinline__ void tile_env_wind_setup(const DevCfg &c, long long env, int index_next, TileEnv &s) {
    double cf[8];
    wind_setup_lane_any(c, env, s.episode, index_next, cf);
#pragma unroll
    for (int m = 0; m < 4; ++m) {
        s.wa[m] = (float)cf[m];
        s.wb[m] = (float)cf[4 + m];
    }
}

// Registers -> the env's state block: dyn slots and index word always, the wind coefficients if they were replaced,
// the episode number if it changed.
template <int WK>
__device__ __forceinline__ void tile_env_store(const DevCfg &c, char *gb, int lane, const TileEnv &s, bool wind_dirty,
                                               bool episode_dirty) {
    constexpr bool kCurves = (WK == WIND_VEL_CURVE || WK == WIND_ANGLE_RECT || WK == WIND_BOTH);
    float dd[D_COUNT];
#pragma unroll
    for (int q = 0; q < D_COUNT; ++q) dd[q] = s.d[q];
    const uint32_t index_word = s.fx.pack(dd, s.index);
    store_vecs<float, D_COUNT>(gb, lane, dd);
    reinterpret_cast<uint32_t *>(gb + c.off_idx)[lane] = index_word;
    if (kCurves && wind_dirty) {
        store_vecs<float, 4>(gb + c.off_wa, lane, s.wa);
        if (WK == WIND_BOTH) store_vecs<float, 4>(gb + c.off_wb, lane, s.wb);
    }
    if (episode_dirty) reinterpret_cast<uint32_t *>(gb + c.off_epi)[lane] = s.episode;
}

// Barrier of the 128 threads of epilogue group g (named barrier 1 + g; the MMA warp never joins it).
__device__ __forceinline__ void group_sync(int g) { asm volatile("bar.sync %0, 128;" ::"r"(1 + g) : "memory"); }

// The recording ring's column j (ids[j] == env) of each env of the tile whose first env is `first`, -1 for an env
// that is not recorded.  The group's 128 threads scan the ids together, ceil(n_ids / 128) loads each, into the
// group's table; ids outside [0, n) match no env.  The first barrier keeps every thread's clearing of its own entry
// ahead of the others' writes, the second keeps their writes ahead of its read.
__device__ __forceinline__ int tile_record_column(const CollectArgs &a, int g, int row, long long first, long long n,
                                                  int *table) {
    table[row] = -1;
    group_sync(g);
    for (int j = row; j < a.rec_n_ids; j += kTileM) {
        const long long id = __ldg(a.rec_ids + j);
        if (id >= first && id < first + kTileM && id < n) table[id - first] = j;
    }
    group_sync(g);
    return table[row];
}

// The recorder row of an env after its step (and its reset, if the episode ended), entry o of the ring: what
// boatenv_record_rows writes after the per-step step_store.  The state is decoded from the bits Fx<float>::pack
// would store, as get_field decodes it once the tile is written back; action, reward and termination code are the
// step's, the episode number is the one after the reset.
__device__ __forceinline__ void tile_env_record(const DevCfg &c, const boatenv_record_ring &ring, long long o,
                                                const TileEnv &s, float action, float rew, int code) {
    float dd[D_COUNT];
#pragma unroll
    for (int q = 0; q < D_COUNT; ++q) dd[q] = s.d[q];
    const uint32_t ixw = s.fx.pack(dd, s.index);
    static_cast<float *>(ring.s_x)[o] = (float)decode_field(c, D_SX, dd[D_SX], ixw);
    static_cast<float *>(ring.s_y)[o] = (float)decode_field(c, D_SY, dd[D_SY], ixw);
    static_cast<float *>(ring.v_x)[o] = (float)decode_field(c, D_VX, dd[D_VX], ixw);
    static_cast<float *>(ring.v_y)[o] = (float)decode_field(c, D_VY, dd[D_VY], ixw);
    static_cast<float *>(ring.s_r)[o] = (float)decode_field(c, D_SR, dd[D_SR], ixw);
    static_cast<float *>(ring.rudder_angle)[o] = (float)decode_field(c, D_RUDDER, dd[D_RUDDER], ixw);
    static_cast<float *>(ring.action)[o] = action;
    static_cast<float *>(ring.reward)[o] = rew;
    ring.term[o] = (uint8_t)code;
    ring.episode[o] = s.episode;
}

// New wind coefficients for the lanes of this warp that ask for them (`need`: an episode was reset, or the next
// sample lies in the next spline piece), for sample s.index of episode s.episode.  Collection resets envs at scattered
// steps, so requests are sparse: the whole warp serves one env at a time (wind_setup_warp, the step kernel's slow
// path), which has a far shorter latency than one lane working alone, and the other 31 envs of the warp wait for it.
// Both mappings give bit-identical coefficients (wind_setup.cuh).
__device__ __forceinline__ void warp_wind_setups(const DevCfg &c, bool need, long long env, TileEnv &s, double *scratch) {
    const unsigned FULL = 0xffffffffu;
    const int lane = threadIdx.x & 31;
    unsigned todo = __ballot_sync(FULL, need);
    while (todo) {
        const int src = __ffs(todo) - 1;
        todo &= todo - 1;
        const uint32_t episode = __shfl_sync(FULL, s.episode, src);
        const int index_next = __shfl_sync(FULL, s.index, src);
        wind_setup_warp(c, env - lane + src, episode, index_next, scratch);
        if (lane == src) {
#pragma unroll
            for (int m = 0; m < 4; ++m) {
                s.wa[m] = (float)scratch[m];
                s.wb[m] = (float)scratch[4 + m];
            }
        }
        __syncwarp();   // scratch is reused by the next env of this warp
    }
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
        if (lane == 0) mma_serve_groups(bars, tmem, sbase, group_done);
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
            char *gb = c.state + (size_t)blk * (size_t)c.block_bytes;
            TileEnv s;
            tile_env_load<WK, kCurves>(c, gb, lane, env, active, a.obs_in, s);
            bool alive = active, wind_dirty = false;
            int code = BOATENV_TERM_NONE, nsteps = 0;
            for (int t = 0;;) {
                actor_stage_a0(b, a0, row, s.o);
                actor_layer1_epilogue(b, (uint32_t)(pass & 1), region, b1);
                float acc[2];
                actor_layer2_heads<2>(b, region, b2, w3, acc);
                ++pass;
                if (alive) {
                    float rew;
                    int j, r;
                    act_and_substep<WK>(c, s, acc, b3, max_a, inv_Lm1, env, a.step0 + (unsigned long long)t, a.seed,
                                        a.deterministic != 0, rew, code, j, r);
                    ++nsteps;
                    if (code != BOATENV_TERM_NONE) {
                        alive = false;   // statistics as the step kernel counts them
                        count_episode_end(c, blk, code, s.d[D_RET]);
                    } else if (kCurves && next_sample_in_next_piece(c, j, r)) {
                        tile_env_wind_setup(c, env, s.index, s);
                        wind_dirty = true;
                    }
                }
                ++t;
                const bool any_alive = group_any(alive, g);
                if (!any_alive || t >= a.max_steps) break;
            }
            // ---- write-back: state (episode number untouched), outputs ----
            if (active) {
                tile_env_store<WK>(c, gb, lane, s, wind_dirty, false);
#pragma unroll
                for (int q = 0; q < kObsDim; ++q) a.obs_out[env * kObsDim + q] = s.o[q];
                a.return_out[env] = s.d[D_RET];
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

// Collection: T steps of every env with auto-reset, each step's transition stored in the replay ring.  Row i of step
// t goes to slot (base_slot + t N + i) mod mem_size; the host guarantees T N <= mem_size, so no two rows of a call
// share a slot (tiles advance at different rates).  kRecord: every step also writes the recorder row of each
// recorded env (a.rec_ids) to row (rec_row0 + t) % capacity of a.rec_ring; the host guarantees T <= capacity.
template <int WK, bool kRecord>
__global__ void __launch_bounds__(kThreads, 1)
boat_collect_kernel(const __grid_constant__ DevCfg c, const __grid_constant__ CollectArgs a) {
    extern __shared__ __align__(128) unsigned char smem[];
    __shared__ uint32_t tmem_base_slot;
    __shared__ volatile int group_done[2];
    constexpr bool kCurves = (WK == WIND_VEL_CURVE || WK == WIND_ANGLE_RECT || WK == WIND_BOTH);
    __shared__ double setup_scratch[kCurves ? kEpiThreads / 32 : 1][kScratchDoubles];   // per epilogue warp
    __shared__ int record_column[kRecord ? 2 : 1][kRecord ? kTileM : 1];                 // per epilogue group
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    uint64_t *bars = reinterpret_cast<uint64_t *>(smem + kOffBar);
    if (tid < 2) group_done[tid] = 0;
    const uint32_t tmem = actor_prologue(a.blob, smem, &tmem_base_slot);
    const uint32_t sbase = smem_u32(smem);
    const long long n = c.n_envs;
    const long long n_tiles = (n + kTileM - 1) / kTileM;
    const long long G = gridDim.x;
    const long long my_tiles = n_tiles > (long long)blockIdx.x ? (n_tiles - blockIdx.x + G - 1) / G : 0;

    if (warp == kMmaWarp) {
        if (lane == 0) mma_serve_groups(bars, tmem, sbase, group_done);
    } else {
        const int g = warp >> 2, wq = warp & 3, row = wq * 32 + lane;
        uint64_t *b = bars + 5 * g;
        const uint32_t region = tmem + 256u * g + ((uint32_t)wq * 32u << 16);
        const float *b1 = reinterpret_cast<const float *>(smem + kOffB1), *b2 = reinterpret_cast<const float *>(smem + kOffB2),
                    *b3 = reinterpret_cast<const float *>(smem + kOffB3), *w3 = reinterpret_cast<const float *>(smem + kOffW3);
        unsigned char *a0 = smem + kOffA0 + g * (kTileM * kK1 * 2);
        const long long cnt = g == 0 ? (my_tiles + 1) / 2 : my_tiles / 2;
        const float max_a = __ldg(a.max_action);
        const float inv_Lm1 = c.f.inv_Lm1;
        const long long mem_size = a.rp.mem_size;
        float *ring_s = reinterpret_cast<float *>(a.rp.state), *ring_n = reinterpret_cast<float *>(a.rp.new_state);
        float *ring_a = reinterpret_cast<float *>(a.rp.action), *ring_r = reinterpret_cast<float *>(a.rp.reward);
        double *scratch = setup_scratch[kCurves ? warp : 0];
        long long pass = 0;
        for (long long i = 0; i < cnt; ++i) {
            const long long tile = (long long)blockIdx.x + (2 * i + g) * G;
            const long long blk = tile * 4 + wq;
            const long long env = blk * 32 + lane;
            const bool active = env < n;
            char *gb = c.state + (size_t)blk * (size_t)c.block_bytes;
            TileEnv s;
            tile_env_load<WK, true>(c, gb, lane, env, active, a.obs_inout, s);
            bool wind_dirty = false, episode_dirty = false;
            int code = BOATENV_TERM_NONE;
            float rew = 0.f;
            long long slot = a.rp.base_slot + env;   // < 2 mem_size: base_slot < mem_size and env < N <= mem_size
            if (slot >= mem_size) slot -= mem_size;
            int rec_col = -1;                        // the env's column in the recording ring, -1: not recorded
            long long rec_row = 0;
            if (kRecord) {
                rec_col = tile_record_column(a, g, row, tile * kTileM, n, record_column[kRecord ? g : 0]);
                rec_row = a.rec_row0;
            }
            for (int t = 0; t < a.steps; ++t) {
                actor_stage_a0(b, a0, row, s.o);
                actor_layer1_epilogue(b, (uint32_t)(pass & 1), region, b1);
                float acc[2];
                actor_layer2_heads<2>(b, region, b2, w3, acc);
                ++pass;
                bool need_wind = false;
                if (active) {
                    // ---- agent.remember (main.py:83-88, buffer.py:13-22): s before the step, s' after it (the
                    // terminal observation of an ending episode: the reset below overwrites o[] only afterwards)
#pragma unroll
                    for (int q = 0; q < kObsDim; ++q) ring_s[slot * kObsDim + q] = s.o[q];
                    int j, r;
                    const float action = act_and_substep<WK>(c, s, acc, b3, max_a, inv_Lm1, env,
                                                             a.step0 + (unsigned long long)t, a.seed, false, rew, code, j, r);
#pragma unroll
                    for (int q = 0; q < kObsDim; ++q) ring_n[slot * kObsDim + q] = s.o[q];
                    ring_a[slot] = action;
                    ring_r[slot] = rew;
                    a.rp.terminal[slot] = a.rp.done_flag_mode ? (code == BOATENV_TERM_REACHED_GOAL) : (code != BOATENV_TERM_NONE);
                    if (code != BOATENV_TERM_NONE) {
                        // ---- auto-reset in the env's own lane, as the step kernel does (Boat.__init__ boat_env.py:144-201)
                        count_episode_end(c, blk, code, s.d[D_RET]);
                        s.episode += 1u;
                        const int sy0 = episode_start_y(c, env, s.episode);   // :166-167, experiment 2 only
                        s.fx.start(c, s.d, sy0);
                        s.index = 0;
                        stage_reset_obs<float>(c, s.o, (float)sy0);
                        episode_dirty = true;
                        need_wind = kCurves;   // the new episode's first piece
                    } else if (kCurves && next_sample_in_next_piece(c, j, r)) {
                        need_wind = true;
                    }
                    if (kRecord && rec_col >= 0)
                        tile_env_record(c, a.rec_ring, rec_row * a.rec_n_ids + rec_col, s, action, rew, code);
                }
                if (kCurves) {
                    warp_wind_setups(c, need_wind, env, s, scratch);
                    wind_dirty |= need_wind;
                }
                slot += n;
                if (slot >= mem_size) slot -= mem_size;
                if (kRecord && ++rec_row == a.rec_ring.capacity) rec_row = 0;
            }
            if (active) {
                tile_env_store<WK>(c, gb, lane, s, wind_dirty, episode_dirty);
#pragma unroll
                for (int q = 0; q < kObsDim; ++q) a.obs_inout[env * kObsDim + q] = s.o[q];
                a.reward_out[env] = rew;
                if (a.done_out) a.done_out[env] = (code != BOATENV_TERM_NONE) ? 1 : 0;
                if (a.term_out) a.term_out[env] = (uint8_t)code;
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

using collect_kern_t = void (*)(const DevCfg, const CollectArgs);

template <bool kRecord>
collect_kern_t collect_kernel_for(int wind_kind) {
    switch (wind_kind) {
    case WIND_NONE: return boat_collect_kernel<WIND_NONE, kRecord>;
    case WIND_CONST: return boat_collect_kernel<WIND_CONST, kRecord>;
    case WIND_VEL_CURVE: return boat_collect_kernel<WIND_VEL_CURVE, kRecord>;
    case WIND_ANGLE_RECT: return boat_collect_kernel<WIND_ANGLE_RECT, kRecord>;
    case WIND_BOTH: return boat_collect_kernel<WIND_BOTH, kRecord>;
    default: return nullptr;
    }
}

template <bool kRecord>
cudaError_t collect_kernels_setup(int &n_sm) {
    return actor_kernels_setup<boat_collect_kernel<WIND_NONE, kRecord>, boat_collect_kernel<WIND_CONST, kRecord>,
                               boat_collect_kernel<WIND_VEL_CURVE, kRecord>, boat_collect_kernel<WIND_ANGLE_RECT, kRecord>,
                               boat_collect_kernel<WIND_BOTH, kRecord>>(n_sm);
}

// one CTA per SM at most: with fewer tiles than SMs every tile gets a CTA (and an SM) of its own rather than
// sharing a CTA with a second tile -- a tile's steps are a dependent chain, a second group only helps once the
// SMs run out (measured against pairing in profiles/rollout_eval.json, DESIGN.md section 8)
unsigned grid_for(long long n_envs, int n_sm) {
    const long long tiles = (n_envs + kTileM - 1) / kTileM;
#ifdef BOAT_ROLLOUT_PAIR_TILES   // measurement only (profiles/rollout_eval.py): two tiles per CTA also below n_sm tiles
    const long long ctas = (tiles + 1) / 2;
#else
    const long long ctas = tiles;
#endif
    return (unsigned)(ctas < n_sm ? ctas : n_sm);
}

}  // namespace

namespace boatenv {

cudaError_t launch_collect(const DevCfg &c, const CollectArgs &a, cudaStream_t stream) {
    const bool record = a.rec_ids != nullptr;
    const collect_kern_t kern = record ? collect_kernel_for<true>(c.wind_kind) : collect_kernel_for<false>(c.wind_kind);
    if (!kern) return cudaErrorInvalidValue;
    int n_sm = 0;
    const cudaError_t e = record ? collect_kernels_setup<true>(n_sm) : collect_kernels_setup<false>(n_sm);
    if (e != cudaSuccess) return e;
    kern<<<grid_for(c.n_envs, n_sm), kThreads, kSmemBytes, stream>>>(c, a);
    count_launch();
    return cudaGetLastError();
}

}  // namespace boatenv

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
    kern<<<grid_for(c.n_envs, n_sm), kThreads, kSmemBytes, (cudaStream_t)stream>>>(c, a);
    count_launch();
    return (int)cudaGetLastError();
}
