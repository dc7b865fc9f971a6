// aux_kernels.cuh -- reset, wind-table export, field access, counters, action filler.
#pragma once
#include "boat_step.cuh"

namespace boatenv {

// BoatEnv.reset()  boat_env.py:120-126 for the masked envs: a new Boat (:144-201) and a new Wind (wind.py:12-18).
// Two instantiations share the body.  LANE = true sets the wind up one env per LANE (no cooperation; 128 registers):
// it serves the warps with many envs to reset -- all of them in a full reset.  LANE = false serves the warps with only
// a few (a sparse mask) one env at a time with the warp-cooperative mapping, which finishes a single env ~5x sooner
// and runs at four times the occupancy.  A masked reset launches both; each skips the other's warps.  The two
// mappings give bit-identical coefficients (wind_setup.cuh).
constexpr int kResetLaneParallelFrom = 5;   // envs per warp from which the lane-parallel mapping is the faster one
template <typename T, bool LANE>
__global__ void __launch_bounds__(kTile, LANE ? 2 : 4) boat_reset_kernel(const __grid_constant__ DevCfg c,
                                                                    const uint8_t *mask, T *obs_out) {
    __shared__ double scratch_s[LANE ? 1 : kWarpsPerCta][LANE ? 1 : kScratchDoubles];
    const unsigned FULL = 0xffffffffu;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const long long i = (long long)blockIdx.x * kTile + threadIdx.x;
    const bool want = i < c.n_envs && (mask == nullptr || mask[i] != 0);
    double w8[8] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
    unsigned todo = __ballot_sync(FULL, want);
    // which instantiation owns this warp: experiments without curves need no setup (LANE owns everything)
    const bool lane_warp = c.ncurves == 0 || mask == nullptr || __popc(todo) >= kResetLaneParallelFrom;
    if (lane_warp != LANE) return;
    const uint32_t e_epi = want ? *episode_ptr(c, i) + 1u : 0u;
    if (c.ncurves > 0) {
        if (LANE) {
            if (want) wind_setup_lane_any(c, i, e_epi, 0, w8);
        } else {
            while (todo) {
                const int src = __ffs(todo) - 1;
                todo &= todo - 1;
                wind_setup_warp(c, __shfl_sync(FULL, i, src), __shfl_sync(FULL, e_epi, src), 0, scratch_s[LANE ? 0 : warp]);
                if (lane == src) {
#pragma unroll
                    for (int m = 0; m < 8; ++m) w8[m] = scratch_s[LANE ? 0 : warp][m];
                }
                __syncwarp();  // scratch is reused by the next env of this warp
            }
        }
    }
    if (!want) return;
    T d[D_COUNT], wa[4], wb[4], obs[kObsDim];
    const int sy0 = episode_start_y(c, i, e_epi);  // boat_env.py:166-167
    Fx<T> fx;
    fx.start(c, d, sy0);
    const uint32_t index_word = fx.pack(d, 0);
#pragma unroll
    for (int m = 0; m < 4; ++m) {
        wa[m] = (T)w8[m];
        wb[m] = (T)w8[4 + m];
    }
    store_vecs<T, D_COUNT>(block_section(c, i, 0), lane, d);
    *index_ptr(c, i) = index_word;
    *episode_ptr(c, i) = e_epi;
    if (c.ncurves >= 1) store_vecs<T, 4>(block_section(c, i, c.off_wa), lane, wa);
    if (c.ncurves >= 2) store_vecs<T, 4>(block_section(c, i, c.off_wb), lane, wb);
    if (obs_out) {
        stage_reset_obs<T>(c, obs, (T)sy0);
#pragma unroll
        for (int q = 0; q < kObsDim; ++q) obs_out[i * kObsDim + q] = obs[q];
    }
}

#ifndef BOAT_SETUPQ_MINBLOCKS
#define BOAT_SETUPQ_MINBLOCKS 2
#endif
// Follow-up of a K > 1 step launch: the episode-end queue (one region per step CTA) is drained one entry per
// THREAD (lane-parallel wind setup); the new episode's first-piece coefficients go straight into the env's state
// block.  Warps are dealt to regions round-robin; warp j of a region takes entries 32 j .. 32 j + 31, then
// strides by 32 * warps_per_region.
template <typename T>
__global__ void __launch_bounds__(kTile, BOAT_SETUPQ_MINBLOCKS) boat_setup_queue_kernel(const __grid_constant__ DevCfg c,
                                                                   const uint2 *__restrict__ entries,
                                                                   const unsigned *__restrict__ counts, int n_regions,
                                                                   int cap, int warps_per_region) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int w = (int)blockIdx.x * kWarpsPerCta + warp;
    const int region = w % n_regions, j0 = w / n_regions;
    if (j0 >= warps_per_region) return;
    const unsigned cnt = counts[region];
    for (unsigned e = (unsigned)j0 * 32u + (unsigned)lane; e < cnt; e += 32u * (unsigned)warps_per_region) {
        const uint2 en = __ldg(entries + (size_t)region * cap + e);
        double w8[8];
        wind_setup_lane_any(c, (long long)en.x, en.y, 0, w8);
        T w4[4];
#pragma unroll
        for (int m = 0; m < 4; ++m) w4[m] = (T)w8[m];
        store_vecs<T, 4>(block_section(c, en.x, c.off_wa), (int)(en.x & 31u), w4);
        if (c.ncurves >= 2) {
#pragma unroll
            for (int m = 0; m < 4; ++m) w4[m] = (T)w8[4 + m];
            store_vecs<T, 4>(block_section(c, en.x, c.off_wb), (int)(en.x & 31u), w4);
        }
    }
}

// env.boat.wind.wind_velocity / wind_angle (wind.py:16-17) of one env's CURRENT episode,
// as the step kernel sees them: per-piece folded coefficients evaluated at every sample.
// One warp.
static __global__ void __launch_bounds__(32) boat_wind_table_kernel(const __grid_constant__ DevCfg c, long long env,
                                                             double *wv, double *wa) {
    __shared__ double scratch_s[kScratchDoubles];
    __shared__ double folded[kMaxKnots - 1][8];
    const int lane = threadIdx.x;
    const double PI = 3.14159265358979323846;
    const uint32_t episode = *episode_ptr(c, env);
    if (c.ncurves > 0) {
        for (int j = 0; j < c.npieces; ++j) {
            const int first_index = (j * c.Lm1 + c.npieces - 1) / c.npieces;
            wind_setup_warp(c, env, episode, first_index, scratch_s);
            if (lane < 8) folded[j][lane] = scratch_s[lane];
            __syncwarp();
        }
    }
    __syncwarp();
    for (int idx = lane; idx < c.L; idx += 32) {
        double v = 0.0, th = 0.0;
        int j = 0, r = 0;
        double va = 0.0, vb = 0.0;
        if (c.ncurves > 0) {
            piece_of(c, idx, j, r);
            const double s = (double)r * c.inv_Lm1;
            const double *f = folded[j];
            va = ((f[3] * s + f[2]) * s + f[1]) * s + f[0];
            vb = ((f[7] * s + f[6]) * s + f[5]) * s + f[4];
        }
        switch (c.wind_kind) {
        case WIND_NONE: break;
        case WIND_CONST: v = c.p.max_velocity; th = c.direction_rad; break;
        case WIND_VEL_CURVE: v = va; th = c.direction_rad; break;
        case WIND_ANGLE_RECT: v = c.p.max_velocity; th = ((va <= 0.25) ? 0.0 : 1.0) * PI + PI / 2.0; break;
        case WIND_BOTH: v = va; th = vb; break;
        }
        wv[idx] = v;
        wa[idx] = th;
    }
}

// Scalar `field` (DynSlot order) of env i inside its block: vector row field / VW, slot field % VW.
template <typename T>
__device__ __forceinline__ T *dyn_scalar(const DevCfg &c, long long i, int field) {
    constexpr int W = VecOf<T>::W;
    return reinterpret_cast<T *>(block_section(c, i, 0)) + ((field / W) * 32 + (int)(i & 31)) * W + (field % W);
}

// Field access decodes / encodes the fixed-point carriers of the fp32 mode (struct Fx<float>, common.cuh):
// rudder_angle, s_x and s_y are exchanged as plain numbers (rounded to T on the way out).
__device__ __forceinline__ double read_field(const DevCfg &c, long long i, int field, double) {
    return *dyn_scalar<double>(c, i, field);
}
__device__ __forceinline__ double read_field(const DevCfg &c, long long i, int field, float) {
    const float raw = *dyn_scalar<float>(c, i, field);
    return decode_field(c, field, raw, field == D_RUDDER ? *index_ptr(c, i) : 0u);
}
__device__ __forceinline__ void write_field(const DevCfg &c, long long i, int field, double v, double) {
    *dyn_scalar<double>(c, i, field) = v;
}
__device__ __forceinline__ int fixed_from(double v, int shift) {
    const double x = rint(v * (double)(1 << shift));
    return x >= 2147483647.0 ? 2147483647 : (x <= -2147483648.0 ? (int)0x80000000 : (int)x);
}
__device__ __forceinline__ void write_field(const DevCfg &c, long long i, int field, double v, float) {
    float *p = dyn_scalar<float>(c, i, field);
    if (field == D_RUDDER) {
        double x = rint(v * 4398046511104.0);
        x = fmin(fmax(x, -(double)kRudLimit), (double)kRudLimit);
        const long long rud = (long long)x;
        *p = __int_as_float((int)(rud >> kRudLoBits));
        uint32_t *ix = index_ptr(c, i);
        *ix = (*ix & kIndexMask) | (((uint32_t)rud & ((1u << kRudLoBits) - 1u)) << kIndexBits);
    } else if (field == D_SX) {
        *p = __int_as_float(fixed_from(v, c.f.sx_shift));
    } else if (field == D_SY) {
        *p = __int_as_float(fixed_from(v, c.f.sy_shift));
    } else {
        *p = (float)v;
    }
}

template <typename T>
__global__ void boat_get_field_kernel(const __grid_constant__ DevCfg c, int field, void *out) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= c.n_envs) return;
    if (field < D_COUNT) {
        reinterpret_cast<T *>(out)[i] = (T)read_field(c, i, field, T());
    } else {
        reinterpret_cast<uint32_t *>(out)[i] = (field == BOATENV_F_STEP_INDEX) ? (*index_ptr(c, i) & kIndexMask) : *episode_ptr(c, i);
    }
}

template <typename T>
__global__ void boat_set_field_kernel(const __grid_constant__ DevCfg c, int field, const void *in) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= c.n_envs) return;
    if (field < D_COUNT) {
        write_field(c, i, field, (double)reinterpret_cast<const T *>(in)[i], T());
    } else {
        const uint32_t x = reinterpret_cast<const uint32_t *>(in)[i];
        if (field == BOATENV_F_STEP_INDEX) {
            uint32_t *ix = index_ptr(c, i);
            *ix = (*ix & ~kIndexMask) | (x & kIndexMask);   // the bits above the index belong to the rudder (fp32 mode)
        } else {
            *episode_ptr(c, i) = x;
        }
    }
}

// All ten fields (boatenv_field order) of ONE env as doubles: what env.boat.* / return_all_data
// (boat_env.py:128-140, main.py:94) read after a step.  One thread.
template <typename T>
__global__ void boat_env_state_kernel(const __grid_constant__ DevCfg c, long long i, double *out) {
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
#pragma unroll
    for (int f = 0; f < D_COUNT; ++f) out[f] = read_field(c, i, f, T());
    out[BOATENV_F_STEP_INDEX] = (double)(*index_ptr(c, i) & kIndexMask);
    out[BOATENV_F_EPISODE] = (double)*episode_ptr(c, i);
}

// counters[kCounterSlots][32 doubles, first 8 used] -> out[8]
static __global__ void boat_reduce_counters_kernel(const double *counters, double *out) {
    const int t = threadIdx.x;
    if (t < kNumCounters) {
        double s = 0.0;
        for (int r = 0; r < kCounterSlots; ++r) s += counters[r * 32 + t];
        out[t] = s;
    }
}

// uniform(-1,1) * scale actions: the policy "A1" of SURVEY.md 8(d).  One Philox4x32-10 call
// yields the actions of FOUR consecutive global envs: env g at step t gets word (g & 3) of
// Philox(counter = (g >> 2, t), key = seed), as a 23-bit value exactly representable in fp32.
// One thread per global quad, 128-bit stores when the shard starts on a quad boundary.
template <typename T>
__global__ void __launch_bounds__(256) boat_fill_actions_kernel(const __grid_constant__ DevCfg c,
                                                                unsigned long long step_counter, double scale, T *out) {
    const long long q = (long long)blockIdx.x * blockDim.x + threadIdx.x;  // quad index within the shard
    const long long quad = (c.env_id_offset >> 2) + q;                     // global quad
    const long long first = quad * 4 - c.env_id_offset;                    // local index of the quad's first env
    if (first >= c.n_envs) return;
    const Philox4 r = philox4x32_10((uint32_t)quad, (uint32_t)((unsigned long long)quad >> 32), (uint32_t)step_counter,
                                    kStreamAction | (uint32_t)((step_counter >> 32) & 0x0fffffffu), (uint32_t)c.seed,
                                    (uint32_t)(c.seed >> 32));
    const float sc = (float)scale;
    T v[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) v[k] = (T)(sc * ((float)(philox_word(r, k) >> 8) * (1.0f / 8388608.0f) - 1.0f));
    if (first >= 0 && first + 4 <= c.n_envs && ((reinterpret_cast<uintptr_t>(out + first) & 15u) == 0)) {
        using V = typename VecOf<T>::type;
        constexpr int W = VecOf<T>::W;
#pragma unroll
        for (int k = 0; k < 4 / W; ++k) __stcs(reinterpret_cast<V *>(out + first) + k, pack(&v[k * W]));
    } else {
#pragma unroll
        for (int k = 0; k < 4; ++k)
            if (first + k >= 0 && first + k < c.n_envs) out[first + k] = v[k];
    }
}

}  // namespace boatenv
