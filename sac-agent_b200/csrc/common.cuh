// common.cuh -- shared host/device definitions of libboatenv (sm_100a).
//
// State layout in HBM (DESIGN.md "data layout"): tile-blocked structure-of-arrays.  The
// carried state of 32 consecutive envs (one warp's tile) is ONE contiguous, 16-byte
// aligned block
//     [dyn vector 0 x 32][dyn vector 1 x 32]..[step index (u32) x 32][wind A vectors x 32][wind B vectors x 32][episode (u32) x 32]
// of 16-byte vectors (VW = 16/sizeof(T) scalars each), so that
//   * everything a step reads is fetched by a single TMA bulk copy (cp.async.bulk) into shared memory,
//   * a warp's access to one vector row is one fully coalesced 512-byte LDS/LDG/STG.128.
// The episode number sits at the END of the block, outside the bulk copy: only a reset reads or writes it, so it
// costs no HBM traffic on the common path (it used to travel with the step index: 8 bytes per env-step).
// Block size: 32 * (16*ND + 4 + 16*NW*ncurves + 4) bytes = 1280 / 1792 / 2304 (fp32; exp 1-3 / 4-5 / 6).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/boatenv.h"

namespace boatenv {

constexpr int kObsDim = BOATENV_OBS_DIM;
#ifndef BOAT_CTA_THREADS
#define BOAT_CTA_THREADS 256
#endif
constexpr int kTile = BOAT_CTA_THREADS;  // threads per CTA (8 self-contained warps)
constexpr int kWarpsPerCta = kTile / 32;
constexpr int kMaxKnots = 16;   // fixed_points supported by this build (reference default 8)
constexpr int kCounterSlots = 32;  // replicated counter rows (spread atomics over L2 slices)
constexpr int kNumCounters = 8;

// Dynamic scalars carried per env (group "dyn"), in this order.
enum DynSlot { D_VX = 0, D_VY = 1, D_VR = 2, D_RUDDER = 3, D_SX = 4, D_SY = 5, D_SR = 6, D_RET = 7, D_COUNT = 8 };

// Wind treatment per experiment (wind.py:26-63).
enum WindKind {
    WIND_NONE = 0,        // exp 1, 2: zero wind
    WIND_CONST = 1,       // exp 3: constant velocity and direction
    WIND_VEL_CURVE = 2,   // exp 4: random velocity curve, constant direction
    WIND_ANGLE_RECT = 3,  // exp 5: constant velocity, rectified random direction
    WIND_BOTH = 4         // exp 6: random velocity curve and random direction curve
};

// fp32 production constants: the reference's chains of config multiplications folded
// on the host in double precision, then rounded once.
struct FastConsts {
    float dt, tenth;
    float kdx, kJ, kT, cxy, inv_mx;     // surge   boat_env.py:213-239
    float kdy, kru, cyx, inv_my;        // sway    boat_env.py:241-265
    float kh, kmr, inv_I;               // yaw     boat_env.py:267-281
    float kwx, kwy;                     // wind drag factors
    float fwx_c, fwy_c;                 // exp 3: constant wind force components
    float cos_dir, sin_dir;             // exp 4: constant direction
    float fwx_lo, fwy_lo, fwx_hi, fwy_hi;  // exp 5: force for angle pi/2 and 3pi/2
    float inv_goal, inv_5, inv_ax, W, inv_2W, inv_2, inv_ay, inv_2pi, inv_vr, inv_ar,
        third_pi, inv_rud, inv_fuel;    // obs normalisers boat_env.py:308-326
    float fuel0, goal, oob, pi3, pi4, pi2;
    float rew_inv_W, rew_k, rew_y0;     // reward_functions.py:52-54
    float inv_Lm1;                      // 1 / (L - 1): wind sample index -> local spline coordinate
    // exact carriers of the fp32 mode (struct Fx<float> below): fixed-point positions and rudder
    float sx_k, sy_k;                   // dt * 2^sx_shift, dt * 2^sy_shift: position increment -> fixed-point units
    float sx_inv, sy_inv;               // 2^-sx_shift, 2^-sy_shift
    int sx_shift, sy_shift;
    int sx_goal;                        // s_x >= goal_line        <=> sx >= sx_goal   (boat_env.py:85)
    int sy_oob;                         // abs(s_y) > W + offset   <=> |sy| > sy_oob   (boat_env.py:90)
    unsigned sy_oob2;                   // 2 * sy_oob
    float sx_obs, sy_obs;               // 2^-sx_shift / goal_line, 2^-sy_shift / (2 W): fixed point -> normalised observation
};

struct DevCfg {
    long long n_envs;
    long long env_id_offset;
    unsigned long long seed;
    int experiment, wind_kind, test_mode, ncurves;
    int fp, npieces;          // wind.fixed_points and fp - 1
    int L, Lm1;               // wind table length int(t_max/dt) (wind.py:14-15), L - 1
    unsigned magic_m, magic_s;  // floor(n / Lm1) == __umulhi(n, magic_m) >> magic_s for n <= L * npieces
    double inv_Lm1;           // 1.0 / Lm1
    int timeout_steps;        // first step count n with accumulated t >= t_max (boat_env.py:98)
    int fuel_steps;           // first step count n with fuel - n < 0 (boat_env.py:70,94)
    int s_y_half;             // int(track_width * 0.8) (boat_env.py:148-149)
    boatenv_params p;         // raw reference parameters (fp64 validation mode uses these)
    double direction_rad;     // float(direction) * (pi/180)   wind.py:44
    double prop_d4;           // np.power(propeller_diameter, 4)  boat_env.py:226
    FastConsts f;
    // device buffers (owned by the handle)
    char *state;              // [ceil(n_envs / 32)][block_bytes] tile-blocked state (see top of file)
    int block_bytes;          // bytes of one 32-env block
    int off_idx, off_wa, off_wb;  // byte offsets of the step-index / wind A / wind B sections inside a block
    int off_epi;              // byte offset of the episode row (the last 128 bytes of a block) = bytes the step kernel's bulk copy fetches
    const double *basis;      // [npieces][4][fp] cardinal not-a-knot spline basis
    const int *piece_bounds;  // [npieces][2] first / last wind sample index that piece_of() assigns to each spline piece
    float per_piece, inv_per_piece;  // Lm1 / npieces: wind samples per spline piece, and its reciprocal
    double *counters;         // [kCounterSlots][kNumCounters]
    const int32_t *ovr_s_y;   // optional episode-draw overrides (validation)
    const double *ovr_knots;
};

struct ReplayView {   // fused agent.remember (main.py:83-88, buffer.py:13-22); null = off
    void *state, *new_state, *action, *reward;
    uint8_t *terminal;
    long long mem_size, base_slot;   // base_slot = mem_cntr % mem_size: env i goes to slot base_slot + i (mod size)
    int done_flag_mode;
};

struct StepArgs {
    long long env_begin, env_end;   // this launch covers envs [env_begin, env_end)
    const void *actions;
    long long action_stride;   // elements between sub-step k and k+1 of one env (0: repeat)
    int ksteps;
    void *obs_out, *reward_out;
    uint8_t *done_out, *term_out;
    void *final_obs_out;
    int32_t *steps_out;
    const void *obs_in;        // previous observations (fused replay store only)
    uint32_t flags;
    int reverse;               // sweep direction of this launch (alternates, see boat_step.cuh)
    int no_bulk;               // outputs live in mapped HOST memory (small-N zero-copy step): element-wise stores only
    // K > 1 launches: finished episodes are queued here (one region per CTA) and get their new wind
    // coefficients from a follow-up kernel at full occupancy (boat_setup_queue_kernel); null = inline
    uint2 *kq_entries;         // [regions][kq_cap] (env, new episode)
    unsigned *kq_counts;       // [regions]
    long long kq_total;        // entries allocated
    int kq_cap;                // entries per region (set by the launcher)
    ReplayView rp;
};

// ---------------------------------------------------------------------------------
// Philox4x32-10 (Salmon et al., SC'11), counter-based: no per-env RNG state in HBM.
// ---------------------------------------------------------------------------------
struct Philox4 { uint32_t x, y, z, w; };

__host__ __device__ __forceinline__ void mulhilo32(uint32_t a, uint32_t b, uint32_t &hi, uint32_t &lo) {
#ifdef __CUDA_ARCH__
    hi = __umulhi(a, b);
    lo = a * b;
#else
    uint64_t p = (uint64_t)a * (uint64_t)b;
    hi = (uint32_t)(p >> 32);
    lo = (uint32_t)p;
#endif
}

__host__ __device__ __forceinline__ Philox4 philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3,
                                                         uint32_t k0, uint32_t k1) {
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        uint32_t hi0, lo0, hi1, lo1;
        mulhilo32(0xD2511F53u, c0, hi0, lo0);
        mulhilo32(0xCD9E8D57u, c2, hi1, lo1);
        uint32_t n0 = hi1 ^ c1 ^ k0, n1 = lo1, n2 = hi0 ^ c3 ^ k1, n3 = lo0;
        c0 = n0; c1 = n1; c2 = n2; c3 = n3;
        k0 += 0x9E3779B9u;
        k1 += 0xBB67AE85u;
    }
    Philox4 o = {c0, c1, c2, c3};
    return o;
}

__host__ __device__ __forceinline__ uint32_t philox_word(const Philox4 &p, int i) {
    return i == 0 ? p.x : (i == 1 ? p.y : (i == 2 ? p.z : p.w));
}

// Counter layout: (env_lo, env_hi, episode_or_step, stream | block).
constexpr uint32_t kStreamEpisode = 0x00000000u;  // block 0: s_y_start; block 1+: knots
constexpr uint32_t kStreamAction = 0xA0000000u;   // uniform(-1,1) test / bench policy
constexpr uint32_t kStreamReplay = 0xB0000000u;   // replay-buffer sample indices
constexpr uint32_t kStreamToy = 0xC0000000u;      // toy-env parameter jitter

// np.random.sample() stand-in: 23 random bits -> (2k+1) * 2^-24, strictly inside (0,1)
// and exactly representable in fp32 AND fp64 (both precisions see identical knots).
__host__ __device__ __forceinline__ double knot_from_word(uint32_t w) {
    return (double)(((w >> 9) << 1) | 1u) * (1.0 / 16777216.0);
}

// np.random.randint(-half, half) stand-in (multiply-shift range reduction).
__host__ __device__ __forceinline__ int s_y_from_word(uint32_t w, int half) {
    return -half + (int)(((uint64_t)w * (uint64_t)(2 * half)) >> 32);
}

__host__ __device__ __forceinline__ double episode_knot(unsigned long long seed, long long genv, uint32_t episode,
                                                       int flat_index /* curve * fp + k */) {
    Philox4 r = philox4x32_10((uint32_t)genv, (uint32_t)((unsigned long long)genv >> 32), episode,
                              kStreamEpisode | (uint32_t)(1 + (flat_index >> 2)), (uint32_t)seed,
                              (uint32_t)(seed >> 32));
    return knot_from_word(philox_word(r, flat_index & 3));
}

__host__ __device__ __forceinline__ int episode_s_y_start(unsigned long long seed, long long genv, uint32_t episode,
                                                         int half) {
    Philox4 r = philox4x32_10((uint32_t)genv, (uint32_t)((unsigned long long)genv >> 32), episode, kStreamEpisode,
                              (uint32_t)seed, (uint32_t)(seed >> 32));
    return s_y_from_word(r.x, half);
}

// ---------------------------------------------------------------------------------
// 16-byte vector access
// ---------------------------------------------------------------------------------
template <typename T> struct VecOf;
template <> struct VecOf<float> { using type = float4; static constexpr int W = 4; };
template <> struct VecOf<double> { using type = double2; static constexpr int W = 2; };

// ---------------------------------------------------------------------------------
// Exact carriers of the fp32 production mode.  The termination cascade (boat_env.py:84-105) and the rudder
// penalty (:107) compare ACCUMULATED quantities with thresholds; accumulated in fp32 they drift by ~1e-6 (rudder)
// / ~5e-3 m (s_x) and flip a threshold one step early or late in ~1e-4 of the episodes.  So the fp32 mode carries
//   rudder  as a 44-bit fixed-point number, 2^-42 rad per unit, range +-2 rad (saturating): the upper 32 bits
//           sit in the D_RUDDER slot of the state, the lower 12 in bits 20..31 of the step-index word.  The
//           rudder depends on the actions only, so it stays within ~2e-12 rad of the reference's fp64 sum.
//   s_x,s_y as int32 fixed-point numbers (2^-19 m / 2^-21 m for the reference track, saturating) in their slots.
// No extra bytes per env.  The fp64 validation mode carries plain doubles (Fx<double> is empty).
// ---------------------------------------------------------------------------------
constexpr int kRudShift = 42;            // rudder units per rad = 2^42
constexpr int kRudLoBits = 12;           // low bits of the rudder stored beside the step index
constexpr int kIndexBits = 20;           // step index: bits 0..19 of the index word (L <= 2^20 - 64)
constexpr uint32_t kIndexMask = (1u << kIndexBits) - 1u;
constexpr long long kRudLimit = (1LL << 43) - 1;   // |rudder| saturates just below 2 rad
// abs(rudder) > pi/3, pi/4 (boat_env.py:102,107) <=> |rud| > floor(fp64(pi/3) * 2^42), floor(fp64(pi/4) * 2^42)
constexpr double kRudPi3 = 4605623536476.0, kRudPi4 = 3454217652357.0;
constexpr unsigned long long kRudPi3Bits = 0x4290C152382D7000ull, kRudPi4Bits = 0x428921FB54442800ull;  // their bit patterns

#ifdef __CUDACC__
// position accumulation: saturating (5 instructions) in the K = 1 kernels, where an env that was not reset after
// its episode ended can be stepped on and on; plain (1 instruction) in the issue-bound K > 1 kernels, where an env
// stops at its first done inside a window.  Identical wherever nothing overflows.
template <bool SAT> __device__ __forceinline__ int add_fixed(int a, int b) {
    if (!SAT) return a + b;
    int r;
    asm("add.sat.s32 %0, %1, %2;" : "=r"(r) : "r"(a), "r"(b));
    return r;
}

template <typename T> struct Fx;
template <> struct Fx<double> {
    __device__ __forceinline__ void load(const DevCfg &, const double (&)[D_COUNT], uint32_t ixw, int &index) { index = (int)(ixw & kIndexMask); }
    __device__ __forceinline__ uint32_t pack(double (&)[D_COUNT], int index) const { return (uint32_t)index; }
    __device__ __forceinline__ void start(const DevCfg &, double (&d)[D_COUNT], int s_y0) {  // Boat.__init__ boat_env.py:144-201
#pragma unroll
        for (int q = 0; q < D_COUNT; ++q) d[q] = 0.0;
        d[D_SY] = (double)s_y0;
    }
};
template <> struct Fx<float> {
    // rudder angle in units of 2^-42 rad, held as an INTEGER-VALUED double while a launch runs (sums of integers
    // below 2^53 are exact, and the fp64 pipe does them in 1 instruction where int64 needs 2-4); stored as 44 bits
    double rud;
    int sx, sy;
    __device__ __forceinline__ void load(const DevCfg &, const float (&d)[D_COUNT], uint32_t ixw, int &index) {
        index = (int)(ixw & kIndexMask);
        rud = fma((double)__float_as_int(d[D_RUDDER]), (double)(1 << kRudLoBits), (double)(ixw >> kIndexBits));
        sx = __float_as_int(d[D_SX]);
        sy = __float_as_int(d[D_SY]);
    }
    __device__ __forceinline__ long long rud_bits() const {   // saturated to the 44 stored bits
        return __double2ll_rn(fmin(fmax(rud, -(double)kRudLimit), (double)kRudLimit));
    }
    // the bit patterns that go to HBM (d keeps its float views; call on a copy or right before the store);
    // returns the step-index word (the index and the low rudder bits)
    __device__ __forceinline__ uint32_t pack(float (&d)[D_COUNT], int index) const {
        const long long q = rud_bits();
        d[D_RUDDER] = __int_as_float((int)(q >> kRudLoBits));
        d[D_SX] = __int_as_float(sx);
        d[D_SY] = __int_as_float(sy);
        return (uint32_t)index | (((uint32_t)q & ((1u << kRudLoBits) - 1u)) << kIndexBits);
    }
    __device__ __forceinline__ float rudder_view() const { return (float)rud * 2.27373675443232059478759765625e-13f; }  // 2^-42
    __device__ __forceinline__ void start(const DevCfg &c, float (&d)[D_COUNT], int s_y0) {
#pragma unroll
        for (int q = 0; q < D_COUNT; ++q) d[q] = 0.0f;
        d[D_SY] = (float)s_y0;
        rud = 0.0;
        sx = 0;
        sy = s_y0 * (1 << c.f.sy_shift);   // |s_y0| <= 0.8 W: no overflow (the shift leaves room for W + offset)
    }
};

// The plain value of dyn slot `field` of an fp32 env from the bits Fx<float>::pack stores: `raw` the slot, `ixw` the
// step-index word (read for the rudder only).  The fixed-point carriers (rudder_angle, s_x, s_y) are decoded; the
// other slots are plain floats.  boatenv_get_field, boatenv_record_rows and the recording collect kernel all read
// the state through this one decode.
__device__ __forceinline__ double decode_field(const DevCfg &c, int field, float raw, uint32_t ixw) {
    if (field == D_RUDDER) {
        const long long rud = ((long long)__float_as_int(raw) << kRudLoBits) | (long long)(ixw >> kIndexBits);
        return (double)rud * (1.0 / 4398046511104.0);
    }
    if (field == D_SX) return (double)__float_as_int(raw) * (double)c.f.sx_inv;
    if (field == D_SY) return (double)__float_as_int(raw) * (double)c.f.sy_inv;
    return (double)raw;
}

// ---------------------------------------------------------------------------------
// mbarrier and proxy-fence primitives (sm_90+/sm_100a PTX), shared by the step kernels' TMA pipeline
// (boat_step.cuh) and the tcgen05 actor pass (actor_tc.cuh)
// ---------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_fence_init() {
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "WAIT_%=:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra DONE_%=;\n\t"
        "bra WAIT_%=;\n\t"
        "DONE_%=:\n\t"
        "}" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
// generic-proxy writes (st.shared) -> visible to the async proxy (a bulk store or an MMA that reads them next)
__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// round-to-nearest integer of x * k for |x * k| < 2^22 without the conversion pipe (one FFMA + one IADD)
__device__ __forceinline__ int fixed_increment(float x, float k) {
    return __float_as_int(fmaf(x, k, 12582912.0f)) - 0x4B400000;
}

__device__ __forceinline__ void unpack(const float4 &v, float *o) { o[0] = v.x; o[1] = v.y; o[2] = v.z; o[3] = v.w; }
__device__ __forceinline__ void unpack(const double2 &v, double *o) { o[0] = v.x; o[1] = v.y; }
__device__ __forceinline__ float4 pack(const float *o) { return make_float4(o[0], o[1], o[2], o[3]); }
__device__ __forceinline__ double2 pack(const double *o) { return make_double2(o[0], o[1]); }

// Vectors per env of the two section kinds.
template <typename T> struct Lay {
    static constexpr int ND = D_COUNT * (int)sizeof(T) / 16;  // dyn: 8 scalars
    static constexpr int NW = 4 * (int)sizeof(T) / 16;        // one wind curve: 4 cubic coefficients
};

__host__ __device__ __forceinline__ long long num_blocks(long long n_envs) { return (n_envs + 31) >> 5; }

// Section `off` of the block that holds env i (global memory).
__device__ __forceinline__ char *block_section(const DevCfg &c, long long i, int off) {
    return c.state + (i >> 5) * (long long)c.block_bytes + off;
}

// Step index (Boat.index) and episode number of env i (global memory).
__device__ __forceinline__ uint32_t *index_ptr(const DevCfg &c, long long i) {
    return reinterpret_cast<uint32_t *>(block_section(c, i, c.off_idx)) + (i & 31);
}
__device__ __forceinline__ uint32_t *episode_ptr(const DevCfg &c, long long i) {
    return reinterpret_cast<uint32_t *>(block_section(c, i, c.off_epi)) + (i & 31);
}

// NS scalars of lane `lane` from a section (vector row v at sec + (v*32 + lane)*16).
template <typename T, int NS>
__device__ __forceinline__ void load_vecs(const char *sec, int lane, T (&out)[NS]) {
    using V = typename VecOf<T>::type;
    constexpr int W = VecOf<T>::W;
    static_assert(NS % W == 0, "section must be a whole number of 16-byte vectors");
    const V *p = reinterpret_cast<const V *>(sec) + lane;
#pragma unroll
    for (int v = 0; v < NS / W; ++v) unpack(p[v * 32], &out[v * W]);
}

// State stores: default (evict-normal) L2 policy, unlike the streamed outputs: the state is the only
// data the NEXT launch reads again, and launches alternate their sweep direction (boat_step.cuh).
template <typename V> __device__ __forceinline__ void st_state(V *p, const V &v) { *p = v; }

// 128-bit stores of NS scalars of lane `lane` into a section.
template <typename T, int NS>
__device__ __forceinline__ void store_vecs(char *sec, int lane, const T (&in)[NS]) {
    using V = typename VecOf<T>::type;
    constexpr int W = VecOf<T>::W;
    V *p = reinterpret_cast<V *>(sec) + lane;
#pragma unroll
    for (int v = 0; v < NS / W; ++v) st_state(p + v * 32, pack(&in[v * W]));
}

// Plain per-array SoA helpers (toy envs: 4 scalars per env in [vector][env] order).
template <typename T, int NS>
__device__ __forceinline__ void load_group(const void *base, long long n, long long i, T (&out)[NS]) {
    using V = typename VecOf<T>::type;
    constexpr int W = VecOf<T>::W;
    const V *p = reinterpret_cast<const V *>(base);
#pragma unroll
    for (int v = 0; v < NS / W; ++v) unpack(__ldcs(p + (long long)v * n + i), &out[v * W]);
}
template <typename T, int NS>
__device__ __forceinline__ void store_group(void *base, long long n, long long i, const T (&in)[NS]) {
    using V = typename VecOf<T>::type;
    constexpr int W = VecOf<T>::W;
    V *p = reinterpret_cast<V *>(base);
#pragma unroll
    for (int v = 0; v < NS / W; ++v) __stcs(p + (long long)v * n + i, pack(&in[v * W]));
}

__device__ __forceinline__ double warp_min(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmin(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}
__device__ __forceinline__ double warp_max(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
#endif  // __CUDACC__

}  // namespace boatenv
