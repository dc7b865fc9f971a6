// boat_step.cuh -- the batched BoatEnv.step kernel (boat_env.py:67-115): one thread per env, state in
// registers across K fused sub-steps, in-kernel termination cascade, statistics and auto-reset.
//   * persistent, self-contained step warps walk the 32-env state blocks of the tile-blocked layout
//     (common.cuh); each keeps one TMA bulk copy (cp.async.bulk + mbarrier) of its next block in flight;
//     (the copy skips the block's episode row, which only an ending episode touches, and is held back by a
//     warp vote until every lane's loads of the stage being refilled have returned);
//   * state goes back with 128-bit stores, the [32][11] observation tile with one bulk store;
//   * the fused agent.remember variant also moves the previous observation tile to the replay ring through
//     shared memory with bulk copies only;
//   * K = 1 kernels of the random-wind experiments are warp-specialised: wind-setup requests travel
//     through a shared-memory ring to dedicated setup warps (wind_setup.cuh does the maths).
// Instantiated for float (production) in step_f32.cu and for double (validation, reference operation
// order, compiled with -fmad=false) in step_f64.cu.  Design notes and measurements: DESIGN.md section 4.
#pragma once
#include "common.cuh"
#include "wind_setup.cuh"

namespace boatenv {

// ---------------------------------------------------------------------------------
// fp32 transcendental helpers: Cody-Waite reduction by pi (k = rint(x/pi), r = x - k*pi in
// [-pi/2, pi/2], sin x = (-1)^k sin r, cos x = (-1)^k cos r) + near-minimax polynomials
// (odd degree 9 / even degree 10, fitted on [-pi/2, pi/2]); |error| ~1.3e-7 for |x| up to
// ~1e4, branch-free, no slow path.  13 instructions for sin, 18 for sin+cos.
// ---------------------------------------------------------------------------------
__device__ __forceinline__ float reduce_pi(float x, uint32_t &sign) {
    float k = fmaf(x, 0.318309886f, 12582912.0f);
    sign = (uint32_t)__float_as_int(k) << 31;     // parity of k -> sign bit
    k -= 12582912.0f;
    float r = fmaf(k, -3.14159274e+00f, x);       // fl32(pi)
    return fmaf(k, 8.74227766e-08f, r);           // fl32(pi) - pi = 8.742e-8
}
__device__ __forceinline__ float sin_poly(float r, float r2) {
    float p = fmaf(2.5904564607e-06f, r2, -1.9800881965e-04f);
    p = fmaf(p, r2, 8.3328995679e-03f);
    p = fmaf(p, r2, -1.6666647620e-01f);
    return fmaf(r2 * r, p, r);
}
__device__ __forceinline__ float cos_poly(float r2) {
    float q = fmaf(-2.6051228305e-07f, r2, 2.4760146865e-05f);
    q = fmaf(q, r2, -1.3888361132e-03f);
    q = fmaf(q, r2, 4.1666636239e-02f);
    q = fmaf(q, r2, -4.9999999358e-01f);
    return fmaf(q, r2, 1.0f);
}
__device__ __forceinline__ float fast_sinf(float x) {
    uint32_t sign;
    const float r = reduce_pi(x, sign);
    return __uint_as_float(__float_as_uint(sin_poly(r, r * r)) ^ sign);
}
__device__ __forceinline__ void fast_sincosf(float x, float &s, float &c) {
    uint32_t sign;
    const float r = reduce_pi(x, sign);
    const float r2 = r * r;
    s = __uint_as_float(__float_as_uint(sin_poly(r, r2)) ^ sign);
    c = __uint_as_float(__float_as_uint(cos_poly(r2)) ^ sign);
}

// ---------------------------------------------------------------------------------
// One sub-step of the dynamics.  d[] is the carried state (DynSlot order), `index` the
// pre-increment Boat.index (== sub-steps done in this episode), (w, th) the wind sample
// wind[index].  Updates d[], returns the three accelerations (they are observations),
// the reward and the termination code.
// ---------------------------------------------------------------------------------
template <int WK, bool SAT>
__device__ __forceinline__ void substep(const DevCfg &c, double (&d)[D_COUNT], Fx<double> &, int index, double action,
                                        double w, double th, double (&acc)[3], double &reward, int &code) {
    // fp64 validation mode: the reference's own operation order (Python's a*b*c is
    // (a*b)*c); this translation unit is built with -fmad=false.
    const boatenv_params &p = c.p;
    const double PI = 3.14159265358979323846;
    const bool first = (index == 0);  // control_blocks.py:21-22: call 0 returns initial_value
    double rudder = d[D_RUDDER];
    if (c.test_mode == 0) rudder += action / 10.0;  // boat_env.py:72-73
    double v_x = d[D_VX], v_y = d[D_VY], v_r = d[D_VR];
    const double n = 20.0;  // boat_env.py:178

    double F_Wx = 0.0, F_Wy = 0.0;
    if (WK != WIND_NONE) {  // boat_env.py:230-236, 256-262
        const double sgn = (double)((w > 0.0) - (w < 0.0));
        double sin_th, cos_th;
        sincos(th, &sin_th, &cos_th);   // one argument reduction for both (same values as sin() / cos())
        F_Wx = w * w * sgn * p.c_r_front * 0.5 * p.rho * p.boat_area_front;
        F_Wx = F_Wx * cos_th;
        F_Wy = w * w * sgn * p.c_r_side * 0.5 * p.rho * p.boat_area_side;
        F_Wy = F_Wy * sin_th;
    }
    // eom_longitudinal  boat_env.py:213-239 (old v_x, v_y, v_r)
    double F_R = v_x * v_x * p.c_r_front * 0.5 * p.rho * p.boat_area_front;
    double v_x_w = v_x * (1.0 - p.wake_friction);
    double J = v_x_w / (n * p.propeller_diameter);
    double F_T = sin(J) * (n * n) * p.rho * c.prop_d4 * (1.0 - p.thrust_deduction);
    double F_C = v_y * (p.boat_m + p.boat_m_y) * v_r;
    const double a_x = (-F_R + F_T + F_C + F_Wx) / (p.boat_m + p.boat_m_x);
    v_x = first ? 3.0 : a_x * p.dt + v_x;  // boat_env.py:158,205
    // eom_transverse  boat_env.py:241-265 (NEW v_x, old v_y, v_r)
    const double sin_rud = sin(rudder);
    const double sgn_vy = (double)((v_y > 0.0) - (v_y < 0.0));
    F_R = v_y * v_y * p.c_r_side * 0.5 * p.rho * p.boat_area_side * sgn_vy;
    double F_RU = v_x * v_x * p.c_r_front * 0.5 * p.rho * p.rudder_area;
    F_RU = sin_rud * F_RU;
    F_C = v_x * (p.boat_m + p.boat_m_x) * v_r;
    const double a_y = (-F_R + F_RU + F_C + F_Wy) / (p.boat_m + p.boat_m_y);
    v_y = first ? 0.0 : a_y * p.dt + v_y;  // boat_env.py:163,207
    // eom_yawning  boat_env.py:267-281 (NEW v_x, old v_r)
    const double sgn_vr = (double)((v_r > 0.0) - (v_r < 0.0));
    const double sgn_vx = (double)((v_x > 0.0) - (v_x < 0.0));
    const double M_hull = v_r * v_r * p.c_r_side * 0.5 * p.rho * p.boat_area_side * p.boat_l * 5.0 * sgn_vr;
    const double M_rudder =
        v_x * v_x * p.c_r_side * 0.5 * p.rho * p.rudder_area * sin_rud * (p.boat_b / 2.0) * sgn_vx;
    const double a_r = (-M_hull + M_rudder) / (p.boat_I + p.boat_Iz);
    v_r = first ? 0.0 : a_r * p.dt + v_r;  // boat_env.py:172,209
    // get_kinematics  boat_env.py:283-306
    const double v = sqrt(v_x * v_x + v_y * v_y);
    const double drift = atan2(v_x, v_y);
    const double s_r = v_r * p.dt + d[D_SR];
    const double dir = drift - s_r;
    double sin_dir, cos_dir;
    sincos(dir, &sin_dir, &cos_dir);
    const double s_x = sin_dir * v * p.dt + d[D_SX];
    const double s_y = cos_dir * v * p.dt + d[D_SY];
    const double fuel = p.fuel - (double)(index + 1);  // boat_env.py:70

    // exponential_reward  reward_functions.py:42-57 with y_a = 0.03, y_b = 3.4 (boat_env.py:16-22)
    const double ay = fabs(s_y);
    double r = 0.0 - (ay / p.track_width) / (1.0 + exp((-0.03 / 3.4) * (ay - (p.track_width * 0.2))));
    // termination cascade  boat_env.py:84-105
    code = BOATENV_TERM_NONE;
    if (s_x >= p.goal_line) { code = BOATENV_TERM_REACHED_GOAL; r += 1000.0; }
    else if (ay > p.track_width + p.oob_offset || s_x < 0.0) code = BOATENV_TERM_OUT_OF_BOUNDS;
    else if (fuel < 0.0) code = BOATENV_TERM_OUT_OF_FUEL;
    else if (index + 1 >= c.timeout_steps) code = BOATENV_TERM_TIMEOUT;
    else if (rudder > PI / 3.0 || rudder < -PI / 3.0) code = BOATENV_TERM_RUDDER_BROKEN;
    if (rudder > PI / 4.0 || rudder < -PI / 4.0) r -= fabs(rudder) * 100.0;  // :107-108
    if (fabs(s_r) > PI / 2.0) r -= 1.0;                                       // :110-111
    reward = r;

    acc[0] = a_x; acc[1] = a_y; acc[2] = a_r;
    d[D_VX] = v_x; d[D_VY] = v_y; d[D_VR] = v_r; d[D_RUDDER] = rudder;
    d[D_SX] = s_x; d[D_SY] = s_y; d[D_SR] = s_r; d[D_RET] += r;  // :113
}

template <int WK, bool SAT>
__device__ __forceinline__ void substep(const DevCfg &c, float (&d)[D_COUNT], Fx<float> &fx, int index, float action,
                                        float w, float th, float (&acc)[3], float &reward, int &code) {
    // fp32 production mode: config products folded on the host (FastConsts); the
    // sqrt/atan2/sin/cos chain of get_kinematics collapses algebraically:
    //   sin(atan2(vx,vy) - s_r) * |v| = vx cos(s_r) - vy sin(s_r)
    //   cos(atan2(vx,vy) - s_r) * |v| = vy cos(s_r) + vx sin(s_r)
    // Everything a threshold is applied to after ACCUMULATION is carried exactly (struct Fx, common.cuh):
    // the rudder in 2^-42 rad units (boat_env.py:72-73 is a sum of action / 10 terms), s_x and s_y in fixed point.
    const FastConsts &f = c.f;
    const bool first = (index == 0);
    // The fp32 VIEW of the new angle (what the dynamics and the observation use) is one FFMA behind the action:
    // previous exact angle rounded to fp32, plus action / 10.  The EXACT update runs beside it on the fp64 pipe
    // and only feeds the threshold tests at the end of the sub-step, so it is off the critical path
    // action -> sin(rudder) -> a_y, a_r -> v -> s_r -> sincos -> positions.
    float rudder = fx.rudder_view();
    if (c.test_mode == 0) {  // rudder += action / 10 (boat_env.py:72-73); |action| is nominally <= 1 and not clipped
        // any |action| >= 21 breaks the rudder from any unbroken state, so clamping at 64 changes no outcome; the
        // increment is rounded to a whole number of 2^-42 rad with the 1.5 * 2^52 trick (exact for |x| < 2^51)
        const float a_c = fminf(fmaxf(action, -64.0f), 64.0f);
        rudder = fmaf(a_c, f.tenth, rudder);
        const double t = fma((double)a_c, 4398046511104.0 / 10.0, 6755399441055744.0);
        fx.rud += t - 6755399441055744.0;
    }
    // |rud| > threshold on the bit pattern (non-negative doubles order like their 64-bit patterns): integer
    // compares against immediates, no 64-bit constants to materialise inside the K loop
    const unsigned long long rud_abs = (unsigned long long)__double_as_longlong(fx.rud) & 0x7fffffffffffffffull;
    const bool rud_broken = rud_abs > kRudPi3Bits, rud_penalty = rud_abs > kRudPi4Bits;
    float v_x = d[D_VX], v_y = d[D_VY], v_r = d[D_VR];

    float F_Wx = 0.0f, F_Wy = 0.0f;
    if (WK == WIND_CONST) { F_Wx = f.fwx_c; F_Wy = f.fwy_c; }
    if (WK == WIND_VEL_CURVE) {
        const float ww = w * fabsf(w);
        F_Wx = ww * f.kwx * f.cos_dir;
        F_Wy = ww * f.kwy * f.sin_dir;
    }
    if (WK == WIND_ANGLE_RECT) {  // th carries the (renormalised) rect source curve
        const bool hi = th > 0.25f;  // wind.py:95: value <= middle/2 -> 0 else 1
        F_Wx = hi ? f.fwx_hi : f.fwx_lo;
        F_Wy = hi ? f.fwy_hi : f.fwy_lo;
    }
    if (WK == WIND_BOTH) {
        float st, ct;
        fast_sincosf(th, st, ct);
        const float ww = w * fabsf(w);
        F_Wx = ww * f.kwx * ct;
        F_Wy = ww * f.kwy * st;
    }
    const float a_x = (fmaf(-f.kdx * v_x, v_x, f.kT * fast_sinf(f.kJ * v_x)) + f.cxy * v_y * v_r + F_Wx) * f.inv_mx;
    v_x = first ? 3.0f : fmaf(a_x, f.dt, v_x);
    const float sin_rud = fast_sinf(rudder);
    const float a_y =
        (fmaf(-f.kdy * v_y, fabsf(v_y), sin_rud * f.kru * v_x * v_x) + f.cyx * v_x * v_r + F_Wy) * f.inv_my;
    v_y = first ? 0.0f : fmaf(a_y, f.dt, v_y);
    const float a_r = fmaf(-f.kh * v_r, fabsf(v_r), f.kmr * v_x * fabsf(v_x) * sin_rud) * f.inv_I;
    v_r = first ? 0.0f : fmaf(a_r, f.dt, v_r);
    const float s_r = fmaf(v_r, f.dt, d[D_SR]);
    float sr, cr;
    fast_sincosf(s_r, sr, cr);
    fx.sx = add_fixed<SAT>(fx.sx, fixed_increment(fmaf(v_x, cr, -v_y * sr), f.sx_k));
    fx.sy = add_fixed<SAT>(fx.sy, fixed_increment(fmaf(v_y, cr, v_x * sr), f.sy_k));
    const float s_y = (float)fx.sy * f.sy_inv;   // the float view of s_x is only needed for the observation (stage_obs)
    const float ay = fabsf(s_y);
    float r = -__fdividef(ay * f.rew_inv_W, 1.0f + __expf(f.rew_k * (ay - f.rew_y0)));
    // termination cascade boat_env.py:84-105, lowest priority first (later selects override);
    // fuel < 0 (:94) and t_max <= t (:98) depend on the step count only: integer thresholds
    const float ar = fabsf(rudder);
    const bool goal = fx.sx >= f.sx_goal;
    code = rud_broken ? BOATENV_TERM_RUDDER_BROKEN : BOATENV_TERM_NONE;
    code = (index + 1 >= c.timeout_steps) ? BOATENV_TERM_TIMEOUT : code;
    code = (index + 1 >= c.fuel_steps) ? BOATENV_TERM_OUT_OF_FUEL : code;
    // abs(s_y) > W + offset or s_x < 0 (:90): |sy| > sy_oob <=> (unsigned)(sy + sy_oob) > 2 sy_oob; sign bit of sx
    code = ((unsigned)fx.sy + (unsigned)f.sy_oob > f.sy_oob2 || fx.sx < 0) ? BOATENV_TERM_OUT_OF_BOUNDS : code;
    code = goal ? BOATENV_TERM_REACHED_GOAL : code;
    r += goal ? 1000.0f : 0.0f;
    if (rud_penalty) r = fmaf(-100.0f, ar, r);
    if (fabsf(s_r) > f.pi2) r -= 1.0f;
    reward = r;

    acc[0] = a_x; acc[1] = a_y; acc[2] = a_r;
    d[D_VX] = v_x; d[D_VY] = v_y; d[D_VR] = v_r; d[D_RUDDER] = rudder;
    d[D_SY] = s_y; d[D_SR] = s_r; d[D_RET] += r;
}

// The wind sample wind[index] of an env (wind.py:26-63, boat_env.py:230-236) from its carried piece coefficients
// wa / wb; j, r: the spline piece of the sample and its remainder (piece_of), for next_sample_in_next_piece.
template <typename T, int WK>
__device__ __forceinline__ void wind_sample(const DevCfg &c, int index, const T (&wa)[4], const T (&wb)[4], T inv_Lm1,
                                            T &w, T &th, int &j, int &r) {
    constexpr bool kCurves = (WK == WIND_VEL_CURVE || WK == WIND_ANGLE_RECT || WK == WIND_BOTH);
    w = (T)0; th = (T)0;
    j = 0; r = 0;
    if (kCurves) {
        piece_of(c, min(index, c.L - 1), j, r);
        const T s = (T)r * inv_Lm1;
        const T va = ((wa[3] * s + wa[2]) * s + wa[1]) * s + wa[0];
        if (WK == WIND_ANGLE_RECT) {
            if (sizeof(T) == 8) {  // wind.py:57-58,95: (value<=0.25 ? 0 : 1)*pi + pi/2
                w = (T)c.p.max_velocity;
                th = (T)(((double)va <= 0.25 ? 0.0 : 1.0) * 3.14159265358979323846 + 3.14159265358979323846 / 2.0);
            } else {
                th = va;  // the fp32 path thresholds inside substep()
            }
        } else {
            w = va;
            th = (T)c.direction_rad;
        }
        if (WK == WIND_BOTH) th = ((wb[3] * s + wb[2]) * s + wb[1]) * s + wb[0];
    }
    if (WK == WIND_CONST) { w = (T)c.p.max_velocity; th = (T)c.direction_rad; }
}

// Does wind[index + 1] (the next sub-step's sample) live in the next spline piece, given piece j and remainder r of
// wind[index]?  Then the env needs the next piece's coefficients (wind_setup_*) before its next sub-step.
__device__ __forceinline__ bool next_sample_in_next_piece(const DevCfg &c, int j, int r) {
    return r + c.npieces >= c.Lm1 && j + 1 <= c.npieces - 1;
}

// Statistics of an episode that ended with termination `code` and return `ret` (info dict, boat_env.py:24-32,87-113),
// counted in fp64 into the counter row of state block `blk`: sparse events -> per-env REDs.
template <typename T>
__device__ __forceinline__ void count_episode_end(const DevCfg &c, int blk, int code, T ret) {
    double *cnt = c.counters + (blk & (kCounterSlots - 1)) * 32;
    const double r = (double)ret;
    atomicAdd(cnt + (code - 1), 1.0);
    atomicAdd(cnt + 5, 1.0);
    atomicAdd(cnt + 6, r);
    atomicAdd(cnt + 7, r * r);
}

// A NaN bit pattern that no arithmetic instruction produces (their NaNs are canonical): see the stage-refill vote.
__device__ __forceinline__ bool is_poison(float v) { return __float_as_uint(v) == 0x7fc00001u; }
__device__ __forceinline__ bool is_poison(double v) { return __double_as_longlong(v) == 0x7ff8000000000001ll; }

// return_state  boat_env.py:308-326: the 11 normalised observations of an env, written to
// its row of the warp's shared-memory staging tile.  `index` = Boat.index after the step.
__device__ __forceinline__ void stage_obs(const DevCfg &c, double *row, const double (&d)[D_COUNT], const Fx<double> &,
                                          const double (&acc)[3], int index) {
    const boatenv_params &p = c.p;
    const double PI = 3.14159265358979323846;
    row[0] = (d[D_SX] - 0.0) / (p.goal_line - 0.0);
    row[1] = d[D_VX] / 5.0;
    row[2] = acc[0] / 0.025;
    row[3] = (d[D_SY] - (-p.track_width)) / (p.track_width - (-p.track_width));
    row[4] = d[D_VY] / 2.0;
    row[5] = acc[1] / 0.37;
    row[6] = d[D_SR] / (2.0 * PI);
    row[7] = d[D_VR] / 8.5e-3;
    row[8] = acc[2] / 1.4e-5;
    row[9] = (d[D_RUDDER] - (-PI / 3.0)) / (PI / 3.0 - (-PI / 3.0));
    row[10] = (p.fuel - (double)index) / p.fuel;
}
__device__ __forceinline__ void stage_obs(const DevCfg &c, float *row, const float (&d)[D_COUNT], const Fx<float> &fx,
                                          const float (&acc)[3], int index) {
    const FastConsts &f = c.f;
    row[0] = (float)fx.sx * f.sx_obs;
    row[1] = d[D_VX] * f.inv_5;
    row[2] = acc[0] * f.inv_ax;
    row[3] = (d[D_SY] + f.W) * f.inv_2W;
    row[4] = d[D_VY] * f.inv_2;
    row[5] = acc[1] * f.inv_ay;
    row[6] = d[D_SR] * f.inv_2pi;
    row[7] = d[D_VR] * f.inv_vr;
    row[8] = acc[2] * f.inv_ar;
    row[9] = (d[D_RUDDER] + f.third_pi) * f.inv_rud;
    row[10] = (f.fuel0 - (float)index) * f.inv_fuel;
}

// The reset observation (boat_env.py:124 after Boat.__init__): all zeros except s_y,
// rudder (0.5) and fuel (1).
template <typename T>
__device__ __forceinline__ void stage_reset_obs(const DevCfg &c, T *row, T s_y0) {
#pragma unroll
    for (int k = 0; k < kObsDim; ++k) row[k] = (T)0;
    row[3] = (T)(((double)s_y0 + c.p.track_width) / (c.p.track_width + c.p.track_width));
    row[9] = (T)0.5;
    row[10] = (T)1;
}

// ---------------------------------------------------------------------------------
// TMA bulk-copy primitives (sm_90+/sm_100a PTX; the mbarrier ones are in common.cuh).  The copies are 1-D
// (cp.async.bulk, no tensor map): a warp's state block is contiguous in HBM.
// ---------------------------------------------------------------------------------
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
// global -> shared bulk copy, completion counted in bytes on `bar`.  Default L2 policy: an evict_first
// cache hint measured 3 % slower (the alternating sweep lets the tail of a launch hit L2 in the next one).
__device__ __forceinline__ void tma_load_1d(void *smem_dst, const void *gmem_src, uint32_t bytes, uint64_t *bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::
                     "r"(smem_u32(smem_dst)), "l"(gmem_src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
// shared -> global bulk copy (bulk async-group completion)
__device__ __forceinline__ void tma_store_1d(void *gmem_dst, const void *smem_src, uint32_t bytes) {
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(gmem_dst), "r"(smem_u32(smem_src)),
                 "r"(bytes) : "memory");
}
__device__ __forceinline__ void tma_store_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
// wait until the bulk stores of all committed groups have finished READING shared memory
__device__ __forceinline__ void tma_store_wait_read() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void tma_store_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
// Build-time switches.  BOAT_MINBLOCKS_F32 / BOAT_STAGES / BOAT_SETUP_WARPS / BOAT_CTA_THREADS are tuning
// knobs (defaults = measured optimum); the BOAT_DEBUG_* macros remove parts of the kernel for the
// ablation measurements quoted in DESIGN.md section 4 and are never defined in a product build.
#ifndef BOAT_MINBLOCKS_F32
#define BOAT_MINBLOCKS_F32 2  // 256-thread CTAs per SM the fp32 kernel is register-budgeted for
#endif
#ifndef BOAT_STAGES
#define BOAT_STAGES 1         // state blocks in flight per warp beyond the one being computed (TMA pipeline depth)
#endif
#ifndef BOAT_MINBLOCKS_F64
#define BOAT_MINBLOCKS_F64 3  // the same for the K = 1 fp64 validation kernels: they are latency bound (dependent
#endif                        // DFMA chains), 3 CTAs per SM at 56-80 registers beat 1 CTA at 134 by 7-24 %
template <typename T, bool KMULTI> struct StepTuning;
template <bool KMULTI> struct StepTuning<float, KMULTI> { static constexpr int kMinBlocks = BOAT_MINBLOCKS_F32; };
template <> struct StepTuning<double, false> { static constexpr int kMinBlocks = BOAT_MINBLOCKS_F64; };
template <> struct StepTuning<double, true> { static constexpr int kMinBlocks = 1; };  // 230 registers live across the K loop
constexpr int kStages = BOAT_STAGES;

#ifndef BOAT_SETUP_WARPS
#define BOAT_SETUP_WARPS 2    // dedicated wind-setup warps per CTA in the K = 1 kernels of experiments 4-6 (round-2 A/B on one
                              // box, 16 M envs of exp 6: 1 warp 0.566 ms, 2 warps 0.4696, 4 warps 0.4750; profiles/jobs/r02y.sh)
#endif
// K = 1 kernels of the random-wind experiments run warp-specialised: 8 step warps stream the state
// and push their (rare) wind-setup requests into a shared-memory queue, kSetup extra warps serve it.
template <int WK, bool KMULTI>
__host__ __device__ constexpr int setup_warps() {
    return (!KMULTI && (WK == WIND_VEL_CURVE || WK == WIND_ANGLE_RECT || WK == WIND_BOTH)) ? BOAT_SETUP_WARPS : 0;
}

// Bounded multi-producer / multi-consumer ring in shared memory (ticket + per-slot sequence number).
// Producers: lanes of the step warps (one request per env that needs new wind coefficients);
// consumers: the setup warps.  A full ring blocks the producer, consumers always make progress.
constexpr int kQueueSlots = 64;
struct SetupRequest { int env; uint32_t episode; int index_next; int pad; };
struct SetupQueue {
    unsigned tail, head, producers_done, pad;
    unsigned seq[kQueueSlots];
    SetupRequest slot[kQueueSlots];
};

__device__ __forceinline__ void queue_push(SetupQueue *q, const SetupRequest &r) {
    const unsigned ticket = atomicAdd(&q->tail, 1u);
    const unsigned s = ticket % kQueueSlots;
    volatile unsigned *seq = q->seq + s;
    while (*seq != ticket) __nanosleep(64);      // slot still holds an unconsumed older request
    q->slot[s] = r;
    __threadfence_block();
    *seq = ticket + 1u;                           // publish
}

// Called by lane 0 of a setup warp.  Returns false when every producer has finished and the ring is drained.
__device__ __forceinline__ bool queue_pop(SetupQueue *q, int n_producers, SetupRequest &r) {
    const unsigned ticket = atomicAdd(&q->head, 1u);
    const unsigned s = ticket % kQueueSlots;
    volatile unsigned *seq = q->seq + s;
    volatile unsigned *done = &q->producers_done, *tail = &q->tail;
    // Nobody waits for the coefficients before the NEXT launch, so an idle consumer sleeps long (up to
    // ~1 us per poll) instead of burning issue slots and power next to the streaming warps.
    unsigned backoff = 128u;
    while (*seq != ticket + 1u) {
        if (*done == (unsigned)n_producers && (int)(ticket - *tail) >= 0) return false;
        __nanosleep(backoff);
        backoff = min(backoff * 2u, 1024u);
    }
    __threadfence_block();
    r = q->slot[s];
    __threadfence_block();
    *seq = ticket + kQueueSlots;                  // free the slot for its next ticket
    return true;
}

// Dynamic shared memory of a CTA: per step warp the TMA stages, the observation staging tile,
// (inline slow path only) the scratch, the stage barriers; then the request queue and the
// scratch of the setup warps.
template <typename T>
struct WarpSmem {
    int tile_off, prev_off, scratch_off, bar_off, bytes;
    // prev_tiles: 2 when the launch also stores the transition (fused agent.remember): double-buffered
    // TMA staging of the PREVIOUS observation tile, which leaves again as the ring's `state` rows
    __host__ __device__ WarpSmem(int block_bytes, int scratch_dbl, int prev_tiles) {
        const int tile_bytes = 32 * kObsDim * (int)sizeof(T);  // 1408 / 2816: a multiple of 128
        tile_off = kStages * block_bytes;
        prev_off = tile_off + tile_bytes;
        scratch_off = prev_off + prev_tiles * tile_bytes;
        bar_off = scratch_off + scratch_dbl * 8;
        bytes = (bar_off + (kStages + 2) * 8 + 127) / 128 * 128;
    }
};
template <typename T>
struct CtaSmem {
    WarpSmem<T> warp;
    int queue_off, setup_scratch_off, setup_scratch_bytes, kq_off, bytes;
    __host__ __device__ CtaSmem(int block_bytes, int ncurves, int npieces, int n_setup, bool fused_store)
        : warp(block_bytes, n_setup > 0 ? 0 : scratch_doubles(ncurves, npieces), fused_store ? 2 : 0) {
        queue_off = kWarpsPerCta * warp.bytes;
        setup_scratch_off = queue_off + (n_setup > 0 ? (int)sizeof(SetupQueue) : 0);
        setup_scratch_bytes = (scratch_doubles(ncurves, npieces) * 8 + 127) / 128 * 128;
        kq_off = setup_scratch_off + n_setup * setup_scratch_bytes;  // two counters of the K > 1 episode-end queue
        bytes = kq_off + 16;
    }
};

// Persistent kernel, one thread per env, every warp self-contained: warp w walks the 32-env
// state blocks w, w + W, w + 2W, ... (W = warps in the grid).  Its lane 0 keeps kStages TMA
// bulk copies of upcoming blocks in flight (mbarrier-completed), so the HBM latency is hidden
// by the pipeline instead of by occupancy; lanes read their state from shared memory, run the
// K sub-steps in registers, write the state back with coalesced 128-bit stores and the
// [32][11] observation tile with one bulk store.  No CTA-wide barrier anywhere.
//
// KMULTI = false is the gym-faithful one-sub-step-per-launch instantiation: the state is
// written back right after the sub-step and the (rare) slow path patches the affected envs
// in global memory, so that almost nothing is live in registers across the slow path.
template <typename T, int WK, bool KMULTI>
__global__ void __launch_bounds__(kTile + 32 * setup_warps<WK, KMULTI>(), StepTuning<T, KMULTI>::kMinBlocks)
boat_step_kernel(const __grid_constant__ DevCfg c, const __grid_constant__ StepArgs a) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    constexpr bool kCurves = (WK == WIND_VEL_CURVE || WK == WIND_ANGLE_RECT || WK == WIND_BOTH);
    constexpr int kSetup = setup_warps<WK, KMULTI>();
    constexpr int kTileBytes = 32 * kObsDim * (int)sizeof(T);
    const unsigned FULL = 0xffffffffu;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int bb = c.block_bytes;

    const bool fused_store = !KMULTI && a.rp.state != nullptr;
    const CtaSmem<T> cta(bb, c.ncurves, c.npieces, kSetup, fused_store);
    const WarpSmem<T> &lay = cta.warp;
    SetupQueue *queue = reinterpret_cast<SetupQueue *>(smem_raw + cta.queue_off);
    if (kSetup > 0) {
        for (int t = threadIdx.x; t < kQueueSlots; t += blockDim.x) queue->seq[t] = (unsigned)t;
        if (threadIdx.x == 0) { queue->tail = 0u; queue->head = 0u; queue->producers_done = 0u; }
        __syncthreads();  // the only CTA-wide barrier: once, before any work
        if (warp >= kWarpsPerCta) {
            // ===== setup warps: serve wind-setup requests until the step warps are done and the ring is empty =====
            double *scr = reinterpret_cast<double *>(smem_raw + cta.setup_scratch_off +
                                                     (warp - kWarpsPerCta) * cta.setup_scratch_bytes);
            for (;;) {
                SetupRequest r;
                r.env = -1; r.episode = 0u; r.index_next = 0; r.pad = 0;
                if (lane == 0 && !queue_pop(queue, kWarpsPerCta, r)) r.env = -1;
                const int env = __shfl_sync(FULL, r.env, 0);
                if (env < 0) break;
                const uint32_t epi = __shfl_sync(FULL, r.episode, 0);
                const int idx_next = __shfl_sync(FULL, r.index_next, 0);
#ifdef BOAT_DEBUG_SKIP_SETUP  // experiment only: requests are popped and dropped
                continue;
#endif
                wind_setup_warp(c, (long long)env, epi, idx_next, scr);
                if (lane < 2 && (lane == 0 || WK == WIND_BOTH)) {  // lane 0: first curve, lane 1: second curve
                    T w4[4];
#pragma unroll
                    for (int m = 0; m < 4; ++m) w4[m] = (T)scr[lane * 4 + m];
                    char *gb = c.state + (size_t)(env >> 5) * (size_t)bb;
                    store_vecs<T, 4>(gb + (lane ? c.off_wb : c.off_wa), env & 31, w4);
                }
                __syncwarp();
            }
            return;
        }
    }
    // K > 1 kernels of the random-wind experiments: finished episodes are deferred to a follow-up kernel
    const bool kq_on = KMULTI && kCurves && a.kq_entries != nullptr;
    unsigned *kq_cnt = reinterpret_cast<unsigned *>(smem_raw + cta.kq_off);  // [0] entries pushed, [1] warps finished
    if (KMULTI && kCurves) {
        if (threadIdx.x == 0) { kq_cnt[0] = 0u; kq_cnt[1] = 0u; }
        __syncthreads();
    }
    auto kq_finish = [&]() {  // the last step warp of the CTA publishes the region's entry count
        __syncwarp();
        if (lane == 0) {
            __threadfence();
            if (atomicAdd(kq_cnt + 1, 1u) == (unsigned)(kWarpsPerCta - 1))
                a.kq_counts[blockIdx.x] = *reinterpret_cast<volatile unsigned *>(kq_cnt);
        }
    };
    unsigned char *wbase = smem_raw + (size_t)warp * lay.bytes;
    unsigned char *stage_base = wbase;                                  // kStages * bb   (16-byte aligned)
    T *tile = reinterpret_cast<T *>(wbase + lay.tile_off);              // [32][11]
    double *scratch = reinterpret_cast<double *>(wbase + lay.scratch_off);
    uint64_t *full = reinterpret_cast<uint64_t *>(wbase + lay.bar_off);
    uint64_t *pfull = full + kStages;                                   // [2] barriers of the previous-obs tiles
    unsigned char *prev_base = wbase + lay.prev_off;                    // [2][kTileBytes]  (fused store only)
    T *row = tile + lane * kObsDim;

    // env indices of one handle fit 32 bits (checked at create).  The warp walks SEQUENCE numbers
    // seq, seq + W, ...; block = seq on even launches and (last - seq) on odd ones: consecutive
    // launches sweep the state in opposite directions, so the blocks written last (still dirty in
    // the 126 MB L2) are the first ones the next launch reads.
    const int n_end = (int)a.env_end, blk_end = (n_end + 31) >> 5;
    const int wstride = (int)gridDim.x * kWarpsPerCta;
    const int blk_first = (int)(a.env_begin >> 5), blk_last = blk_end - 1;
    const bool rev = a.reverse != 0;
    int seq = blk_first + (int)blockIdx.x * kWarpsPerCta + warp;  // CTA-major: 8 consecutive blocks per CTA (warp-major measured 2 % slower)
    if (seq >= blk_end) {
        if (kSetup > 0 && lane == 0) atomicAdd(&queue->producers_done, 1u);
        if (kq_on) kq_finish();
        return;
    }
    auto block_of = [&](int q) { return rev ? (blk_last - (q - blk_first)) : q; };

    if (lane == 0) {
#pragma unroll
        for (int s = 0; s < kStages; ++s) mbar_init(full + s, 1);
        mbar_init(pfull, 1);
        mbar_init(pfull + 1, 1);
        mbar_fence_init();
    }
    __syncwarp();
    // fused store: the tile of observations the PREVIOUS step wrote for a (full) block is fetched one block
    // ahead by a bulk copy of its own and leaves again as the ring's `state` rows without touching registers
    const T *prev_obs = reinterpret_cast<const T *>(a.obs_in);
    auto prev_prefetch = [&](int q, int buf) {  // lane 0 only
        const int b = block_of(q);
        if (b * 32 + 32 <= n_end) {
            mbar_expect_tx(pfull + buf, (uint32_t)kTileBytes);
            tma_load_1d(prev_base + buf * kTileBytes, prev_obs + (size_t)b * (32 * kObsDim), (uint32_t)kTileBytes, pfull + buf);
        }
    };
    // K = 1 (HBM bound): the bulk copy stops before the episode row, which only an ending episode touches.
    // K > 1 (issue bound): the whole block, the slow path then finds the episode number in shared memory.
    const uint32_t tma_bytes = KMULTI ? (uint32_t)bb : (uint32_t)c.off_epi;
    if (lane == 0) {  // prologue: fill the pipeline
#pragma unroll
        for (int s = 0; s < kStages; ++s) {
            const int q = seq + s * wstride;
            if (q < blk_end) {
                mbar_expect_tx(full + s, tma_bytes);
                tma_load_1d(stage_base + s * bb, c.state + (size_t)block_of(q) * (size_t)bb, tma_bytes, full + s);
            }
        }
        if (fused_store) prev_prefetch(seq, 0);
    }
    int pbuf = 0;            // previous-obs buffer of the current block
    uint32_t pphase = 0u;    // bit b: parity the next wait on pfull[b] expects
    const T *act = reinterpret_cast<const T *>(a.actions);
    const T inv_Lm1 = sizeof(T) == 8 ? (T)c.inv_Lm1 : (T)c.f.inv_Lm1;
    const bool auto_reset = (a.flags & BOATENV_AUTO_RESET) != 0;
    const int ksteps = KMULTI ? a.ksteps : 1;
    T action_next = __ldcs(act + min(block_of(seq) * 32 + lane, n_end - 1));
    int stage = 0;
    uint32_t parity = 0;
    bool tile_in_flight = false;  // a bulk store of `tile` may still be reading it

    for (; seq < blk_end; seq += wstride) {
        const int blk = block_of(seq);
        const int i = blk * 32 + lane;
        const bool active = i < n_end;  // inactive lanes are the padding of the last block (no stores)
        T action = action_next;
        if (seq + wstride < blk_end) action_next = __ldcs(act + min(block_of(seq + wstride) * 32 + lane, n_end - 1));

        // ---- state: wait for the TMA copy of this block, read it from shared memory ----
        const unsigned char *sb = stage_base + stage * bb;
        mbar_wait(full + stage, parity);
        T d[D_COUNT];
        T wa[4] = {0, 0, 0, 0}, wb[4] = {0, 0, 0, 0};
        load_vecs<T, D_COUNT>(reinterpret_cast<const char *>(sb), lane, d);
        if (kCurves) load_vecs<T, 4>(reinterpret_cast<const char *>(sb) + c.off_wa, lane, wa);
        if (WK == WIND_BOTH) load_vecs<T, 4>(reinterpret_cast<const char *>(sb) + c.off_wb, lane, wb);
        const uint32_t epi_s = KMULTI ? reinterpret_cast<const uint32_t *>(sb + c.off_epi)[lane] : 0u;
        const uint32_t ixw = reinterpret_cast<const uint32_t *>(sb + c.off_idx)[lane];
        int index;
        Fx<T> fx;                     // fp32 mode: exact rudder / position carriers decoded from their slots
        fx.load(c, d, ixw, index);
        uint32_t episode_k = epi_s;   // K > 1 only: this launch's view of the env's episode number
        // The refill below overwrites this stage, so it must not be issued before EVERY lane's loads of the stage
        // have returned (issuing them is not enough: a refill served from L2 can land within a few hundred
        // cycles).  The vote consumes a register of each of the loads above in every lane -- the compiler is free
        // to order them, so all of them take part -- and lane 0's block number depends on the vote: a true
        // dependency for the hardware scoreboard.  The predicate is never true: a step index never reaches
        // 2^20 - 1 (L <= 2^20 - 64, checked at create), no arithmetic produces the poison NaN, and the inspected
        // registers are genuine floating-point slots (fp32 mode: v_r and s_r; the rudder / position slots hold
        // fixed-point bit patterns and are not looked at).  The padding lanes of a ragged last block read the
        // 0xFF fill, whose index field IS the pattern: they are excluded (their loads still complete before the
        // vote, a lane's instructions issue in order).
        bool never = ((ixw & kIndexMask) == kIndexMask && active) || (KMULTI && epi_s == 0x7fc00001u && (ixw & kIndexMask) == kIndexMask - 1u);
        constexpr int W = VecOf<T>::W;   // one register of every 16-byte vector load
        constexpr int kProbe = sizeof(T) == 4 ? 2 : 0;
#pragma unroll
        for (int v = 0; v < D_COUNT / W; ++v) never |= is_poison(d[v * W + kProbe]);
#pragma unroll
        for (int v = 0; v < 4 / W; ++v) {
            if (kCurves) never |= is_poison(wa[v * W]);
            if (WK == WIND_BOTH) never |= is_poison(wb[v * W]);
        }
#ifdef BOAT_DEBUG_NO_REFILL_VOTE  // ablation only (profiles/r02_refill_vote_ablation.txt): the benchmark-regime parity tests must fail
        const unsigned never_mask = 0u;
#else
        const unsigned never_mask = __ballot_sync(FULL, never);
#endif
        if (lane == 0) {
            // The stage is consumed: refill it kStages blocks ahead.
            const int q = seq + kStages * wstride + (never_mask != 0u ? 1 : 0);
            if (q < blk_end) {
                mbar_expect_tx(full + stage, tma_bytes);
                tma_load_1d(stage_base + stage * bb, c.state + (size_t)block_of(q) * (size_t)bb, tma_bytes, full + stage);
            }
        }
        if (++stage == kStages) { stage = 0; parity ^= 1u; }

        T rsum = (T)0;
        int code = BOATENV_TERM_NONE, nsteps = 0;
        bool alive = true, wind_dirty = false;
        if (tile_in_flight) {  // the previous block's bulk stores must be done reading `tile` (and its previous-obs buffer)
            if (lane == 0) tma_store_wait_read();
            __syncwarp();
            tile_in_flight = false;
        }
        if (fused_store && lane == 0 && seq + wstride < blk_end) prev_prefetch(seq + wstride, pbuf ^ 1);
        bool ring_in_flight = false;
        char *gb = c.state + (size_t)blk * (size_t)bb;

        // the carried scalars + step index of this lane's env -> its block in HBM (fp32 mode: d[] keeps the float
        // views of rudder / s_x / s_y that stage_obs() reads; a copy gets the fixed-point bit patterns)
        auto store_dyn = [&]() {
            T dd[D_COUNT];
#pragma unroll
            for (int q = 0; q < D_COUNT; ++q) dd[q] = d[q];
            const uint32_t index_word = fx.pack(dd, index);
            store_vecs<T, D_COUNT>(gb, lane, dd);
            st_state(reinterpret_cast<uint32_t *>(gb + c.off_idx) + lane, index_word);
        };
        // state + per-env outputs of this launch (K = 1: right after the sub-step; K > 1: after the loop)
        auto store_results = [&]() {
            if (active) {
#ifndef BOAT_DEBUG_SKIP_STATE
                store_dyn();
#endif
                if (KMULTI && wind_dirty) {  // wind coefficients change only on the slow path
                    if (kCurves) store_vecs<T, 4>(gb + c.off_wa, lane, wa);
                    if (WK == WIND_BOTH) store_vecs<T, 4>(gb + c.off_wb, lane, wb);
                }
#ifndef BOAT_DEBUG_SKIP_SMALL
                __stcs(reinterpret_cast<T *>(a.reward_out) + i, rsum);
                if (a.done_out) a.done_out[i] = (code != BOATENV_TERM_NONE) ? 1 : 0;   // NULL: the caller reads done = (term != 0)
                if (a.term_out) a.term_out[i] = (uint8_t)code;
#endif
                if (KMULTI) {
                    if (a.steps_out) a.steps_out[i] = nsteps;
                }
            }
        };

        // per-sub-step actions ([K][N] layout): the action of sub-step k + 1 is fetched while sub-step k computes
        const bool per_substep = KMULTI && a.action_stride != 0;
        // the pointer walks one row of the [K][N] action matrix per sub-step (no 64-bit multiply in the loop);
        // with a repeated action (stride 0) it stays where it is and re-reads the same, cached, element
        const T *act_next = act + min(i, n_end - 1) + (size_t)a.action_stride;
        T action_k1 = action;
        if (per_substep && ksteps > 1) action_k1 = __ldcs(act_next);
        for (int k = 0; k < ksteps; ++k) {
            if (KMULTI && k > 0) {
                action = action_k1;
                act_next += (size_t)a.action_stride;
                if (per_substep && k + 1 < ksteps) action_k1 = __ldcs(act_next);
            }
            bool need_setup = false;
            if (alive) {
                // ---- wind sample wind[index] from the carried piece coefficients ----
                T w, th;
                int j, r;
                wind_sample<T, WK>(c, index, wa, wb, inv_Lm1, w, th, j, r);

                T rew, acc[3];
#ifdef BOAT_DEBUG_NOCOMPUTE  // memory-pattern experiment only: stream the state through untouched
                acc[0] = acc[1] = acc[2] = w + th; rew = action; code = BOATENV_TERM_NONE;
#else
                substep<WK, !KMULTI>(c, d, fx, index, action, w, th, acc, rew, code);
#endif
                rsum += rew;
                ++nsteps;
                index += 1;
                if (code != BOATENV_TERM_NONE || k == ksteps - 1) stage_obs(c, row, d, fx, acc, index);
                if (code != BOATENV_TERM_NONE) {
                    alive = false;
                    need_setup = true;  // statistics, and the reset if AUTO_RESET
                } else if (kCurves) {
                    // does wind[index] (the next sub-step) live in the next spline piece?
                    if (next_sample_in_next_piece(c, j, r)) need_setup = true;
                }
            }
            if (!KMULTI) store_results();
            if (!KMULTI && a.rp.state) {
                // ---- fused agent.remember (main.py:83-88, buffer.py:13-22): the transition leaves while the
                // tile still holds the TERMINAL observations (a reset below overwrites the rows of finished
                // envs).  The 32 ring slots of a warp are contiguous (mod mem_size).
                __syncwarp();
                const int rows_w = min(32, n_end - blk * 32);
                long long slot0 = a.rp.base_slot + (long long)blk * 32;
                if (slot0 >= a.rp.mem_size) slot0 -= a.rp.mem_size;
                const T *prev = reinterpret_cast<const T *>(a.obs_in) + (size_t)blk * (32 * kObsDim);
                T *ring_s = reinterpret_cast<T *>(a.rp.state) + slot0 * kObsDim;
                T *ring_n = reinterpret_cast<T *>(a.rp.new_state) + slot0 * kObsDim;
                const bool bulk = rows_w == 32 && slot0 + 32 <= a.rp.mem_size &&
                                  ((reinterpret_cast<uintptr_t>(ring_s) | reinterpret_cast<uintptr_t>(ring_n)) & 15u) == 0;
                const T *prev_tile = reinterpret_cast<const T *>(prev_base + pbuf * kTileBytes);
                if (rows_w == 32) {  // a full block: its previous observations were prefetched into prev_tile
                    mbar_wait(pfull + pbuf, (pphase >> pbuf) & 1u);
                    pphase ^= 1u << pbuf;
                }
                if (bulk) {  // s' = the staged tile, s = the prefetched previous tile: two bulk stores, no registers
                    fence_proxy_async_smem();
                    __syncwarp();
                    if (lane == 0) {
                        tma_store_1d(ring_s, prev_tile, kTileBytes);
                        tma_store_1d(ring_n, tile, kTileBytes);
                        tma_store_commit();
                    }
                    ring_in_flight = true;
                } else {  // ragged last block, ring wrap inside the block or unaligned ring: element-wise
                    const T *src = rows_w == 32 ? prev_tile : prev;
                    for (int e = lane; e < rows_w * kObsDim; e += 32) {
                        const int rr = e / kObsDim, q = e - rr * kObsDim;
                        long long slot = a.rp.base_slot + (long long)blk * 32 + rr;
                        if (slot >= a.rp.mem_size) slot -= a.rp.mem_size;
                        reinterpret_cast<T *>(a.rp.state)[slot * kObsDim + q] = src[e];
                        reinterpret_cast<T *>(a.rp.new_state)[slot * kObsDim + q] = tile[e];
                    }
                }
                if (active) {
                    long long slot = a.rp.base_slot + i;
                    if (slot >= a.rp.mem_size) slot -= a.rp.mem_size;
                    reinterpret_cast<T *>(a.rp.action)[slot] = action;
                    reinterpret_cast<T *>(a.rp.reward)[slot] = rsum;
                    a.rp.terminal[slot] = a.rp.done_flag_mode ? (code == BOATENV_TERM_REACHED_GOAL) : (code != BOATENV_TERM_NONE);
                }
            }
            // ---- slow path: the warp serves its lanes one at a time ----
            if (__ballot_sync(FULL, need_setup && active)) {
                if (ring_in_flight) {  // the bulk store of s' must have read the tile before rows are reset
                    if (lane == 0) tma_store_wait_read();
                    __syncwarp();
                    ring_in_flight = false;
                }
                const bool is_done = need_setup && active && code != BOATENV_TERM_NONE;
                // the episode number lives outside the streamed part of the block: fetched only here, written only
                // when an episode ends
                uint32_t *epi_g = reinterpret_cast<uint32_t *>(gb + c.off_epi) + lane;
                uint32_t episode = KMULTI ? episode_k : ((need_setup && active) ? *epi_g : 0u);
                if (is_done) count_episode_end(c, blk, code, d[D_RET]);
                if (is_done) {  // the terminal observation leaves before a reset overwrites the row
                    if (a.final_obs_out) {
                        T *fo = reinterpret_cast<T *>(a.final_obs_out) + (size_t)i * kObsDim;
#pragma unroll
                        for (int q = 0; q < kObsDim; ++q) fo[q] = row[q];
                    }
                }
                if (kSetup > 0) {
                    // warp-specialised K = 1 path: the env's own lane does the cheap part (Boat.__init__ state,
                    // reset observation) and hands the wind coefficients to the setup warps
                    if (need_setup && active && (!is_done || auto_reset)) {
                        SetupRequest rq;
                        rq.env = i;
                        rq.episode = episode + (is_done ? 1u : 0u);
                        rq.index_next = is_done ? 0 : index;
                        rq.pad = 0;
#ifndef BOAT_DEBUG_SKIP_PUSH
                        queue_push(queue, rq);
#endif
                        if (is_done) {  // Boat.__init__  boat_env.py:144-201
                            fx.start(c, d, 0);
                            index = 0;
                            stage_reset_obs<T>(c, row, (T)0);  // only experiment 2 starts off the centre line (:166-167)
                            store_dyn();
                            *epi_g = rq.episode;
                        }
                    }
                }
                bool deferred = false;
                if (kq_on && is_done && auto_reset) {
                    // K > 1: the env is frozen for the rest of the window, so its new wind coefficients are not
                    // needed before the next launch: queue (env, new episode) for boat_setup_queue_kernel and do
                    // only the cheap part of Boat.__init__ (boat_env.py:144-201) here
                    const unsigned pos = atomicAdd(kq_cnt, 1u);
                    a.kq_entries[(size_t)blockIdx.x * a.kq_cap + pos] = make_uint2((unsigned)i, episode + 1u);
                    fx.start(c, d, 0);
                    index = 0;
                    episode += 1u;
                    *epi_g = episode;
                    episode_k = episode;
                    wind_dirty = false;  // the old episode's coefficients are dead; the follow-up kernel writes the new ones
                    stage_reset_obs<T>(c, row, (T)0);  // only experiment 2 starts off the centre line (:166-167)
                    deferred = true;
                }
                unsigned todo = kSetup > 0 ? 0u
                                           : __ballot_sync(FULL, need_setup && active && !deferred && (!is_done || auto_reset));
                while (todo) {
                    const int src = __ffs(todo) - 1;
                    todo &= todo - 1;
                    const int e_done = __shfl_sync(FULL, (int)is_done, src);
                    const uint32_t e_epi = __shfl_sync(FULL, episode, src) + (e_done ? 1u : 0u);
                    const int e_idx = e_done ? 0 : __shfl_sync(FULL, index, src);
                    if (kCurves) wind_setup_warp(c, (long long)(blk * 32 + src), e_epi, e_idx, scratch);
                    if (lane == src) {
                        if (kCurves) {
#pragma unroll
                            for (int m = 0; m < 4; ++m) {
                                wa[m] = (T)scratch[m];
                                wb[m] = (T)scratch[4 + m];
                            }
                            wind_dirty = true;
                            if (!KMULTI) {  // patch the block in global memory
                                store_vecs<T, 4>(gb + c.off_wa, lane, wa);
                                if (WK == WIND_BOTH) store_vecs<T, 4>(gb + c.off_wb, lane, wb);
                            }
                        }
                        if (e_done) {  // Boat.__init__  boat_env.py:144-201
                            const int sy0 = episode_start_y(c, i, e_epi);  // :166-167
                            fx.start(c, d, sy0);
                            index = 0;
                            episode = e_epi;
                            episode_k = e_epi;
                            *epi_g = e_epi;
                            stage_reset_obs<T>(c, row, (T)sy0);
                            if (!KMULTI) store_dyn();
                        }
                    }
                    __syncwarp();  // scratch is reused by the next env of this warp
                }
            }
        }
        if (KMULTI) store_results();

        const int rows = min(32, n_end - blk * 32);
        // ---- observations: the [rows][11] tile is contiguous in obs_out -> one bulk store ----
        T *gobs = reinterpret_cast<T *>(a.obs_out) + (size_t)blk * (32 * kObsDim);
        if (rows == 32 && !a.no_bulk) {
            fence_proxy_async_smem();  // each lane: its st.shared rows -> visible to the async proxy
            __syncwarp();
#ifndef BOAT_DEBUG_SKIP_OBS
            if (lane == 0) {
                tma_store_1d(gobs, tile, kTileBytes);
                tma_store_commit();
            }
            tile_in_flight = true;
#endif
        } else {
            __syncwarp();
            for (int e = lane; e < rows * kObsDim; e += 32) gobs[e] = tile[e];
        }
        pbuf ^= 1;
    }
    if (kSetup > 0) {
        __syncwarp();
        if (lane == 0) {
            __threadfence_block();
            atomicAdd(&queue->producers_done, 1u);
        }
    }
    if (kq_on) kq_finish();
    if (tile_in_flight && lane == 0) tma_store_wait_all();  // smem must stay valid until the last store has read it
}

}  // namespace boatenv
