// toys.cu -- batched versions of the reference's two integrator demos,
// environment/toy_car.py:7-33 and environment/toy_parachute.py:8-41, on the Integrator
// semantics of control_theory/control_blocks.py:16-36 (call 0 returns initial_value and
// ignores the input; the STORED value is clamped, the RETURNED one is not).
//
// One thread per env, k loop iterations per launch with the env state in registers.
// The scripts' constants are per-env parameters: env i uses param * (1 + jitter * u),
// u = Philox uniform(-1,1) keyed (seed, env, param) and re-derived at every launch (no
// parameter array in HBM); env 0 is never jittered, so with default parameters it
// reproduces the scripts' known answers.  Compiled with -fmad=false: the fp64
// instantiation keeps the reference's rounding.
#include <cstring>
#include <new>

#include "common.cuh"
#include "launch.h"

using namespace boatenv;

constexpr int kToyMaxParams = 9;
constexpr int kCarParams = 4;        // accel, v_limit, dtheta, dt
constexpr int kParachuteParams = 9;  // h0, h1, area_free, area_chute, mass, c_w, rho, g, dt_integrator

struct ToyCfg {
    long long n_envs;
    unsigned long long seed;
    double jitter;
    double params[kToyMaxParams];
};

struct boattoy_handle {
    ToyCfg cfg;
    int kind, precision, device, n_params;
    size_t esize;
    void *state;      // 4 scalars per env, one 16-byte (fp32) / two 16-byte (fp64) vectors
    uint32_t *calls;  // integrator calls made so far (bit 31: finished)
};

namespace {

// Parameter k of env `env`: the script constant, jittered by Philox for env != 0.  Host and device evaluate the
// same expression (boattoy_params_host hands the values to a CPU reference).
__host__ __device__ __forceinline__ double toy_param_value(const ToyCfg &c, long long env, int k) {
    double v = c.params[k];
    if (env != 0 && c.jitter != 0.0) {
        const Philox4 r = philox4x32_10((uint32_t)env, (uint32_t)((unsigned long long)env >> 32), (uint32_t)(k >> 2),
                                        kStreamToy, (uint32_t)c.seed, (uint32_t)(c.seed >> 32));
        const double u = (double)(philox_word(r, k & 3) >> 8) * (1.0 / 8388608.0) - 1.0;
        v = v * (1.0 + c.jitter * u);
    }
    return v;
}
template <typename T>
__device__ __forceinline__ T toy_param(const ToyCfg &c, long long env, int k) { return (T)toy_param_value(c, env, k); }

// control_blocks.py:16-36 for calls > 0: returns x*dt + last (unclamped), stores clamped.
template <typename T>
__device__ __forceinline__ T integrate(T x, T dt, T &last, T upper) {
    const T y = x * dt + last;
    last = (y >= upper) ? upper : y;
    return y;
}

// toy_car.py:22-32.  state = {car_angle, a_integrator.last, s_x, s_y}
template <typename T>
__global__ void __launch_bounds__(256) toy_car_kernel(const __grid_constant__ ToyCfg c, T *state, uint32_t *calls,
                                                      int k, T *out, uint8_t *done_out) {
    using V = typename VecOf<T>::type;
    constexpr int W = VecOf<T>::W;
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= c.n_envs) return;
    const T accel = toy_param<T>(c, i, 0), v_limit = toy_param<T>(c, i, 1), dtheta = toy_param<T>(c, i, 2),
            dt = toy_param<T>(c, i, 3);
    T s[4];
    load_group<T, 4>(state, c.n_envs, i, s);
    uint32_t n = calls[i];
    T angle = s[0], v_last = s[1], s_x = s[2], s_y = s[3], v = (T)0;
    const T inf = (T)__int_as_float(0x7f800000);
    // fp32 mode: 5000 additions of 0.01 in fp32 would drift by ~1e-4 rad, so the heading is (calls + 1) * dtheta
    // in fp64 (the reference's accumulated sum equals it to ~1e-13), reduced to [-pi, pi] before the fp32 sincos
    const double dtheta_d = toy_param_value(c, i, 2);
    for (int it = 0; it < k; ++it) {
        if (sizeof(T) == 8) angle += dtheta;                          // :23
        else angle = (T)((double)(n + 1u) * dtheta_d);
        if (n == 0) {                                                 // call 0 of all three integrators
            v = (T)0;                                                 // Integrator(upper_limit=10): initial 0
            v_last = (v >= v_limit) ? v_limit : v;
            s_x = (T)0;
            s_y = (T)0;
        } else {
            v = integrate<T>(accel, dt, v_last, v_limit);             // :24
            T sn, cs;
            if (sizeof(T) == 8) { sn = (T)sin((double)angle); cs = (T)cos((double)angle); }
            else {
                const double ang = (double)(n + 1u) * dtheta_d;
                const double red = ang - 6.283185307179586476925 * rint(ang * 0.15915494309189533577);
                float a, b;
                sincosf((float)red, &a, &b);
                sn = (T)a; cs = (T)b;
            }
            T dummy_last = s_x;
            s_x = integrate<T>(v * cs, dt, dummy_last, inf);          // :26,29
            dummy_last = s_y;
            s_y = integrate<T>(v * sn, dt, dummy_last, inf);          // :27,30
        }
        ++n;
    }
    s[0] = angle; s[1] = v_last; s[2] = s_x; s[3] = s_y;
    store_group<T, 4>(state, c.n_envs, i, s);
    calls[i] = n;
    T o[4] = {s_x, s_y, v, angle};
    V *ov = reinterpret_cast<V *>(out) + i * (4 / W);
#pragma unroll
    for (int q = 0; q < 4 / W; ++q) ov[q] = pack(&o[q * W]);
    if (done_out) done_out[i] = 0;
}

// toy_parachute.py:23-40.  state = {total_a, a_integrator.last (v), v_integrator.last (s), v}
template <typename T>
__global__ void __launch_bounds__(256) toy_parachute_kernel(const __grid_constant__ ToyCfg c, T *state, uint32_t *calls,
                                                            int k, T *out, uint8_t *done_out) {
    using V = typename VecOf<T>::type;
    constexpr int W = VecOf<T>::W;
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= c.n_envs) return;
    const T h0 = toy_param<T>(c, i, 0), h1 = toy_param<T>(c, i, 1), area_free = toy_param<T>(c, i, 2),
            area_chute = toy_param<T>(c, i, 3), mass = toy_param<T>(c, i, 4), c_w = toy_param<T>(c, i, 5),
            rho = toy_param<T>(c, i, 6), g = toy_param<T>(c, i, 7), dt = toy_param<T>(c, i, 8);
    T s4[4];
    load_group<T, 4>(state, c.n_envs, i, s4);
    uint32_t word = calls[i];
    bool finished = (word >> 31) != 0;
    uint32_t n = word & 0x7fffffffu;
    // state slots: {total_a, v (= a_integrator.last: its limits are infinite), height}.  The height s is the sum of
    // ~2650 increments and decides the stopping iteration (:29), so the fp32 mode carries it in fp64 -- its two
    // 32-bit halves take slots 2 and 3 (no extra bytes); the fp64 mode keeps {.., s_last, v}.
    T total_a = s4[0], v_last = s4[1], v = s4[1];
    double s_acc = sizeof(T) == 8 ? (double)s4[2]
                                  : __hiloint2double(__float_as_int((float)s4[3]), __float_as_int((float)s4[2]));
    if (sizeof(T) == 8) v = s4[3];
    double s_d = (n == 0) ? toy_param_value(c, i, 0) : s_acc;
    const double h1_d = (double)h1;
    const T inf = (T)__int_as_float(0x7f800000);
    for (int it = 0; it < k && !finished; ++it) {
        total_a -= g;                                                 // :24
        if (n == 0) { v = (T)0; v_last = v; s_d = sizeof(T) == 8 ? (double)h0 : toy_param_value(c, i, 0); }  // call 0: initial values (:18-19)
        else {
            v = integrate<T>(total_a, dt, v_last, inf);               // :25
            s_d = sizeof(T) == 8 ? (double)((T)v * dt + (T)s_d) : (double)(v * dt) + s_d;   // :26
        }
        ++n;
        if (s_d < 0.0) { finished = true; break; }                    // :29-30
        const T area = (s_d < h1_d) ? area_chute : area_free;         // :33-36
        const T F_w = v * v * (T)0.5 * rho * c_w * area;
        total_a = F_w / mass;                                         // :38
    }
    const T s = (T)s_d;
    s4[0] = total_a; s4[1] = v_last;
    if (sizeof(T) == 8) { s4[2] = (T)s_d; s4[3] = v; }
    else { s4[2] = (T)__int_as_float(__double2loint(s_d)); s4[3] = (T)__int_as_float(__double2hiint(s_d)); }
    store_group<T, 4>(state, c.n_envs, i, s4);
    calls[i] = n | (finished ? 0x80000000u : 0u);
    T o[4] = {s, v, total_a, (T)n};
    V *ov = reinterpret_cast<V *>(out) + i * (4 / W);
#pragma unroll
    for (int q = 0; q < 4 / W; ++q) ov[q] = pack(&o[q * W]);
    if (done_out) done_out[i] = finished ? 1 : 0;
}

}  // namespace

extern "C" {

int boattoy_create(int kind, int64_t n_envs, const double *params_host, int32_t n_params, double jitter, uint64_t seed,
                   int precision, int device, boattoy_t *out) {
    if (!out || n_envs <= 0 || !params_host) return BOATENV_EINVAL;
    if (kind != BOATTOY_CAR && kind != BOATTOY_PARACHUTE) return BOATENV_EINVAL;
    if (n_params != (kind == BOATTOY_CAR ? kCarParams : kParachuteParams)) return BOATENV_EINVAL;
    if (precision != 32 && precision != 64) return BOATENV_EINVAL;
    *out = nullptr;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0 || device < 0 || device >= ndev) return BOATENV_ENODEVICE;
    boatenv::DeviceGuard _guard(device);
    if (!_guard.ok()) return (int)_guard.error();
    boattoy_handle *t = new (std::nothrow) boattoy_handle();
    if (!t) return BOATENV_EINVAL;
    std::memset(t, 0, sizeof(*t));
    t->kind = kind;
    t->precision = precision;
    t->device = device;
    t->n_params = n_params;
    t->esize = precision == 32 ? 4 : 8;
    t->cfg.n_envs = n_envs;
    t->cfg.seed = seed;
    t->cfg.jitter = jitter;
    for (int k = 0; k < n_params; ++k) t->cfg.params[k] = params_host[k];
    cudaError_t e = cudaMalloc(&t->state, (size_t)n_envs * 4 * t->esize);
    if (e == cudaSuccess) e = cudaMalloc((void **)&t->calls, (size_t)n_envs * sizeof(uint32_t));
    if (e != cudaSuccess) {
        boattoy_destroy(t);
        return (int)e;
    }
    *out = t;
    return boattoy_reset(t, nullptr);
}

int boattoy_params_host(int kind, const double *params_host, int32_t n_params, double jitter, uint64_t seed,
                        int64_t env_begin, int64_t n_envs, double *out) {
    if (!params_host || !out || env_begin < 0 || n_envs < 0) return BOATENV_EINVAL;
    if (kind != BOATTOY_CAR && kind != BOATTOY_PARACHUTE) return BOATENV_EINVAL;
    if (n_params != (kind == BOATTOY_CAR ? kCarParams : kParachuteParams)) return BOATENV_EINVAL;
    ToyCfg c;
    std::memset(&c, 0, sizeof(c));
    c.seed = seed;
    c.jitter = jitter;
    for (int k = 0; k < n_params; ++k) c.params[k] = params_host[k];
    for (int64_t e = 0; e < n_envs; ++e)
        for (int k = 0; k < n_params; ++k) out[e * n_params + k] = toy_param_value(c, env_begin + e, k);
    return BOATENV_OK;
}

int boattoy_destroy(boattoy_t t) {
    if (!t) return BOATENV_EINVAL;
    boatenv::DeviceGuard _guard(t->device);
    cudaFree(t->state);
    cudaFree(t->calls);
    delete t;
    return BOATENV_OK;
}

int boattoy_reset(boattoy_t t, void *stream) {
    if (!t) return BOATENV_EINVAL;
    GUARD_DEVICE(t);
    CUDA_TRY(cudaMemsetAsync(t->state, 0, (size_t)t->cfg.n_envs * 4 * t->esize, (cudaStream_t)stream));
    CUDA_TRY(cudaMemsetAsync(t->calls, 0, (size_t)t->cfg.n_envs * sizeof(uint32_t), (cudaStream_t)stream));
    return BOATENV_OK;
}

int boattoy_step(boattoy_t t, int32_t k, void *out, uint8_t *done_out, void *stream) {
    if (!t || !out || k < 1) return BOATENV_EINVAL;
    if ((reinterpret_cast<uintptr_t>(out) & 15u) != 0) return BOATENV_EALIGN;
    GUARD_DEVICE(t);
    const unsigned grid = (unsigned)((t->cfg.n_envs + 255) / 256);
    cudaStream_t st = (cudaStream_t)stream;
    if (t->kind == BOATTOY_CAR) {
        if (t->precision == 32) toy_car_kernel<float><<<grid, 256, 0, st>>>(t->cfg, (float *)t->state, t->calls, k, (float *)out, done_out);
        else toy_car_kernel<double><<<grid, 256, 0, st>>>(t->cfg, (double *)t->state, t->calls, k, (double *)out, done_out);
    } else {
        if (t->precision == 32) toy_parachute_kernel<float><<<grid, 256, 0, st>>>(t->cfg, (float *)t->state, t->calls, k, (float *)out, done_out);
        else toy_parachute_kernel<double><<<grid, 256, 0, st>>>(t->cfg, (double *)t->state, t->calls, k, (double *)out, done_out);
    }
    count_launch();
    CUDA_TRY(cudaGetLastError());
    return BOATENV_OK;
}

}  // extern "C"
