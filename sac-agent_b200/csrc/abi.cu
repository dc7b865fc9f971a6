// abi.cu -- the extern "C" front end of libboatenv.so (include/boatenv.h): handle
// management, config derivation, launches.  No compute happens on the host.
#include <algorithm>
#include <atomic>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <new>
#include <vector>

#include "common.cuh"
#include "launch.h"

using namespace boatenv;

namespace boatenv {
static std::atomic<long long> g_launches{0};
void count_launch() { g_launches.fetch_add(1, std::memory_order_relaxed); }
}  // namespace boatenv

struct boatenv_handle {
    DevCfg cfg;
    int precision, device;
    size_t esize;
    bool was_reset;
    unsigned launch_parity;    // consecutive step launches sweep the state in opposite directions
    uint2 *kq_entries;         // episode-end queue of the K > 1 kernels (allocated on first use)
    unsigned *kq_counts;
    long long kq_total;
    double *basis_dev;
    int *piece_bounds_dev;
    int32_t *ovr_s_y;
    double *ovr_knots;
    double *counters_out_dev;  // 8 doubles
    // step_host staging
    void *h_act, *h_obs, *h_rew;
    uint8_t *h_done, *h_term;
    cudaStream_t copy_in, compute, copy_out;
    cudaEvent_t ev_in[8], ev_k[8], ev_caller;
    int32_t *h_steps;          // step_k_host: executed sub-steps per env
    void *h_act_k;             // step_k_host: [K][n_envs] action staging (grown on demand)
    int h_act_k_rows;
    bool host_path_ready;
    // small-N zero-copy staging: one mapped pinned allocation the kernels read / write over PCIe directly
    // (no copy engine, one launch + one synchronize per call): [act | obs | rew | done | term | 10 doubles]
    char *zc_host, *zc_dev;
    size_t zc_act, zc_obs, zc_rew, zc_done, zc_term, zc_fields;   // byte offsets
};

// envs up to which boatenv_step_host* runs zero-copy (beyond it the chunked copy-engine pipeline wins)
constexpr long long kZeroCopyMaxEnvs = 2048;

// ---------------------------------------------------------------------------------
// Cardinal basis of the not-a-knot cubic spline through `fp` uniform knots (the curve
// scipy's interp1d(kind='cubic') builds at wind.py:82-84), per piece in the local
// coordinate s in [0,1]:  coefficient m of piece j = sum_k basis[(j*4+m)*fp + k] * y_k.
// Dimensionless moments m_i = h^2 S''(x_i) solve
//   m_0 - 2 m_1 + m_2 = 0,  m_{i-1}/6 + 2 m_i/3 + m_{i+1}/6 = y_{i-1} - 2 y_i + y_{i+1},
//   m_{n-3} - 2 m_{n-2} + m_{n-1} = 0.
// ---------------------------------------------------------------------------------
static void compute_spline_basis(int fp, std::vector<double> &basis) {
    const int n = fp;
    basis.assign((size_t)(n - 1) * 4 * n, 0.0);
    std::vector<double> A((size_t)n * n), rhs(n), m(n);
    for (int k = 0; k < n; ++k) {
        std::fill(A.begin(), A.end(), 0.0);
        std::vector<double> y(n, 0.0);
        y[k] = 1.0;
        A[0] = 1.0; A[1] = -2.0; A[2] = 1.0; rhs[0] = 0.0;
        for (int i = 1; i < n - 1; ++i) {
            A[(size_t)i * n + i - 1] = 1.0 / 6.0;
            A[(size_t)i * n + i] = 2.0 / 3.0;
            A[(size_t)i * n + i + 1] = 1.0 / 6.0;
            rhs[i] = y[i - 1] - 2.0 * y[i] + y[i + 1];
        }
        A[(size_t)(n - 1) * n + n - 3] = 1.0; A[(size_t)(n - 1) * n + n - 2] = -2.0;
        A[(size_t)(n - 1) * n + n - 1] = 1.0; rhs[n - 1] = 0.0;
        for (int c = 0; c < n; ++c) {  // Gaussian elimination, partial pivoting
            int piv = c;
            for (int r = c + 1; r < n; ++r)
                if (std::fabs(A[(size_t)r * n + c]) > std::fabs(A[(size_t)piv * n + c])) piv = r;
            if (piv != c) {
                for (int q = 0; q < n; ++q) std::swap(A[(size_t)c * n + q], A[(size_t)piv * n + q]);
                std::swap(rhs[c], rhs[piv]);
            }
            for (int r = c + 1; r < n; ++r) {
                const double f = A[(size_t)r * n + c] / A[(size_t)c * n + c];
                for (int q = c; q < n; ++q) A[(size_t)r * n + q] -= f * A[(size_t)c * n + q];
                rhs[r] -= f * rhs[c];
            }
        }
        for (int r = n - 1; r >= 0; --r) {
            double s = rhs[r];
            for (int q = r + 1; q < n; ++q) s -= A[(size_t)r * n + q] * m[q];
            m[r] = s / A[(size_t)r * n + r];
        }
        for (int j = 0; j < n - 1; ++j) {
            const double c0 = y[j];
            const double c1 = (y[j + 1] - y[j]) - (2.0 * m[j] + m[j + 1]) / 6.0;
            const double c2 = m[j] / 2.0;
            const double c3 = (m[j + 1] - m[j]) / 6.0;
            basis[((size_t)j * 4 + 0) * n + k] = c0;
            basis[((size_t)j * 4 + 1) * n + k] = c1;
            basis[((size_t)j * 4 + 2) * n + k] = c2;
            basis[((size_t)j * 4 + 3) * n + k] = c3;
        }
    }
}

static int derive_config(const boatenv_params *p, DevCfg &c) {
    const double PI = 3.14159265358979323846;
    std::memset(&c, 0, sizeof(c));
    c.p = *p;
    c.experiment = p->experiment;
    c.test_mode = p->test_mode;
    switch (p->experiment) {  // wind.py:30-67
    case 1: case 2: c.wind_kind = WIND_NONE; c.ncurves = 0; break;
    case 3: c.wind_kind = WIND_CONST; c.ncurves = 0; break;
    case 4: c.wind_kind = WIND_VEL_CURVE; c.ncurves = 1; break;
    case 5: c.wind_kind = WIND_ANGLE_RECT; c.ncurves = 1; break;
    case 6: c.wind_kind = WIND_BOTH; c.ncurves = 2; break;
    default: return BOATENV_EEXPERIMENT;
    }
    if (!(p->dt > 0.0) || !(p->t_max > 0.0) || !(p->track_width > 0.0) || !(p->fuel != 0.0)) return BOATENV_EINVAL;
    c.fp = p->fixed_points;
    if (c.ncurves > 0) {
        if (c.fp < 4) return BOATENV_EFIXEDPOINTS;  // wind.py:73-75
        if (c.fp > kMaxKnots) return BOATENV_EUNSUPPORTED;
    } else if (c.fp < 2 || c.fp > kMaxKnots) {
        c.fp = 8;  // unused without random curves
    }
    c.npieces = c.fp - 1;
    const double Ld = p->t_max / p->dt;  // wind.py:14-15
    if (!(Ld >= 2.0) || Ld > 1048576.0 - 64.0) return BOATENV_EUNSUPPORTED;  // fp32 root location in wind_setup_warp; 20-bit step index
    if (Ld < 4.0) return BOATENV_EUNSUPPORTED;
    c.L = (int)Ld;
    c.Lm1 = c.L - 1;
    c.inv_Lm1 = 1.0 / (double)c.Lm1;
    {   // exact floor(n / Lm1) for 0 <= n <= L * npieces as a multiply-high (Granlund & Montgomery):
        // p = max(32, N + l) with 2^N > n_max, 2^l >= Lm1;  m = ceil(2^p / Lm1) < 2^32
        const unsigned long long nmax = (unsigned long long)c.L * (unsigned long long)c.npieces;
        int N = 1, l = 0;
        while ((1ULL << N) <= nmax) ++N;
        while ((1ULL << l) < (unsigned long long)c.Lm1) ++l;
        int pw = N + l < 32 ? 32 : N + l;
        const unsigned __int128 two_p = (unsigned __int128)1 << pw;
        const unsigned __int128 m = (two_p + (unsigned)c.Lm1 - 1) / (unsigned)c.Lm1;
        if (m >> 32) return BOATENV_EUNSUPPORTED;
        c.magic_m = (unsigned)m;
        c.magic_s = (unsigned)(pw - 32);
    }
    {   // boat_env.py:69,98: t accumulates dt; timeout at the first step with t_max <= t
        double t = 0.0;
        int n = 0;
        while (n < c.L + 16) { t += p->dt; ++n; if (p->t_max <= t) break; }
        c.timeout_steps = n;
    }
    {   // boat_env.py:70,94: fuel starts at p->fuel, loses 1 per step, out_of_fuel when fuel < 0
        const double fs = std::floor(p->fuel) + 1.0;
        c.fuel_steps = fs < 1.0 ? 1 : (fs > 2147483647.0 ? 2147483647 : (int)fs);
    }
    c.s_y_half = (int)(p->track_width * 0.8);  // boat_env.py:148-149
    if (c.s_y_half < 1) c.s_y_half = 1;
    c.direction_rad = p->direction * (PI / 180.0);
    c.prop_d4 = std::pow(p->propeller_diameter, 4.0);

    FastConsts &f = c.f;
    const double n = 20.0;
    f.dt = (float)p->dt;
    f.tenth = 0.1f;
    const double kdx = p->c_r_front * 0.5 * p->rho * p->boat_area_front;
    const double kdy = p->c_r_side * 0.5 * p->rho * p->boat_area_side;
    f.kdx = (float)kdx;
    f.kJ = (float)((1.0 - p->wake_friction) / (n * p->propeller_diameter));
    f.kT = (float)(n * n * p->rho * c.prop_d4 * (1.0 - p->thrust_deduction));
    f.cxy = (float)(p->boat_m + p->boat_m_y);
    f.inv_mx = (float)(1.0 / (p->boat_m + p->boat_m_x));
    f.kdy = (float)kdy;
    f.kru = (float)(p->c_r_front * 0.5 * p->rho * p->rudder_area);
    f.cyx = (float)(p->boat_m + p->boat_m_x);
    f.inv_my = (float)(1.0 / (p->boat_m + p->boat_m_y));
    f.kh = (float)(kdy * p->boat_l * 5.0);
    f.kmr = (float)(p->c_r_side * 0.5 * p->rho * p->rudder_area * (p->boat_b / 2.0));
    f.inv_I = (float)(1.0 / (p->boat_I + p->boat_Iz));
    f.kwx = (float)kdx;
    f.kwy = (float)kdy;
    const double wv = p->max_velocity, ww = wv * std::fabs(wv);
    f.fwx_c = (float)(ww * kdx * std::cos(c.direction_rad));
    f.fwy_c = (float)(ww * kdy * std::sin(c.direction_rad));
    f.cos_dir = (float)std::cos(c.direction_rad);
    f.sin_dir = (float)std::sin(c.direction_rad);
    const double th_lo = PI / 2.0, th_hi = PI + PI / 2.0;  // wind.py:57-58
    f.fwx_lo = (float)(ww * kdx * std::cos(th_lo));
    f.fwy_lo = (float)(ww * kdy * std::sin(th_lo));
    f.fwx_hi = (float)(ww * kdx * std::cos(th_hi));
    f.fwy_hi = (float)(ww * kdy * std::sin(th_hi));
    f.inv_goal = (float)(1.0 / p->goal_line);
    f.inv_5 = 0.2f;
    f.inv_ax = (float)(1.0 / 0.025);
    f.W = (float)p->track_width;
    f.inv_2W = (float)(1.0 / (2.0 * p->track_width));
    f.inv_2 = 0.5f;
    f.inv_ay = (float)(1.0 / 0.37);
    f.inv_2pi = (float)(1.0 / (2.0 * PI));
    f.inv_vr = (float)(1.0 / 8.5e-3);
    f.inv_ar = (float)(1.0 / 1.4e-5);
    f.third_pi = (float)(PI / 3.0);
    f.inv_rud = (float)(1.0 / (2.0 * PI / 3.0));
    f.inv_fuel = (float)(1.0 / p->fuel);
    f.fuel0 = (float)p->fuel;
    f.goal = (float)p->goal_line;
    f.oob = (float)(p->track_width + p->oob_offset);
    f.pi3 = (float)(PI / 3.0);
    f.pi4 = (float)(PI / 4.0);
    f.pi2 = (float)(PI / 2.0);
    f.rew_inv_W = (float)(1.0 / p->track_width);
    f.rew_k = (float)(-0.03 / 3.4);
    f.rew_y0 = (float)(p->track_width * 0.2);
    f.inv_Lm1 = (float)c.inv_Lm1;
    {   // fixed-point carriers of the fp32 mode (struct Fx<float>): the largest shifts that leave headroom
        // beyond the termination thresholds (positions saturate instead of wrapping in the unstable regime)
        auto shift_for = [](double reach) {
            int sh = 30;
            while (sh > 0 && reach * (double)(1LL << sh) >= 2147483647.0) --sh;
            return sh;
        };
        // ... and that keep one step's increment inside the 1.5 * 2^23 rounding trick (|increment| < 2^22 units) for
        // speeds up to 16 m/s, three times what the boat model reaches (the observation range of v_x ends at 5 m/s)
        int inc_shift = 30;
        while (inc_shift > 0 && 16.0 * p->dt * (double)(1LL << inc_shift) >= 4194304.0) --inc_shift;
        f.sx_shift = std::min(inc_shift, shift_for(std::fabs(p->goal_line) * 1.02 + 16.0));
        f.sy_shift = std::min(inc_shift, shift_for((std::fabs(p->track_width) + std::fabs(p->oob_offset)) * 1.02 + 16.0));
        f.sx_k = (float)(p->dt * (double)(1LL << f.sx_shift));
        f.sy_k = (float)(p->dt * (double)(1LL << f.sy_shift));
        f.sx_inv = (float)(1.0 / (double)(1LL << f.sx_shift));
        f.sy_inv = (float)(1.0 / (double)(1LL << f.sy_shift));
        f.sx_goal = (int)std::ceil(p->goal_line * (double)(1LL << f.sx_shift));
        f.sy_oob = (int)std::floor((p->track_width + p->oob_offset) * (double)(1LL << f.sy_shift));
        f.sy_oob2 = 2u * (unsigned)f.sy_oob;
        {   // the bit patterns of the two rudder thresholds (common.cuh) are those of the doubles
            unsigned long long b3, b4;
            const double d3 = kRudPi3, d4 = kRudPi4;
            std::memcpy(&b3, &d3, 8);
            std::memcpy(&b4, &d4, 8);
            if (b3 != kRudPi3Bits || b4 != kRudPi4Bits) return BOATENV_EUNSUPPORTED;
        }
        if (std::floor((PI / 3.0) * 4398046511104.0) != kRudPi3 || std::floor((PI / 4.0) * 4398046511104.0) != kRudPi4)
            return BOATENV_EUNSUPPORTED;   // the literals in common.cuh are these two numbers
        f.sx_obs = (float)(1.0 / (double)(1LL << f.sx_shift) / p->goal_line);
        f.sy_obs = (float)(1.0 / (double)(1LL << f.sy_shift) / (2.0 * p->track_width));
    }
    return BOATENV_OK;
}

static inline bool aligned16(const void *p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

extern "C" {

const char *boatenv_version(void) { return "boatenv-b200 0.1 (sm_100a)"; }

const char *boatenv_error_string(int code) {
    switch (code) {
    case BOATENV_OK: return "ok";
    case BOATENV_EINVAL: return "invalid argument";
    case BOATENV_EEXPERIMENT: return "Well someone tried to use an experiment that doesnt exist!";
    case BOATENV_EFIXEDPOINTS:
        return "Please select at least 4 fixed_points in your config. The interpolation doesn't work otherwise!";
    case BOATENV_EUNSUPPORTED: return "configuration valid for the reference but unsupported by this build";
    case BOATENV_ENODEVICE: return "no usable CUDA device";
    case BOATENV_ESTATE: return "step() called before reset()";
    case BOATENV_EALIGN: return "tensor pointer is not 16-byte aligned";
    default: return code > 0 ? cudaGetErrorString((cudaError_t)code) : "unknown error";
    }
}

int64_t boatenv_kernel_launches(void) { return (int64_t)g_launches.load(); }

int boatenv_create(const boatenv_params *params, int64_t n_envs, uint64_t seed, int64_t env_id_offset,
                   int precision, int device, boatenv_t *out) {
    if (!params || !out || n_envs <= 0 || env_id_offset < 0) return BOATENV_EINVAL;
    if (precision != 32 && precision != 64) return BOATENV_EINVAL;
    if (n_envs > 2147483647LL - 64) return BOATENV_EUNSUPPORTED;  // per-handle env indices are 32-bit in the kernels
    *out = nullptr;
    DevCfg cfg;
    int rc = derive_config(params, cfg);
    if (rc) return rc;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0 || device < 0 || device >= ndev) return BOATENV_ENODEVICE;
    DeviceGuard _guard(device);
    if (!_guard.ok()) return (int)_guard.error();
    boatenv_handle *h = new (std::nothrow) boatenv_handle();
    if (!h) return BOATENV_EINVAL;
    std::memset(h, 0, sizeof(*h));
    h->precision = precision;
    h->device = device;
    h->esize = precision == 32 ? 4 : 8;
    cfg.n_envs = n_envs;
    cfg.env_id_offset = env_id_offset;
    cfg.seed = seed;
    cudaError_t e = cudaSuccess;
    auto alloc = [&](void **p, size_t bytes) { if (e == cudaSuccess) e = cudaMalloc(p, bytes); };
    {   // tile-blocked state: [dyn][step index][wind A][wind B][episode] sections per 32-env block (common.cuh)
        const int nd = D_COUNT * (int)h->esize / 16, nw = 4 * (int)h->esize / 16;
        cfg.off_idx = 32 * 16 * nd;
        cfg.off_wa = cfg.off_idx + 32 * 4;
        cfg.off_wb = cfg.off_wa + (cfg.ncurves >= 1 ? 32 * 16 * nw : 0);
        cfg.off_epi = cfg.off_wb + (cfg.ncurves >= 2 ? 32 * 16 * nw : 0);
        cfg.block_bytes = cfg.off_epi + 32 * 4;
    }
    const size_t state_bytes = (size_t)num_blocks(n_envs) * (size_t)cfg.block_bytes;
    alloc((void **)&cfg.state, state_bytes);
    alloc((void **)&cfg.counters, kCounterSlots * 32 * sizeof(double));
    alloc((void **)&h->counters_out_dev, kNumCounters * sizeof(double));
    std::vector<double> basis;
    compute_spline_basis(cfg.fp, basis);
    alloc((void **)&h->basis_dev, basis.size() * sizeof(double));
    if (e == cudaSuccess) e = cudaMemcpy(h->basis_dev, basis.data(), basis.size() * sizeof(double), cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaMemset(cfg.state, 0xFF, state_bytes);  // episode -1: reset() makes it 0
    if (e == cudaSuccess) e = cudaMemset(cfg.counters, 0, kCounterSlots * 32 * sizeof(double));
    cfg.basis = h->basis_dev;
    {   // first / last sample that piece_of() assigns to piece j: floor(index*np / Lm1) == j, i.e.
        // ceil(j*Lm1/np) <= index <= floor(((j+1)*Lm1 - 1)/np); the last piece also owns sample L-1
        std::vector<int> pb(2 * (size_t)cfg.npieces);
        for (int j = 0; j < cfg.npieces; ++j) {
            pb[2 * j] = (int)(((long long)j * cfg.Lm1 + cfg.npieces - 1) / cfg.npieces);
            pb[2 * j + 1] = j == cfg.npieces - 1 ? cfg.L - 1
                                                 : (int)((((long long)(j + 1) * cfg.Lm1) - 1) / cfg.npieces);
        }
        alloc((void **)&h->piece_bounds_dev, pb.size() * sizeof(int));
        if (e == cudaSuccess) e = cudaMemcpy(h->piece_bounds_dev, pb.data(), pb.size() * sizeof(int), cudaMemcpyHostToDevice);
        cfg.piece_bounds = h->piece_bounds_dev;
        cfg.per_piece = (float)((double)cfg.Lm1 / (double)cfg.npieces);
        cfg.inv_per_piece = (float)((double)cfg.npieces / (double)cfg.Lm1);
    }
    h->cfg = cfg;
    if (e != cudaSuccess) {
        boatenv_destroy(h);
        return (int)e;
    }
    *out = h;
    return BOATENV_OK;
}

int boatenv_destroy(boatenv_t h) {
    if (!h) return BOATENV_EINVAL;
    DeviceGuard _guard(h->device);
    cudaFree(h->cfg.state);
    cudaFree(h->cfg.counters);
    cudaFree(h->counters_out_dev);
    cudaFree(h->basis_dev);
    cudaFree(h->piece_bounds_dev);
    cudaFree(h->kq_entries);
    cudaFree(h->kq_counts);
    cudaFree(h->ovr_s_y);
    cudaFree(h->ovr_knots);
    cudaFree(h->h_act);
    cudaFree(h->h_obs);
    cudaFree(h->h_rew);
    cudaFree(h->h_done);
    cudaFree(h->h_term);
    cudaFree(h->h_steps);
    cudaFree(h->h_act_k);
    if (h->zc_host) cudaFreeHost(h->zc_host);
    if (h->host_path_ready) {
        cudaStreamDestroy(h->copy_in);
        cudaStreamDestroy(h->compute);
        cudaStreamDestroy(h->copy_out);
        for (int i = 0; i < 8; ++i) { cudaEventDestroy(h->ev_in[i]); cudaEventDestroy(h->ev_k[i]); }
        cudaEventDestroy(h->ev_caller);
    }
    delete h;
    return BOATENV_OK;
}

int boatenv_reset(boatenv_t h, const uint8_t *mask, void *obs_out, void *stream) {
    if (!h) return BOATENV_EINVAL;
    GUARD_DEVICE(h);
    cudaStream_t st = (cudaStream_t)stream;
    CUDA_TRY(h->precision == 32 ? launch_reset_f32(h->cfg, mask, obs_out, st)
                                : launch_reset_f64(h->cfg, mask, obs_out, st));
    if (!mask) h->was_reset = true;
    return BOATENV_OK;
}

static int step_common(boatenv_t h, StepArgs &a, cudaStream_t st) {
    if (!h->was_reset) return BOATENV_ESTATE;
    a.reverse = (int)(h->launch_parity++ & 1u);
    if (!a.actions || !a.obs_out || !a.reward_out || (!a.done_out && !a.term_out) || a.ksteps < 1) return BOATENV_EINVAL;
    if (!aligned16(a.obs_out)) return BOATENV_EALIGN;
    GUARD_DEVICE(h);
    CUDA_TRY(h->precision == 32 ? launch_step_f32(h->cfg, a, st) : launch_step_f64(h->cfg, a, st));
    return BOATENV_OK;
}

int boatenv_step(boatenv_t h, const void *actions, void *obs_out, void *reward_out, uint8_t *done_out,
                 uint8_t *term_out, void *final_obs_out, uint32_t flags, void *stream) {
    if (!h) return BOATENV_EINVAL;
    StepArgs a;
    std::memset(&a, 0, sizeof(a));
    a.env_begin = 0;
    a.env_end = h->cfg.n_envs;
    a.actions = actions;
    a.action_stride = 0;
    a.ksteps = 1;
    a.obs_out = obs_out;
    a.reward_out = reward_out;
    a.done_out = done_out;
    a.term_out = term_out;
    a.final_obs_out = final_obs_out;
    a.flags = flags;
    return step_common(h, a, (cudaStream_t)stream);
}

// The episode-end queue of the K > 1 kernels with wind curves under auto-reset (StepArgs::kq_*), allocated on first
// use.  Sized for every env plus the rounding of up to 1024 per-CTA regions to whole warp tiles; a launch whose
// regions do not fit sets the wind up inline instead (step_impl.inl).
static int ensure_episode_queue(boatenv_t h) {
    if (h->kq_entries) return BOATENV_OK;
    GUARD_DEVICE(h);
    h->kq_total = num_blocks(h->cfg.n_envs) * 32 + 1024LL * kWarpsPerCta * 32;
    CUDA_TRY(cudaMalloc((void **)&h->kq_entries, (size_t)h->kq_total * sizeof(uint2)));
    CUDA_TRY(cudaMalloc((void **)&h->kq_counts, 4096 * sizeof(unsigned)));
    return BOATENV_OK;
}

int boatenv_step_k(boatenv_t h, const void *actions, int64_t action_stride, int32_t k, void *obs_out,
                   void *reward_out, uint8_t *done_out, uint8_t *term_out, int32_t *steps_out, uint32_t flags,
                   void *stream) {
    if (!h || k < 1 || (action_stride != 0 && action_stride < h->cfg.n_envs)) return BOATENV_EINVAL;
    StepArgs a;
    std::memset(&a, 0, sizeof(a));
    a.env_begin = 0;
    a.env_end = h->cfg.n_envs;
    a.actions = actions;
    a.action_stride = action_stride;
    a.ksteps = k;
    a.obs_out = obs_out;
    a.reward_out = reward_out;
    a.done_out = done_out;
    a.term_out = term_out;
    a.steps_out = steps_out;
    a.flags = flags;
    if (k > 1 && h->cfg.ncurves > 0 && (flags & BOATENV_AUTO_RESET)) {  // episode-end queue of the fused kernels
        const int rc = ensure_episode_queue(h);
        if (rc) return rc;
        a.kq_entries = h->kq_entries;
        a.kq_counts = h->kq_counts;
        a.kq_total = h->kq_total;
    }
    return step_common(h, a, (cudaStream_t)stream);
}

static int ensure_host_path(boatenv_t h) {
    if (h->host_path_ready) return BOATENV_OK;
    const size_t n = (size_t)h->cfg.n_envs;
    CUDA_TRY(cudaMalloc(&h->h_act, n * h->esize));
    CUDA_TRY(cudaMalloc(&h->h_obs, n * kObsDim * h->esize));
    CUDA_TRY(cudaMalloc(&h->h_rew, n * h->esize));
    CUDA_TRY(cudaMalloc((void **)&h->h_done, n));
    CUDA_TRY(cudaMalloc((void **)&h->h_term, n));
    CUDA_TRY(cudaStreamCreateWithFlags(&h->copy_in, cudaStreamNonBlocking));
    CUDA_TRY(cudaStreamCreateWithFlags(&h->compute, cudaStreamNonBlocking));
    CUDA_TRY(cudaStreamCreateWithFlags(&h->copy_out, cudaStreamNonBlocking));
    for (int i = 0; i < 8; ++i) {
        CUDA_TRY(cudaEventCreateWithFlags(&h->ev_in[i], cudaEventDisableTiming));
        CUDA_TRY(cudaEventCreateWithFlags(&h->ev_k[i], cudaEventDisableTiming));
    }
    CUDA_TRY(cudaEventCreateWithFlags(&h->ev_caller, cudaEventDisableTiming));
    h->host_path_ready = true;
    return BOATENV_OK;
}

static int step_host_impl(boatenv_t h, const void *actions_host, int k, void *obs_host, void *reward_host,
                          uint8_t *done_host, uint8_t *term_host, int32_t *steps_host, uint32_t flags, cudaStream_t caller);

static int ensure_zero_copy(boatenv_t h) {
    if (h->zc_host) return BOATENV_OK;
    const size_t n = (size_t)std::min<long long>(h->cfg.n_envs, kZeroCopyMaxEnvs), es = h->esize;
    auto up = [](size_t x) { return (x + 127) / 128 * 128; };
    h->zc_act = 0;
    h->zc_obs = up(h->zc_act + n * es);
    h->zc_rew = up(h->zc_obs + n * kObsDim * es);
    h->zc_done = up(h->zc_rew + n * es);
    h->zc_term = up(h->zc_done + n);
    h->zc_fields = up(h->zc_term + n);
    const size_t bytes = h->zc_fields + 16 * sizeof(double);
    void *hp = nullptr, *dp = nullptr;
    CUDA_TRY(cudaHostAlloc(&hp, bytes, cudaHostAllocMapped));
    cudaError_t e = cudaHostGetDevicePointer(&dp, hp, 0);
    if (e != cudaSuccess) { cudaFreeHost(hp); return (int)e; }
    std::memset(hp, 0, bytes);
    h->zc_host = (char *)hp;
    h->zc_dev = (char *)dp;
    return BOATENV_OK;
}

// Small-N step through host buffers: the kernel reads the actions from, and writes its outputs to, mapped
// pinned memory; the caller's buffers (pinned or pageable) are filled by plain memcpy.
static int step_host_zero_copy(boatenv_t h, const void *actions_host, void *obs_host, void *reward_host,
                               uint8_t *done_host, uint8_t *term_host, uint32_t flags) {
    int rc = ensure_zero_copy(h);
    if (rc) return rc;
    const size_t n = (size_t)h->cfg.n_envs, es = h->esize;
    std::memcpy(h->zc_host + h->zc_act, actions_host, n * es);
    StepArgs a;
    std::memset(&a, 0, sizeof(a));
    a.env_begin = 0;
    a.env_end = h->cfg.n_envs;
    a.actions = h->zc_dev + h->zc_act;
    a.ksteps = 1;
    a.obs_out = h->zc_dev + h->zc_obs;
    a.reward_out = h->zc_dev + h->zc_rew;
    a.done_out = (uint8_t *)(h->zc_dev + h->zc_done);
    a.term_out = (uint8_t *)(h->zc_dev + h->zc_term);
    a.flags = flags;
    a.reverse = (int)(h->launch_parity++ & 1u);
    a.no_bulk = 1;
    CUDA_TRY(h->precision == 32 ? launch_step_f32(h->cfg, a, h->compute) : launch_step_f64(h->cfg, a, h->compute));
    CUDA_TRY(cudaStreamSynchronize(h->compute));
    std::memcpy(obs_host, h->zc_host + h->zc_obs, n * kObsDim * es);
    std::memcpy(reward_host, h->zc_host + h->zc_rew, n * es);
    std::memcpy(done_host, h->zc_host + h->zc_done, n);
    if (term_host) std::memcpy(term_host, h->zc_host + h->zc_term, n);
    return BOATENV_OK;
}

int boatenv_step_host(boatenv_t h, const void *actions_host, void *obs_host, void *reward_host, uint8_t *done_host,
                      uint32_t flags) {
    return step_host_impl(h, actions_host, 1, obs_host, reward_host, done_host, nullptr, nullptr, flags, nullptr);
}

int boatenv_step_host_term(boatenv_t h, const void *actions_host, void *obs_host, void *reward_host,
                           uint8_t *done_host, uint8_t *term_host, uint32_t flags) {
    if (!term_host) return BOATENV_EINVAL;
    return step_host_impl(h, actions_host, 1, obs_host, reward_host, done_host, term_host, nullptr, flags, nullptr);
}

int boatenv_step_host_stream(boatenv_t h, const void *actions_host, void *obs_host, void *reward_host,
                             uint8_t *done_host, uint8_t *term_host, uint32_t flags, void *stream) {
    return step_host_impl(h, actions_host, 1, obs_host, reward_host, done_host, term_host, nullptr, flags,
                          (cudaStream_t)stream);
}

int boatenv_step_k_host(boatenv_t h, const void *actions_host, int32_t k, void *obs_host, void *reward_host,
                        uint8_t *done_host, uint8_t *term_host, int32_t *steps_host, uint32_t flags, void *stream) {
    if (k < 1) return BOATENV_EINVAL;
    return step_host_impl(h, actions_host, k, obs_host, reward_host, done_host, term_host, steps_host, flags,
                          (cudaStream_t)stream);
}

// Host-buffer step: H2D of the actions, the step kernel and the D2H of its outputs run as a chunked pipeline on
// three streams of the handle.  `caller` is the stream the caller has been queueing work for this handle on
// (reset / step / learner kernels): the pipeline waits for an event recorded there -- no device-wide synchronise,
// so a learner running on another stream of the same process is not serialised against this call.
static int step_host_impl(boatenv_t h, const void *actions_host, int k, void *obs_host, void *reward_host,
                          uint8_t *done_host, uint8_t *term_host, int32_t *steps_host, uint32_t flags, cudaStream_t caller) {
    if (!h || !actions_host || !obs_host || !reward_host || !done_host) return BOATENV_EINVAL;
    if (!h->was_reset) return BOATENV_ESTATE;
    GUARD_DEVICE(h);
    int rc = ensure_host_path(h);
    if (rc) return rc;
    CUDA_TRY(cudaEventRecord(h->ev_caller, caller));
    CUDA_TRY(cudaStreamWaitEvent(h->copy_in, h->ev_caller, 0));
    CUDA_TRY(cudaStreamWaitEvent(h->compute, h->ev_caller, 0));
    const long long n = h->cfg.n_envs;
    if (k == 1 && !steps_host && n <= kZeroCopyMaxEnvs)
        return step_host_zero_copy(h, actions_host, obs_host, reward_host, done_host, term_host, flags);
    const size_t es = h->esize;
    void *act_dev = h->h_act;
    if (k > 1) {  // [K][n] staging
        if (h->h_act_k_rows < k) {
            cudaFree(h->h_act_k);
            h->h_act_k = nullptr;
            h->h_act_k_rows = 0;
            CUDA_TRY(cudaMalloc(&h->h_act_k, (size_t)k * (size_t)n * es));
            h->h_act_k_rows = k;
        }
        act_dev = h->h_act_k;
        if (steps_host && !h->h_steps) CUDA_TRY(cudaMalloc((void **)&h->h_steps, (size_t)n * sizeof(int32_t)));
        if (h->cfg.ncurves > 0 && (flags & BOATENV_AUTO_RESET)) {  // episode-end queue of the fused kernels
            rc = ensure_episode_queue(h);
            if (rc) return rc;
        }
    }
    // chunks are multiples of the CTA tile so that every tile keeps its 16-byte alignment
    int nchunks = n >= 8LL * 65536 ? 8 : (n >= 4LL * 65536 ? 4 : 1);
    long long per = ((n + nchunks - 1) / nchunks + kTile - 1) / kTile * kTile;
    const int rev = (int)(h->launch_parity++ & 1u);
    for (int cidx = 0; cidx < nchunks; ++cidx) {
        const long long b = (long long)cidx * per, e = std::min(n, b + per);
        if (b >= e) break;
        const size_t cnt = (size_t)(e - b);
        if (k == 1) {
            CUDA_TRY(cudaMemcpyAsync((char *)act_dev + b * es, (const char *)actions_host + b * es, cnt * es,
                                     cudaMemcpyHostToDevice, h->copy_in));
        } else {  // rows k of the [K][n] action matrix, columns [b, e)
            CUDA_TRY(cudaMemcpy2DAsync((char *)act_dev + b * es, (size_t)n * es, (const char *)actions_host + b * es,
                                       (size_t)n * es, cnt * es, (size_t)k, cudaMemcpyHostToDevice, h->copy_in));
        }
        CUDA_TRY(cudaEventRecord(h->ev_in[cidx], h->copy_in));
        CUDA_TRY(cudaStreamWaitEvent(h->compute, h->ev_in[cidx], 0));
        StepArgs a;
        std::memset(&a, 0, sizeof(a));
        a.env_begin = b;
        a.env_end = e;
        a.actions = act_dev;
        a.action_stride = k > 1 ? n : 0;
        a.ksteps = k;
        a.obs_out = h->h_obs;
        a.reward_out = h->h_rew;
        a.done_out = h->h_done;
        a.term_out = term_host ? h->h_term : nullptr;
        a.steps_out = steps_host ? h->h_steps : nullptr;
        a.flags = flags;
        a.reverse = rev;
        if (k > 1 && h->kq_entries && (flags & BOATENV_AUTO_RESET)) {
            a.kq_entries = h->kq_entries;
            a.kq_counts = h->kq_counts;
            a.kq_total = h->kq_total;
        }
        CUDA_TRY(h->precision == 32 ? launch_step_f32(h->cfg, a, h->compute) : launch_step_f64(h->cfg, a, h->compute));
        CUDA_TRY(cudaEventRecord(h->ev_k[cidx], h->compute));
        CUDA_TRY(cudaStreamWaitEvent(h->copy_out, h->ev_k[cidx], 0));
        CUDA_TRY(cudaMemcpyAsync((char *)obs_host + b * kObsDim * es, (char *)h->h_obs + b * kObsDim * es,
                                 cnt * kObsDim * es, cudaMemcpyDeviceToHost, h->copy_out));
        CUDA_TRY(cudaMemcpyAsync((char *)reward_host + b * es, (char *)h->h_rew + b * es, cnt * es,
                                 cudaMemcpyDeviceToHost, h->copy_out));
        CUDA_TRY(cudaMemcpyAsync(done_host + b, h->h_done + b, cnt, cudaMemcpyDeviceToHost, h->copy_out));
        if (term_host) CUDA_TRY(cudaMemcpyAsync(term_host + b, h->h_term + b, cnt, cudaMemcpyDeviceToHost, h->copy_out));
        if (steps_host)
            CUDA_TRY(cudaMemcpyAsync(steps_host + b, h->h_steps + b, cnt * sizeof(int32_t), cudaMemcpyDeviceToHost, h->copy_out));
    }
    CUDA_TRY(cudaStreamSynchronize(h->copy_out));
    return BOATENV_OK;
}

int boatenv_get_field(boatenv_t h, int field, void *out, void *stream) {
    if (!h || !out || field < 0 || field > BOATENV_F_EPISODE) return BOATENV_EINVAL;
    GUARD_DEVICE(h);
    CUDA_TRY(h->precision == 32 ? launch_get_field_f32(h->cfg, field, out, (cudaStream_t)stream)
                                : launch_get_field_f64(h->cfg, field, out, (cudaStream_t)stream));
    return BOATENV_OK;
}

int boatenv_set_field(boatenv_t h, int field, const void *in, void *stream) {
    if (!h || !in || field < 0 || field > BOATENV_F_EPISODE) return BOATENV_EINVAL;
    GUARD_DEVICE(h);
    CUDA_TRY(h->precision == 32 ? launch_set_field_f32(h->cfg, field, in, (cudaStream_t)stream)
                                : launch_set_field_f64(h->cfg, field, in, (cudaStream_t)stream));
    return BOATENV_OK;
}

int boatenv_env_state_host(boatenv_t h, int64_t env_index, double *out_host) {
    if (!h || !out_host || env_index < 0 || env_index >= h->cfg.n_envs) return BOATENV_EINVAL;
    if (!h->was_reset) return BOATENV_ESTATE;
    GUARD_DEVICE(h);
    int rc = ensure_host_path(h);
    if (!rc) rc = ensure_zero_copy(h);
    if (rc) return rc;
    // ordered after the work queued on the legacy default stream (what the single-env drop-in uses): an event wait,
    // not a device-wide synchronise
    CUDA_TRY(cudaEventRecord(h->ev_caller, nullptr));
    CUDA_TRY(cudaStreamWaitEvent(h->compute, h->ev_caller, 0));
    double *dev = reinterpret_cast<double *>(h->zc_dev + h->zc_fields);
    CUDA_TRY(h->precision == 32 ? launch_env_state_f32(h->cfg, env_index, dev, h->compute)
                                : launch_env_state_f64(h->cfg, env_index, dev, h->compute));
    CUDA_TRY(cudaStreamSynchronize(h->compute));
    std::memcpy(out_host, h->zc_host + h->zc_fields, 10 * sizeof(double));
    return BOATENV_OK;
}

int boatenv_wind_length(boatenv_t h) { return h ? h->cfg.L : BOATENV_EINVAL; }

int boatenv_wind_table(boatenv_t h, int64_t env_index, double *wv, double *wa, void *stream) {
    if (!h || !wv || !wa || env_index < 0 || env_index >= h->cfg.n_envs) return BOATENV_EINVAL;
    if (!h->was_reset) return BOATENV_ESTATE;
    GUARD_DEVICE(h);
    CUDA_TRY(launch_wind_table(h->cfg, env_index, wv, wa, (cudaStream_t)stream));
    return BOATENV_OK;
}

int boatenv_set_episode_draws(boatenv_t h, const int32_t *s_y_start, const double *knots, void *stream) {
    if (!h) return BOATENV_EINVAL;
    GUARD_DEVICE(h);
    cudaStream_t st = (cudaStream_t)stream;
    const size_t n = (size_t)h->cfg.n_envs;
    if (s_y_start) {
        if (!h->ovr_s_y) CUDA_TRY(cudaMalloc((void **)&h->ovr_s_y, n * sizeof(int32_t)));
        CUDA_TRY(cudaMemcpyAsync(h->ovr_s_y, s_y_start, n * sizeof(int32_t), cudaMemcpyDeviceToDevice, st));
        h->cfg.ovr_s_y = h->ovr_s_y;
    } else {
        h->cfg.ovr_s_y = nullptr;
    }
    if (knots) {
        const size_t cnt = n * 2 * (size_t)h->cfg.fp;
        if (!h->ovr_knots) CUDA_TRY(cudaMalloc((void **)&h->ovr_knots, cnt * sizeof(double)));
        CUDA_TRY(cudaMemcpyAsync(h->ovr_knots, knots, cnt * sizeof(double), cudaMemcpyDeviceToDevice, st));
        h->cfg.ovr_knots = h->ovr_knots;
    } else {
        h->cfg.ovr_knots = nullptr;
    }
    return BOATENV_OK;
}

int boatenv_episode_draws_host(const boatenv_params *params, uint64_t seed, int64_t global_env_id, uint32_t episode,
                               int32_t *s_y_start_out, double *knots_out) {
    if (!params || global_env_id < 0) return BOATENV_EINVAL;
    DevCfg c;
    int rc = derive_config(params, c);
    if (rc) return rc;
    if (s_y_start_out) *s_y_start_out = episode_s_y_start(seed, global_env_id, episode, c.s_y_half);
    if (knots_out)
        for (int t = 0; t < 2 * c.fp; ++t) knots_out[t] = (2 * c.fp <= 32) ? episode_knot(seed, global_env_id, episode, t) : 0.0;
    return BOATENV_OK;
}

int boatenv_episode_draws_batch_host(const boatenv_params *params, uint64_t seed, const int64_t *global_env_ids,
                                     int64_t n_ids, uint32_t episode_begin, int32_t n_episodes,
                                     int32_t *s_y_start_out, double *knots_out) {
    if (!params || !global_env_ids || n_ids < 0 || n_episodes < 0) return BOATENV_EINVAL;
    DevCfg c;
    int rc = derive_config(params, c);
    if (rc) return rc;
    if (2 * c.fp > 32) return BOATENV_EUNSUPPORTED;
    for (int32_t e = 0; e < n_episodes; ++e)
        for (int64_t j = 0; j < n_ids; ++j) {
            const int64_t g = global_env_ids[j];
            if (g < 0) return BOATENV_EINVAL;
            const size_t o = (size_t)e * (size_t)n_ids + (size_t)j;
            if (s_y_start_out) s_y_start_out[o] = episode_s_y_start(seed, g, episode_begin + (uint32_t)e, c.s_y_half);
            if (knots_out)
                for (int t = 0; t < 2 * c.fp; ++t)
                    knots_out[o * 2 * c.fp + t] = episode_knot(seed, g, episode_begin + (uint32_t)e, t);
        }
    return BOATENV_OK;
}

static size_t state_block_bytes(boatenv_t h) { return (size_t)num_blocks(h->cfg.n_envs) * (size_t)h->cfg.block_bytes; }
static size_t counter_bytes() { return (size_t)kCounterSlots * 32 * sizeof(double); }

int64_t boatenv_state_bytes(boatenv_t h) {
    return h ? (int64_t)(state_block_bytes(h) + counter_bytes()) : (int64_t)BOATENV_EINVAL;
}

int boatenv_export_state(boatenv_t h, void *blob_out, void *stream) {
    if (!h || !blob_out) return BOATENV_EINVAL;
    if (!h->was_reset) return BOATENV_ESTATE;
    GUARD_DEVICE(h);
    cudaStream_t st = (cudaStream_t)stream;
    CUDA_TRY(cudaMemcpyAsync(blob_out, h->cfg.state, state_block_bytes(h), cudaMemcpyDeviceToDevice, st));
    CUDA_TRY(cudaMemcpyAsync((char *)blob_out + state_block_bytes(h), h->cfg.counters, counter_bytes(),
                             cudaMemcpyDeviceToDevice, st));
    return BOATENV_OK;
}

int boatenv_import_state(boatenv_t h, const void *blob_in, void *stream) {
    if (!h || !blob_in) return BOATENV_EINVAL;
    GUARD_DEVICE(h);
    cudaStream_t st = (cudaStream_t)stream;
    CUDA_TRY(cudaMemcpyAsync(h->cfg.state, blob_in, state_block_bytes(h), cudaMemcpyDeviceToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(h->cfg.counters, (const char *)blob_in + state_block_bytes(h), counter_bytes(),
                             cudaMemcpyDeviceToDevice, st));
    h->was_reset = true;
    return BOATENV_OK;
}

int boatenv_reduce_counters(boatenv_t h, double *out_device, void *stream) {
    if (!h || !out_device) return BOATENV_EINVAL;
    GUARD_DEVICE(h);
    CUDA_TRY(launch_reduce_counters(h->cfg.counters, out_device, (cudaStream_t)stream));
    return BOATENV_OK;
}

int boatenv_get_counters(boatenv_t h, double *out_host, void *stream) {
    if (!h || !out_host) return BOATENV_EINVAL;
    GUARD_DEVICE(h);   // the copy and the synchronise below run on the handle's device too
    int rc = boatenv_reduce_counters(h, h->counters_out_dev, stream);
    if (rc) return rc;
    CUDA_TRY(cudaMemcpyAsync(out_host, h->counters_out_dev, kNumCounters * sizeof(double), cudaMemcpyDeviceToHost,
                             (cudaStream_t)stream));
    CUDA_TRY(cudaStreamSynchronize((cudaStream_t)stream));
    return BOATENV_OK;
}

int boatenv_fill_uniform_actions(boatenv_t h, uint64_t step_counter, double scale, void *actions_out, void *stream) {
    if (!h || !actions_out) return BOATENV_EINVAL;
    GUARD_DEVICE(h);
    CUDA_TRY(h->precision == 32 ? launch_fill_actions_f32(h->cfg, step_counter, scale, actions_out, (cudaStream_t)stream)
                                : launch_fill_actions_f64(h->cfg, step_counter, scale, actions_out, (cudaStream_t)stream));
    return BOATENV_OK;
}

}  // extern "C"

// the handle accessors of launch.h
namespace boatenv {
DevCfg *handle_cfg(boatenv_t h) { return &h->cfg; }
int handle_precision(boatenv_t h) { return h->precision; }
int handle_device(boatenv_t h) { return h->device; }
bool handle_was_reset(boatenv_t h) { return h->was_reset; }
int handle_next_parity(boatenv_t h) { return (int)(h->launch_parity++ & 1u); }
}  // namespace boatenv
