// launch.h -- declarations shared by the translation units of libboatenv: the launcher prototypes of the
// per-precision units (step_f32.cu, step_f64.cu), the env-handle accessors (abi.cu) and CUDA_TRY.
#pragma once
#include "common.cuh"

// Every handle-based entry point runs on the handle's device and restores the caller's current device on return
// (a multi-GPU process keeps torch's current device untouched).
namespace boatenv {
class DeviceGuard {
public:
    explicit DeviceGuard(int device) : prev_(-1), err_(cudaSuccess) {
        err_ = cudaGetDevice(&prev_);
        if (err_ == cudaSuccess && prev_ != device) err_ = cudaSetDevice(device); else if (err_ == cudaSuccess) prev_ = -1;
    }
    ~DeviceGuard() { if (prev_ >= 0) cudaSetDevice(prev_); }
    bool ok() const { return err_ == cudaSuccess; }
    cudaError_t error() const { return err_; }
    DeviceGuard(const DeviceGuard &) = delete;
    DeviceGuard &operator=(const DeviceGuard &) = delete;
private:
    int prev_;
    cudaError_t err_;
};
}  // namespace boatenv
#define GUARD_DEVICE(h)                                   \
    boatenv::DeviceGuard _guard((h)->device);                      \
    if (!_guard.ok()) return (int)_guard.error()

// In an int-returning entry point: return a CUDA call's error code unless it succeeded.
#define CUDA_TRY(expr)                                  \
    do {                                                \
        cudaError_t _e = (expr);                        \
        if (_e != cudaSuccess) return (int)_e;          \
    } while (0)

namespace boatenv {

void count_launch();

// Access to an env handle from the other translation units (the handle is defined in abi.cu).
DevCfg *handle_cfg(boatenv_t h);
int handle_precision(boatenv_t h);
int handle_device(boatenv_t h);
bool handle_was_reset(boatenv_t h);
int handle_next_parity(boatenv_t h);   // the sweep direction of the next step launch (alternates)

cudaError_t launch_step_f32(const DevCfg &, const StepArgs &, cudaStream_t);
cudaError_t launch_step_f64(const DevCfg &, const StepArgs &, cudaStream_t);
cudaError_t launch_reset_f32(const DevCfg &, const uint8_t *mask, void *obs_out, cudaStream_t);
cudaError_t launch_reset_f64(const DevCfg &, const uint8_t *mask, void *obs_out, cudaStream_t);
cudaError_t launch_get_field_f32(const DevCfg &, int field, void *out, cudaStream_t);
cudaError_t launch_get_field_f64(const DevCfg &, int field, void *out, cudaStream_t);
cudaError_t launch_set_field_f32(const DevCfg &, int field, const void *in, cudaStream_t);
cudaError_t launch_set_field_f64(const DevCfg &, int field, const void *in, cudaStream_t);
cudaError_t launch_fill_actions_f32(const DevCfg &, unsigned long long step_counter, double scale, void *out,
                                    cudaStream_t);
cudaError_t launch_fill_actions_f64(const DevCfg &, unsigned long long step_counter, double scale, void *out,
                                    cudaStream_t);
cudaError_t launch_env_state_f32(const DevCfg &, long long env, double *out, cudaStream_t);
cudaError_t launch_env_state_f64(const DevCfg &, long long env, double *out, cudaStream_t);
cudaError_t launch_wind_table(const DevCfg &, long long env, double *wv, double *wa, cudaStream_t);
cudaError_t launch_reduce_counters(const double *counters, double *out, cudaStream_t);

// boatagent_collect / boatagent_collect_record (replay.cu checks the arguments, rollout.cu holds the kernel): T steps
// of policy, env step with auto-reset and replay store, fused
struct CollectArgs {
    const unsigned char *blob;
    const float *max_action;
    unsigned long long seed, step0;
    int steps;
    float *obs_inout, *reward_out;
    uint8_t *done_out, *term_out;   // either may be NULL
    ReplayView rp;
    // recording (boatagent_collect_record only; rec_ids == NULL: plain collection).  Appended, so that the fields
    // above keep their parameter offsets.  Step t's row goes to row (rec_row0 + t) % rec_ring.capacity, with
    // 0 <= rec_row0 < capacity and T <= capacity.
    const long long *rec_ids;
    int rec_n_ids;
    boatenv_record_ring rec_ring;
    long long rec_row0;
};
cudaError_t launch_collect(const DevCfg &, const CollectArgs &, cudaStream_t);

}  // namespace boatenv
