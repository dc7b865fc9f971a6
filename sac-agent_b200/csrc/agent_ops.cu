// agent_ops.cu -- the tanh-squashed Gaussian head of the reference's actor
// (networks/networks.py:47-70, ActorNetwork.sample_normal) as ONE kernel forward and ONE kernel
// backward.  In PyTorch the head is ~23 element-wise launches forward and ~35 backward on [B, n_actions]
// tensors -- 80 of the ~190 kernels of a captured SAC update, all launch-latency.  The formulas are in
// agent_math.cuh, shared with the fused learner (learner.cu).
#include <cstdint>
#include <cuda_runtime.h>

#include "../../include/boatenv.h"
#include "agent_math.cuh"
#include "launch.h"

namespace {

using boatenv::gaussian_head_bwd;
using boatenv::gaussian_head_fwd;

__global__ void __launch_bounds__(256) gaussian_head_fwd_kernel(const float *__restrict__ mean,
                                                                const float *__restrict__ raw_std,
                                                                const float *__restrict__ eps,
                                                                const float *__restrict__ max_action, long long rows,
                                                                int n_actions, float *__restrict__ action_out,
                                                                float *__restrict__ log_prob_out) {
    const long long b = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= rows) return;
    float lp = 0.0f;
    for (int a = 0; a < n_actions; ++a) {
        const long long i = b * n_actions + a;
        float act;
        lp += gaussian_head_fwd(mean[i], raw_std[i], eps[i], max_action[a], act);
        action_out[i] = act;
    }
    log_prob_out[b] = lp;
}

__global__ void __launch_bounds__(256) gaussian_head_bwd_kernel(
    const float *__restrict__ mean, const float *__restrict__ raw_std, const float *__restrict__ eps,
    const float *__restrict__ max_action, const float *__restrict__ grad_action /* may be null */,
    const float *__restrict__ grad_log_prob /* [rows], may be null */, long long rows, int n_actions,
    float *__restrict__ grad_mean, float *__restrict__ grad_raw_std) {
    const long long b = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= rows) return;
    const float glp = grad_log_prob ? grad_log_prob[b] : 0.0f;
    for (int a = 0; a < n_actions; ++a) {
        const long long i = b * n_actions + a;
        gaussian_head_bwd(mean[i], raw_std[i], eps[i], max_action[a], grad_action ? grad_action[i] : 0.0f, glp,
                          grad_mean[i], grad_raw_std[i]);
    }
}

}  // namespace

extern "C" {

int boatagent_gaussian_head_forward(const float *mean, const float *raw_std, const float *eps, const float *max_action,
                                    int64_t rows, int32_t n_actions, float *action_out, float *log_prob_out,
                                    void *stream) {
    if (!mean || !raw_std || !eps || !max_action || !action_out || !log_prob_out || rows <= 0 || n_actions <= 0)
        return BOATENV_EINVAL;
    gaussian_head_fwd_kernel<<<(unsigned)((rows + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
        mean, raw_std, eps, max_action, rows, n_actions, action_out, log_prob_out);
    boatenv::count_launch();
    return (int)cudaGetLastError();
}

int boatagent_gaussian_head_backward(const float *mean, const float *raw_std, const float *eps, const float *max_action,
                                     const float *grad_action, const float *grad_log_prob, int64_t rows,
                                     int32_t n_actions, float *grad_mean_out, float *grad_raw_std_out, void *stream) {
    if (!mean || !raw_std || !eps || !max_action || !grad_mean_out || !grad_raw_std_out || rows <= 0 || n_actions <= 0)
        return BOATENV_EINVAL;
    gaussian_head_bwd_kernel<<<(unsigned)((rows + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
        mean, raw_std, eps, max_action, grad_action, grad_log_prob, rows, n_actions, grad_mean_out, grad_raw_std_out);
    boatenv::count_launch();
    return (int)cudaGetLastError();
}

}  // extern "C"

// ---------------------------------------------------------------------------------
// Adam (torch.optim.Adam defaults, networks.py:31,88,121) for every network of the agent plus the
// Polyak average of the target value network (continuous_agent.py:66-80) in ONE launch.
// torch's multi-tensor Adam hands each CTA a 65536-element chunk: the agent's ~350 k parameters then
// run on a dozen CTAs (~70 us per optimiser, twice per update, plus two more launches for the Polyak
// average).  Here a CTA takes 2048 elements; the slot table travels as a kernel argument, so the launch
// captures into a CUDA graph as it is.
// ---------------------------------------------------------------------------------
namespace {

using boatenv::kAdamChunk;
using boatenv::kAdamThreads;
struct AdamTable {
    boatagent_adam_slot slot[BOATAGENT_ADAM_MAX_SLOTS];
    int n_slots;
    float beta1, beta2, eps, tau;
};

__global__ void __launch_bounds__(kAdamThreads) adam_polyak_kernel(const __grid_constant__ AdamTable tab,
                                                                   long long *__restrict__ state /* [step, ticket] */) {
    boatenv::adam_polyak_chunk(tab.slot, tab.n_slots, tab.beta1, tab.beta2, tab.eps, tab.tau, state, blockIdx.x,
                               gridDim.x, threadIdx.x);
}

}  // namespace

extern "C" int boatagent_adam_polyak_step(const boatagent_adam_slot *slots_host, int32_t n_slots, float beta1, float beta2,
                                          float eps, float tau, int64_t *state_dev, void *stream) {
    if (!slots_host || n_slots <= 0 || n_slots > BOATAGENT_ADAM_MAX_SLOTS || !state_dev) return BOATENV_EINVAL;
    AdamTable tab;
    long long chunks = 0;
    for (int k = 0; k < n_slots; ++k) {
        const boatagent_adam_slot &s = slots_host[k];
        if (!s.param || !s.grad || !s.exp_avg || !s.exp_avg_sq || s.numel <= 0) return BOATENV_EINVAL;
        tab.slot[k] = s;
        chunks += (s.numel + kAdamChunk - 1) / kAdamChunk;
    }
    tab.n_slots = n_slots;
    tab.beta1 = beta1;
    tab.beta2 = beta2;
    tab.eps = eps;
    tab.tau = tau;
    adam_polyak_kernel<<<(unsigned)chunks, kAdamThreads, 0, (cudaStream_t)stream>>>(tab, (long long *)state_dev);
    boatenv::count_launch();
    return (int)cudaGetLastError();
}
