// agent_math.cuh -- per-element formulas of the SAC update shared by the kernels that run them: the tanh-squashed
// Gaussian head of the actor (agent_ops.cu's head kernels and the fused learner, learner.cu) and the Adam + Polyak
// element update (agent_ops.cu's adam_polyak_kernel and the learner's second kernel).  One copy each, so the fused
// learner computes exactly what the fp32 learner's kernels compute.
//
//   t = tanh(raw_std);  log_std = -5 + 3.5 (t + 1);  std = exp(log_std)          (networks.py:53-56)
//   u = mean + eps * std                     (Normal.rsample / .sample, :60-63; eps ~ N(0, 1) supplied)
//   action = tanh(u) * max_action                                               (:65)
//   log_prob = sum_a [ -(u - mean)^2 / (2 std^2) - log_std - log sqrt(2 pi) - log(1 - action^2 + 1e-6) ]   (:66-68)
//
// Backward is for the reparameterised draw (u a function of mean and std).  The Gaussian term is then
// -eps^2 / 2 exactly: autograd's two paths into it cancel, so its gradient is 0 here.
#pragma once
#include <cuda_runtime.h>

#include "../../include/boatenv.h"

namespace boatenv {

constexpr float kLogStdMin = -5.0f, kLogStdHalfSpan = 3.5f;  // 0.5 * (LOG_STD_MAX - LOG_STD_MIN)
constexpr float kHalfLog2Pi = 0.91893853320467274178f;
constexpr float kReparamNoise = 1e-6f;

// One action dimension of the draw: writes the action, returns this dimension's log-probability term.
__device__ __forceinline__ float gaussian_head_fwd(float m, float raw_std, float e, float max_action, float &act_out) {
    const float log_std = kLogStdMin + kLogStdHalfSpan * (tanhf(raw_std) + 1.0f);
    const float sd = expf(log_std);
    const float u = m + e * sd;
    const float act = tanhf(u) * max_action;
    const float d = u - m;
    act_out = act;
    return -(d * d) / (2.0f * sd * sd) - log_std - kHalfLog2Pi - logf(1.0f - act * act + kReparamNoise);
}

// One action dimension of the backward pass: ga = dL/d action, glp = dL/d log_prob (the row's sum).
__device__ __forceinline__ void gaussian_head_bwd(float m, float raw_std, float e, float ma, float ga, float glp,
                                                  float &grad_mean, float &grad_raw_std) {
    const float t = tanhf(raw_std);
    const float dls = kLogStdHalfSpan * (1.0f - t * t);          // d log_std / d raw_std
    const float sd = expf(kLogStdMin + kLogStdHalfSpan * (t + 1.0f));
    const float th = tanhf(m + e * sd);
    const float act = th * ma;
    const float dact = ma * (1.0f - th * th);                      // d action / d u
    // d/du of -log(1 - action^2 + 1e-6) is 2 action dact / (1 - action^2 + 1e-6)
    const float gu = ga * dact + glp * (2.0f * act * dact) / (1.0f - act * act + kReparamNoise);
    grad_mean = gu;
    grad_raw_std = gu * e * sd * dls - glp * dls;                  // through std (u) and through -log_std
}

// torch.optim.Adam (defaults, foreach form) for element i of a slot with gradient g, then the Polyak average into the
// slot's target: step_size = lr / (1 - beta1^t), bc2_sqrt = sqrt(1 - beta2^t).
__device__ __forceinline__ void adam_polyak_element(const boatagent_adam_slot &sl, long long i, float g, float beta1,
                                                    float beta2, float eps, float tau, float step_size, float bc2_sqrt) {
    const float m = sl.exp_avg[i] + (g - sl.exp_avg[i]) * (1.0f - beta1);   // lerp_(grad, 1 - beta1)
    const float v = sl.exp_avg_sq[i] * beta2 + (1.0f - beta2) * g * g;     // mul_(beta2).addcmul_(g, g, 1 - beta2)
    const float denom = sqrtf(v) / bc2_sqrt + eps;
    const float p = sl.param[i] - step_size * (m / denom);                  // addcdiv_(m, denom, -step_size)
    sl.exp_avg[i] = m;
    sl.exp_avg_sq[i] = v;
    sl.param[i] = p;
    if (sl.target) sl.target[i] = tau * p + (1.0f - tau) * sl.target[i];
}

// Bias corrections of Adam step t (1-based), in double as torch computes them on the host.
__device__ __forceinline__ void adam_bias_corrections(long long t_steps, float beta1, float beta2, float &bc1,
                                                      float &bc2_sqrt) {
    const double t = (double)t_steps;
    bc1 = (float)(1.0 - pow((double)beta1, t));
    bc2_sqrt = (float)sqrt(1.0 - pow((double)beta2, t));
}

// The coalesced Adam + Polyak step of one agent's n_slots slots (agent_ops.cu's adam_polyak_kernel, and each member
// of learner.cu's adam_polyak_members_kernel): CTA `chunk` of the `n_ctas` CTAs that step the agent takes kAdamChunk
// consecutive elements of one slot (the slots' chunks in slot order), and the last of them to finish advances the step
// counter state[0] (state[1] is its ticket).
constexpr int kAdamChunk = 2048, kAdamThreads = 256;
__device__ __forceinline__ void adam_polyak_chunk(const boatagent_adam_slot *slot, int n_slots, float beta1,
                                                  float beta2, float eps, float tau, long long *__restrict__ state,
                                                  long long chunk, unsigned n_ctas, int tid) {
    __shared__ int s_slot;
    __shared__ long long s_first;
    __shared__ float s_bc1, s_bc2_sqrt;
    if (tid == 0) {
        int k = 0;
        for (; k < n_slots; ++k) {
            const long long nchunks = (slot[k].numel + kAdamChunk - 1) / kAdamChunk;
            if (chunk < nchunks) break;
            chunk -= nchunks;
        }
        s_slot = k;
        s_first = chunk * kAdamChunk;
        // this step's number
        adam_bias_corrections(*reinterpret_cast<volatile long long *>(state) + 1, beta1, beta2, s_bc1, s_bc2_sqrt);
    }
    __syncthreads();
    if (s_slot < n_slots) {
        const boatagent_adam_slot &sl = slot[s_slot];
        const float step_size = sl.lr / s_bc1;
        const long long end = min(s_first + (long long)kAdamChunk, (long long)sl.numel);
        for (long long i = s_first + tid; i < end; i += kAdamThreads) {
            adam_polyak_element(sl, i, sl.grad[i], beta1, beta2, eps, tau, step_size, s_bc2_sqrt);
        }
    }
    __syncthreads();
    if (tid == 0) {  // the last CTA to finish publishes the new step count
        __threadfence();
        const unsigned long long done = atomicAdd(reinterpret_cast<unsigned long long *>(state + 1), 1ULL) + 1ULL;
        if (done == n_ctas) {
            state[1] = 0;
            state[0] += 1;
        }
    }
}

}  // namespace boatenv
