// record.cu -- the device side of the episode recorder (postprocessing/recorder.py:18-56): after a step,
// one small launch copies the recorded envs' state and the step's action / reward / termination into a
// caller-owned ring; nothing crosses to the host until the caller flushes the ring.
#include "aux_kernels.cuh"
#include "launch.h"

using namespace boatenv;

namespace boatenv {
constexpr int kRecordBlock = 128;

// One thread per recorded env.  The state is decoded by read_field, the same decode boat_get_field_kernel
// uses, so every column equals what get_field returns for that env (fixed-point rudder / positions included).
template <typename T>
__global__ void __launch_bounds__(kRecordBlock) boat_record_kernel(const __grid_constant__ DevCfg c,
                                                                  const long long *__restrict__ ids, int n_ids,
                                                                  const T *__restrict__ actions,
                                                                  const T *__restrict__ reward,
                                                                  const uint8_t *__restrict__ term,
                                                                  const boatenv_record_ring ring, long long slot) {
    const int j = (int)blockIdx.x * kRecordBlock + (int)threadIdx.x;
    if (j >= n_ids) return;
    const long long i = __ldg(ids + j);
    if (i < 0 || i >= c.n_envs) return;
    const long long o = slot * n_ids + j;
    static_cast<T *>(ring.s_x)[o] = (T)read_field(c, i, D_SX, T());
    static_cast<T *>(ring.s_y)[o] = (T)read_field(c, i, D_SY, T());
    static_cast<T *>(ring.v_x)[o] = (T)read_field(c, i, D_VX, T());
    static_cast<T *>(ring.v_y)[o] = (T)read_field(c, i, D_VY, T());
    static_cast<T *>(ring.s_r)[o] = (T)read_field(c, i, D_SR, T());
    static_cast<T *>(ring.rudder_angle)[o] = (T)read_field(c, i, D_RUDDER, T());
    static_cast<T *>(ring.action)[o] = actions ? actions[i] : T(0);
    static_cast<T *>(ring.reward)[o] = reward ? reward[i] : T(0);
    ring.term[o] = term ? term[i] : (uint8_t)0;
    ring.episode[o] = *episode_ptr(c, i);
}

template <typename T>
cudaError_t launch_record(const DevCfg &c, const long long *ids, int n_ids, const void *actions, const void *reward,
                          const uint8_t *term, const boatenv_record_ring &ring, long long slot, cudaStream_t st) {
    boat_record_kernel<T><<<(unsigned)((n_ids + kRecordBlock - 1) / kRecordBlock), kRecordBlock, 0, st>>>(
        c, ids, n_ids, static_cast<const T *>(actions), static_cast<const T *>(reward), term, ring, slot);
    count_launch();
    return cudaGetLastError();
}

}  // namespace boatenv

extern "C" {

int boatenv_record_rows(boatenv_t h, const int64_t *ids, int64_t n_ids, const void *actions, const void *reward,
                        const uint8_t *term, const boatenv_record_ring *ring, int64_t row, void *stream) {
    if (!h || !ids || n_ids <= 0 || n_ids > 2147483647LL || !ring || row < 0) return BOATENV_EINVAL;
    if (!ring->s_x || !ring->s_y || !ring->v_x || !ring->v_y || !ring->s_r || !ring->rudder_angle || !ring->action ||
        !ring->reward || !ring->term || !ring->episode || ring->capacity <= 0)
        return BOATENV_EINVAL;
    if (!handle_was_reset(h)) return BOATENV_ESTATE;
    boatenv::DeviceGuard _guard(handle_device(h));
    if (!_guard.ok()) return (int)_guard.error();
    const DevCfg &c = *handle_cfg(h);
    const long long slot = row % ring->capacity;
    const cudaError_t e =
        handle_precision(h) == 32
            ? launch_record<float>(c, (const long long *)ids, (int)n_ids, actions, reward, term, *ring, slot,
                                   (cudaStream_t)stream)
            : launch_record<double>(c, (const long long *)ids, (int)n_ids, actions, reward, term, *ring, slot,
                                    (cudaStream_t)stream);
    return e == cudaSuccess ? BOATENV_OK : (int)e;
}

}  // extern "C"
