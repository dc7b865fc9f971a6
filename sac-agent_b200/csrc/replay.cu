// replay.cu -- device-resident ReplayBuffer (agent/buffer.py:3-35): ring store,
// uniform-with-replacement sample-gather, the fused env.step + agent.remember
// launch (main.py:81-88) and the entry point of the fused act + step + remember
// collection kernel (rollout.cu).  Rows are kept exactly as the reference keeps them --
// five parallel arrays state[size][obs], new_state[size][obs], action[size][na],
// reward[size], terminal[size] -- so a sampled batch is five dense tensors the
// learner can consume without a transpose.
#include <algorithm>
#include <cstring>
#include <new>

#include "common.cuh"
#include "launch.h"

using namespace boatenv;

struct boatreplay_handle {
    void *state, *new_state, *action, *reward;
    uint8_t *terminal;
    long long mem_size, mem_cntr;
    int obs_dim, n_actions, precision, device;
    size_t esize;
};

namespace {

// store_transition (buffer.py:13-22) for a run of rows whose ring slots are CONTIGUOUS (the host splits
// a batch at the wrap point): five flat copies src[row0 ..] -> ring[slot0 ..].  128-bit path when source
// and destination of an array are both 16-byte aligned, scalar (still coalesced) otherwise.
template <typename T>
__device__ __forceinline__ void copy_flat(T *__restrict__ dst, const T *__restrict__ src, long long count, long long tid,
                                          long long nthreads) {
    using V = typename VecOf<T>::type;
    constexpr int W = VecOf<T>::W;
    if (((reinterpret_cast<uintptr_t>(dst) | reinterpret_cast<uintptr_t>(src)) & 15u) == 0) {
        const long long nvec = count / W;
        const V *sv = reinterpret_cast<const V *>(src);
        V *dv = reinterpret_cast<V *>(dst);
        long long v = tid;
#pragma unroll 1
        for (; v + 3 * nthreads < nvec; v += 4 * nthreads) {  // four independent 128-bit loads in flight per thread
            const V x0 = __ldcs(sv + v), x1 = __ldcs(sv + v + nthreads), x2 = __ldcs(sv + v + 2 * nthreads),
                    x3 = __ldcs(sv + v + 3 * nthreads);
            dv[v] = x0;
            dv[v + nthreads] = x1;
            dv[v + 2 * nthreads] = x2;
            dv[v + 3 * nthreads] = x3;
        }
        for (; v < nvec; v += nthreads) dv[v] = __ldcs(sv + v);
        for (long long e = nvec * W + tid; e < count; e += nthreads) dst[e] = src[e];
    } else {
        for (long long e = tid; e < count; e += nthreads) dst[e] = __ldcs(src + e);
    }
}

// blockIdx.y picks the array (0 state, 1 new_state, 2 action, 3 reward, 4 terminal): every CTA runs one
// flat copy loop, so the four loads in flight per thread cost a handful of registers.
template <typename T>
__global__ void __launch_bounds__(256) replay_store_kernel(
    T *__restrict__ state, T *__restrict__ new_state, T *__restrict__ action, T *__restrict__ reward,
    uint8_t *__restrict__ terminal, const T *__restrict__ s, const T *__restrict__ a, const T *__restrict__ r,
    const T *__restrict__ s2, const uint8_t *__restrict__ done, long long rows, long long row0, long long slot0,
    int obs_dim, int n_actions) {
    const long long tid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long nthreads = (long long)gridDim.x * blockDim.x;
    switch (blockIdx.y) {
    case 0: copy_flat<T>(state + slot0 * obs_dim, s + row0 * obs_dim, rows * obs_dim, tid, nthreads); break;
    case 1: copy_flat<T>(new_state + slot0 * obs_dim, s2 + row0 * obs_dim, rows * obs_dim, tid, nthreads); break;
    case 2: copy_flat<T>(action + slot0 * n_actions, a + row0 * n_actions, rows * n_actions, tid, nthreads); break;
    case 3: copy_flat<T>(reward + slot0, r + row0, rows, tid, nthreads); break;
    default:
        for (long long e = tid; e < rows; e += nthreads)
            terminal[slot0 + e] = done[row0 + e] ? 1 : 0;  // np.zeros(..., bool) storage (buffer.py:11,20)
    }
}

// np.random.choice(max_mem, batch) stand-in (buffer.py:27): draw b = word (b & 3) of
// Philox(counter = (b >> 2, sample counter), key = seed), reduced by multiply-shift.
__device__ __forceinline__ long long replay_index(unsigned long long seed, unsigned long long counter, long long b,
                                                  long long max_mem) {
    const unsigned long long blk = (unsigned long long)b >> 2;
    const Philox4 r = philox4x32_10((uint32_t)blk, (uint32_t)(blk >> 32), (uint32_t)counter,
                                    kStreamReplay | (uint32_t)((counter >> 32) & 0x0fffffffu), (uint32_t)seed,
                                    (uint32_t)(seed >> 32));
    const uint32_t w = philox_word(r, (int)(b & 3));
    return (long long)__umul64hi((unsigned long long)w << 32, (unsigned long long)max_mem);
}

// sample_buffer's gather (buffer.py:29-33).  A CTA serves kGatherRows consecutive output rows: it first
// puts their ring indices into shared memory (drawn in-kernel -- one Philox call per 4 rows -- or read
// from idx_in), then its threads walk the flat [rows][obs_dim] element range of state and new_state
// (consecutive threads = consecutive output elements: coalesced stores, row-contiguous loads) and the
// first threads move action / reward / done.
// USE_IDX: indices supplied by the caller; otherwise drawn in-kernel (and optionally exported).
// blockIdx.x / gridDim.x stride over ONE ring's batch (the population launch puts its members on blockIdx.y).
constexpr int kGatherRows = 128;
template <typename T, bool USE_IDX>
__device__ __forceinline__ void gather_rows(
    const T *__restrict__ state, const T *__restrict__ new_state, const T *__restrict__ action,
    const T *__restrict__ reward, const uint8_t *__restrict__ terminal, const long long *__restrict__ idx_in,
    long long *__restrict__ idx_out, T *__restrict__ s_out, T *__restrict__ a_out, T *__restrict__ r_out,
    T *__restrict__ s2_out, uint8_t *__restrict__ d_out, long long batch, long long max_mem, long long size,
    unsigned long long seed, unsigned long long counter, int obs_dim, int n_actions) {
    __shared__ long long jrow[kGatherRows];
    const int tid = threadIdx.x;
    for (long long row0 = (long long)blockIdx.x * kGatherRows; row0 < batch; row0 += (long long)gridDim.x * kGatherRows) {
        const int rows = (int)min((long long)kGatherRows, batch - row0);
        if (tid < rows) {
            const long long b = row0 + tid;
            long long j = USE_IDX ? idx_in[b] : replay_index(seed, counter, b, max_mem);
            if (USE_IDX && j < 0) j += size;  // numpy negative indexing
            if (!USE_IDX && idx_out) idx_out[b] = j;
            jrow[tid] = j;
        }
        __syncthreads();
        const int nelem = rows * obs_dim;
        T *so = s_out + row0 * obs_dim, *no = s2_out + row0 * obs_dim;
        for (int e = tid; e < nelem; e += 256) {
            const int r = e / obs_dim, col = e - r * obs_dim;
            const long long src = jrow[r] * obs_dim + col;
            so[e] = __ldg(state + src);
            no[e] = __ldg(new_state + src);
        }
        for (int e = tid; e < rows * n_actions; e += 256) {
            const int r = e / n_actions, col = e - r * n_actions;
            a_out[row0 * n_actions + e] = __ldg(action + jrow[r] * n_actions + col);
        }
        if (tid < rows) {
            r_out[row0 + tid] = __ldg(reward + jrow[tid]);
            d_out[row0 + tid] = terminal[jrow[tid]];
        }
        __syncthreads();  // jrow is reused by the next group of rows
    }
}

template <typename T, bool USE_IDX>
__global__ void __launch_bounds__(256) replay_gather_kernel(
    const T *__restrict__ state, const T *__restrict__ new_state, const T *__restrict__ action,
    const T *__restrict__ reward, const uint8_t *__restrict__ terminal, const long long *__restrict__ idx_in,
    long long *__restrict__ idx_out, T *__restrict__ s_out, T *__restrict__ a_out, T *__restrict__ r_out,
    T *__restrict__ s2_out, uint8_t *__restrict__ d_out, long long batch, long long max_mem, long long size,
    unsigned long long seed, unsigned long long counter, int obs_dim, int n_actions) {
    gather_rows<T, USE_IDX>(state, new_state, action, reward, terminal, idx_in, idx_out, s_out, a_out, r_out, s2_out,
                            d_out, batch, max_mem, size, seed, counter, obs_dim, n_actions);
}

// boatreplay_sample_members: one ring's in-kernel draw and gather per blockIdx.y
struct GatherMember {
    const void *state, *new_state, *action, *reward;
    const uint8_t *terminal;
    void *s_out, *a_out, *r_out, *s2_out;
    uint8_t *d_out;
    long long max_mem, size;
    unsigned long long seed, counter;
    int obs_dim, n_actions;
};
struct GatherMembers {
    GatherMember m[BOATAGENT_SAC_MAX_MEMBERS];
};

template <typename T>
__global__ void __launch_bounds__(256) replay_gather_members_kernel(const __grid_constant__ GatherMembers args,
                                                                    long long batch) {
    const GatherMember &g = args.m[blockIdx.y];
    gather_rows<T, false>((const T *)g.state, (const T *)g.new_state, (const T *)g.action, (const T *)g.reward,
                          g.terminal, nullptr, nullptr, (T *)g.s_out, (T *)g.a_out, (T *)g.r_out, (T *)g.s2_out, g.d_out,
                          batch, g.max_mem, g.size, g.seed, g.counter, g.obs_dim, g.n_actions);
}

template <typename T>
cudaError_t launch_store(boatreplay_t r, long long n, const void *s, const void *a, const void *rew, const void *s2,
                         const uint8_t *done, cudaStream_t st) {
    // rows older than the last mem_size are overwritten inside this very call: skip them; then split the
    // remaining run at the ring's wrap point so that every launch sees contiguous slots
    long long row0 = n > r->mem_size ? n - r->mem_size : 0;
    while (row0 < n) {
        const long long slot0 = (r->mem_cntr + row0) % r->mem_size;
        const long long rows = std::min(n - row0, r->mem_size - slot0);
        long long blocks = (rows * r->obs_dim / 4 + 255) / 256;
        blocks = std::max(1LL, std::min(blocks, 148LL * 8));
        replay_store_kernel<T><<<dim3((unsigned)blocks, 5), 256, 0, st>>>(
            (T *)r->state, (T *)r->new_state, (T *)r->action, (T *)r->reward, r->terminal, (const T *)s, (const T *)a,
            (const T *)rew, (const T *)s2, done, rows, row0, slot0, r->obs_dim, r->n_actions);
        count_launch();
        cudaError_t e = cudaGetLastError();
        if (e != cudaSuccess) return e;
        row0 += rows;
    }
    return cudaSuccess;
}

template <typename T>
cudaError_t launch_gather(boatreplay_t r, long long batch, const long long *idx_in, long long *idx_out,
                          unsigned long long seed, unsigned long long counter, void *s_out, void *a_out, void *r_out,
                          void *s2_out, uint8_t *d_out, cudaStream_t st) {
    const long long max_mem = r->mem_cntr < r->mem_size ? r->mem_cntr : r->mem_size;
    long long blocks = (batch + kGatherRows - 1) / kGatherRows;
    blocks = std::max(1LL, std::min(blocks, 148LL * 32));
    if (idx_in)
        replay_gather_kernel<T, true><<<(unsigned)blocks, 256, 0, st>>>(
            (const T *)r->state, (const T *)r->new_state, (const T *)r->action, (const T *)r->reward, r->terminal,
            idx_in, nullptr, (T *)s_out, (T *)a_out, (T *)r_out, (T *)s2_out, d_out, batch, max_mem, r->mem_size, seed,
            counter, r->obs_dim, r->n_actions);
    else
        replay_gather_kernel<T, false><<<(unsigned)blocks, 256, 0, st>>>(
            (const T *)r->state, (const T *)r->new_state, (const T *)r->action, (const T *)r->reward, r->terminal,
            nullptr, idx_out, (T *)s_out, (T *)a_out, (T *)r_out, (T *)s2_out, d_out, batch, max_mem, r->mem_size, seed,
            counter, r->obs_dim, r->n_actions);
    count_launch();
    return cudaGetLastError();
}

}  // namespace

extern "C" {

int boatreplay_create(int64_t max_size, int32_t obs_dim, int32_t n_actions, int precision, int device,
                      boatreplay_t *out) {
    if (!out || max_size <= 0 || obs_dim <= 0 || n_actions <= 0) return BOATENV_EINVAL;
    if (precision != 32 && precision != 64) return BOATENV_EINVAL;
    *out = nullptr;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0 || device < 0 || device >= ndev) return BOATENV_ENODEVICE;
    boatenv::DeviceGuard _guard(device);
    if (!_guard.ok()) return (int)_guard.error();
    boatreplay_handle *r = new (std::nothrow) boatreplay_handle();
    if (!r) return BOATENV_EINVAL;
    std::memset(r, 0, sizeof(*r));
    r->mem_size = max_size;
    r->obs_dim = obs_dim;
    r->n_actions = n_actions;
    r->precision = precision;
    r->device = device;
    r->esize = precision == 32 ? 4 : 8;
    const size_t n = (size_t)max_size;
    cudaError_t e = cudaSuccess;
    auto alloc = [&](void **p, size_t bytes) {  // np.zeros(...)  buffer.py:7-11
        if (e == cudaSuccess) e = cudaMalloc(p, bytes);
        if (e == cudaSuccess) e = cudaMemset(*p, 0, bytes);
    };
    alloc(&r->state, n * obs_dim * r->esize);
    alloc(&r->new_state, n * obs_dim * r->esize);
    alloc(&r->action, n * n_actions * r->esize);
    alloc(&r->reward, n * r->esize);
    alloc((void **)&r->terminal, n);
    if (e != cudaSuccess) {
        boatreplay_destroy(r);
        return (int)e;
    }
    *out = r;
    return BOATENV_OK;
}

int boatreplay_destroy(boatreplay_t r) {
    if (!r) return BOATENV_EINVAL;
    boatenv::DeviceGuard _guard(r->device);
    cudaFree(r->state);
    cudaFree(r->new_state);
    cudaFree(r->action);
    cudaFree(r->reward);
    cudaFree(r->terminal);
    delete r;
    return BOATENV_OK;
}

int boatreplay_store(boatreplay_t r, int64_t n, const void *s, const void *a, const void *rew, const void *s2,
                     const uint8_t *done, void *stream) {
    if (!r || n < 0 || !s || !a || !rew || !s2 || !done) return BOATENV_EINVAL;
    if (n == 0) return BOATENV_OK;
    GUARD_DEVICE(r);
    CUDA_TRY(r->precision == 32 ? launch_store<float>(r, n, s, a, rew, s2, done, (cudaStream_t)stream)
                                : launch_store<double>(r, n, s, a, rew, s2, done, (cudaStream_t)stream));
    r->mem_cntr += n;  // buffer.py:22
    return BOATENV_OK;
}

int boatreplay_sample(boatreplay_t r, int64_t batch, uint64_t seed, uint64_t counter, void *s_out, void *a_out,
                      void *r_out, void *s2_out, uint8_t *done_out, int64_t *idx_out, void *stream) {
    if (!r || batch <= 0 || !s_out || !a_out || !r_out || !s2_out || !done_out) return BOATENV_EINVAL;
    if (r->mem_cntr <= 0) return BOATENV_ESTATE;  // np.random.choice(0, n) raises ValueError
    GUARD_DEVICE(r);
    CUDA_TRY(r->precision == 32
                 ? launch_gather<float>(r, batch, nullptr, (long long *)idx_out, seed, counter, s_out, a_out, r_out,
                                        s2_out, done_out, (cudaStream_t)stream)
                 : launch_gather<double>(r, batch, nullptr, (long long *)idx_out, seed, counter, s_out, a_out, r_out,
                                         s2_out, done_out, (cudaStream_t)stream));
    return BOATENV_OK;
}

int boatreplay_sample_members(const boatreplay_sample_member *members_host, int32_t n_members, int64_t batch,
                              void *stream) {
    if (!members_host || n_members < 1 || n_members > BOATAGENT_SAC_MAX_MEMBERS || batch <= 0) return BOATENV_EINVAL;
    const boatreplay_t r0 = members_host[0].ring;
    if (!r0) return BOATENV_EINVAL;
    GatherMembers a;
    std::memset(&a, 0, sizeof(a));
    for (int m = 0; m < n_members; ++m) {
        const boatreplay_sample_member &e = members_host[m];
        const boatreplay_t r = e.ring;
        if (!r || !e.s_out || !e.a_out || !e.r_out || !e.s2_out || !e.done_out) return BOATENV_EINVAL;
        if (r->precision != r0->precision || r->device != r0->device) return BOATENV_EINVAL;
        if (r->mem_cntr <= 0) return BOATENV_ESTATE;
        GatherMember &g = a.m[m];
        g.state = r->state;
        g.new_state = r->new_state;
        g.action = r->action;
        g.reward = r->reward;
        g.terminal = r->terminal;
        g.s_out = e.s_out;
        g.a_out = e.a_out;
        g.r_out = e.r_out;
        g.s2_out = e.s2_out;
        g.d_out = e.done_out;
        g.max_mem = r->mem_cntr < r->mem_size ? r->mem_cntr : r->mem_size;
        g.size = r->mem_size;
        g.seed = e.seed;
        g.counter = e.counter;
        g.obs_dim = r->obs_dim;
        g.n_actions = r->n_actions;
    }
    GUARD_DEVICE(r0);
    long long blocks = (batch + kGatherRows - 1) / kGatherRows;
    blocks = std::max(1LL, std::min(blocks, 148LL * 32));
    const dim3 grid((unsigned)blocks, (unsigned)n_members);
    if (r0->precision == 32)
        replay_gather_members_kernel<float><<<grid, 256, 0, (cudaStream_t)stream>>>(a, batch);
    else
        replay_gather_members_kernel<double><<<grid, 256, 0, (cudaStream_t)stream>>>(a, batch);
    count_launch();
    CUDA_TRY(cudaGetLastError());
    return BOATENV_OK;
}

int boatreplay_gather(boatreplay_t r, int64_t batch, const int64_t *idx, void *s_out, void *a_out, void *r_out,
                      void *s2_out, uint8_t *done_out, void *stream) {
    if (!r || batch <= 0 || !idx || !s_out || !a_out || !r_out || !s2_out || !done_out) return BOATENV_EINVAL;
    GUARD_DEVICE(r);
    CUDA_TRY(r->precision == 32 ? launch_gather<float>(r, batch, (const long long *)idx, nullptr, 0, 0, s_out, a_out,
                                                       r_out, s2_out, done_out, (cudaStream_t)stream)
                                : launch_gather<double>(r, batch, (const long long *)idx, nullptr, 0, 0, s_out, a_out,
                                                        r_out, s2_out, done_out, (cudaStream_t)stream));
    return BOATENV_OK;
}

int boatreplay_set_mem_cntr(boatreplay_t r, int64_t mem_cntr) {
    if (!r || mem_cntr < 0) return BOATENV_EINVAL;
    r->mem_cntr = mem_cntr;
    return BOATENV_OK;
}
int64_t boatreplay_mem_cntr(boatreplay_t r) { return r ? r->mem_cntr : BOATENV_EINVAL; }
int64_t boatreplay_mem_size(boatreplay_t r) { return r ? r->mem_size : BOATENV_EINVAL; }

int boatenv_step_store(boatenv_t h, boatreplay_t r, const void *actions, void *obs_inout, void *reward_out,
                       uint8_t *done_out, uint8_t *term_out, int done_flag_mode, uint32_t flags, void *stream) {
    if (!h || !r || !actions || !obs_inout || !reward_out || (!done_out && !term_out)) return BOATENV_EINVAL;
    if (!handle_was_reset(h)) return BOATENV_ESTATE;
    const DevCfg &c = *handle_cfg(h);
    if (handle_precision(h) != r->precision || handle_device(h) != r->device || r->obs_dim != kObsDim ||
        r->n_actions != 1)
        return BOATENV_EINVAL;
    if (c.n_envs > r->mem_size) return BOATENV_EUNSUPPORTED;  // a step must not lap the ring
    if ((reinterpret_cast<uintptr_t>(obs_inout) & 15u) != 0) return BOATENV_EALIGN;
    GUARD_DEVICE(r);
    StepArgs a;
    std::memset(&a, 0, sizeof(a));
    a.env_begin = 0;
    a.env_end = c.n_envs;
    a.actions = actions;
    a.ksteps = 1;
    a.obs_out = obs_inout;
    a.obs_in = obs_inout;
    a.reward_out = reward_out;
    a.done_out = done_out;
    a.term_out = term_out;
    a.flags = flags;
    a.rp.state = r->state;
    a.rp.new_state = r->new_state;
    a.rp.action = r->action;
    a.rp.reward = r->reward;
    a.rp.terminal = r->terminal;
    a.rp.mem_size = r->mem_size;
    a.rp.base_slot = r->mem_cntr % r->mem_size;
    a.rp.done_flag_mode = done_flag_mode;
    a.reverse = boatenv::handle_next_parity(h);
    CUDA_TRY(r->precision == 32 ? launch_step_f32(c, a, (cudaStream_t)stream)
                                : launch_step_f64(c, a, (cudaStream_t)stream));
    r->mem_cntr += c.n_envs;
    return BOATENV_OK;
}


// boatagent_collect, and boatagent_collect_record with rec_ids != NULL (its own arguments checked by the caller)
static int collect(boatenv_t h, boatreplay_t r, const void *weight_blob, const float *max_action, uint64_t seed,
                   uint64_t step0, int32_t steps, int done_flag_mode, float *obs_inout, float *reward_out,
                   uint8_t *done_out, uint8_t *term_out, const int64_t *rec_ids, int64_t rec_n_ids,
                   const boatenv_record_ring *rec_ring, int64_t rec_row, void *stream) {
    if (!h || !r || !weight_blob || !max_action || !obs_inout || !reward_out || (!done_out && !term_out) || steps < 1 ||
        (done_flag_mode != 0 && done_flag_mode != 1))
        return BOATENV_EINVAL;
    if (handle_precision(h) != 32 || r->precision != 32 || r->obs_dim != kObsDim || r->n_actions != 1)
        return BOATENV_EUNSUPPORTED;
    if (!handle_was_reset(h)) return BOATENV_ESTATE;
    const DevCfg &c = *handle_cfg(h);
    // tiles advance at different rates: two rows of one call in the same slot would race
    if (handle_device(h) != r->device || (long long)steps * c.n_envs > r->mem_size) return BOATENV_EINVAL;
    if ((reinterpret_cast<uintptr_t>(weight_blob) & 15u) != 0) return BOATENV_EALIGN;
    GUARD_DEVICE(r);
    CollectArgs a;
    std::memset(&a, 0, sizeof(a));
    a.blob = static_cast<const unsigned char *>(weight_blob);
    a.max_action = max_action;
    a.seed = seed;
    a.step0 = step0;
    a.steps = steps;
    a.obs_inout = obs_inout;
    a.reward_out = reward_out;
    a.done_out = done_out;
    a.term_out = term_out;
    a.rp.state = r->state;
    a.rp.new_state = r->new_state;
    a.rp.action = r->action;
    a.rp.reward = r->reward;
    a.rp.terminal = r->terminal;
    a.rp.mem_size = r->mem_size;
    a.rp.base_slot = r->mem_cntr % r->mem_size;
    a.rp.done_flag_mode = done_flag_mode;
    if (rec_ids) {
        a.rec_ids = (const long long *)rec_ids;
        a.rec_n_ids = (int)rec_n_ids;
        a.rec_ring = *rec_ring;
        a.rec_row0 = rec_row % rec_ring->capacity;
    }
    CUDA_TRY(launch_collect(c, a, (cudaStream_t)stream));
    r->mem_cntr += (long long)steps * c.n_envs;
    return BOATENV_OK;
}

int boatagent_collect(boatenv_t h, boatreplay_t r, const void *weight_blob, const float *max_action, uint64_t seed,
                      uint64_t step0, int32_t steps, int done_flag_mode, float *obs_inout, float *reward_out,
                      uint8_t *done_out, uint8_t *term_out, void *stream) {
    return collect(h, r, weight_blob, max_action, seed, step0, steps, done_flag_mode, obs_inout, reward_out, done_out,
                   term_out, nullptr, 0, nullptr, 0, stream);
}

int boatagent_collect_record(boatenv_t h, boatreplay_t r, const void *weight_blob, const float *max_action,
                             uint64_t seed, uint64_t step0, int32_t steps, int done_flag_mode, float *obs_inout,
                             float *reward_out, uint8_t *done_out, uint8_t *term_out, const int64_t *ids,
                             int64_t n_ids, const boatenv_record_ring *ring, int64_t row, void *stream) {
    if (!ids || n_ids <= 0 || n_ids > 2147483647LL || !ring || row < 0) return BOATENV_EINVAL;
    if (!ring->s_x || !ring->s_y || !ring->v_x || !ring->v_y || !ring->s_r || !ring->rudder_angle || !ring->action ||
        !ring->reward || !ring->term || !ring->episode || ring->capacity <= 0)
        return BOATENV_EINVAL;
    if (steps > ring->capacity) return BOATENV_EINVAL;   // one call would overwrite its own rows
    return collect(h, r, weight_blob, max_action, seed, step0, steps, done_flag_mode, obs_inout, reward_out, done_out,
                   term_out, ids, n_ids, ring, row, stream);
}

}  // extern "C"
