// priority.cu -- prioritized experience replay (Schaul et al. 2016) over one replay ring: a sum tree of the slots'
// priorities, stratified sampling with importance weights, and the priority update from the learner's TD errors.
//
// Tree: level 0 holds one fp32 priority per slot (0 for a slot never written); level k >= 1 holds fp64 sums of
// kFan = 1024 consecutive entries of level k - 1, up to a level of one entry, the total.  Every level is allocated
// in whole blocks of kFan entries, zero padded, so no kernel needs a bounds check inside a block.  A block is summed
// by one warp in one fixed order (block_sum), and no float atomics are used, so a tree is bit-reproducible and a
// host restatement (tests/test_prioritized_replay.py) repeats it exactly.
//
// The ring and its store / step-store / collect kernels know nothing of priorities: the host fills the slots written
// since the last sample with max_priority (boatper_fill_new) before it draws.
#include <algorithm>
#include <cfloat>
#include <cstring>
#include <new>

#include "common.cuh"
#include "launch.h"

using namespace boatenv;

namespace {

constexpr int kFan = 1024, kFanLog = 10, kMaxLevels = 6, kPerThreads = 256;

}  // namespace

struct boatper_handle {
    float *leaves;                   // level 0: [blocks(count[0]) * kFan]
    double *sums[kMaxLevels];        // levels 1 .. n_levels - 1 (sums[0] unused)
    long long count[kMaxLevels];     // entries per level; count[n_levels - 1] == 1
    int n_levels, device;
    float *max_priority;             // device scalar, starts at 1
    unsigned *min_bits;              // scratch of boatper_sample: the smallest drawn priority (fp32 bits)
    int *bad;                        // set by boatper_update for an index outside the ring or a bad TD error
    long long mem_size, filled;      // filled: slots ever given a priority (<= mem_size)
};

namespace {

struct PerTree {
    const float *leaves;
    const double *sums[kMaxLevels];
    int n_levels;
};

// inclusive prefix sum over the lanes, lane l adding lane l - o's value for o = 1, 2, 4, 8, 16
__device__ __forceinline__ double warp_scan(double v, int lane) {
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const double u = __shfl_up_sync(0xffffffffu, v, o);
        if (lane >= o) v = v + u;
    }
    return v;
}

// lane l's chunk of a block: entries 32 l .. 32 l + 31, summed in order in fp64
__device__ __forceinline__ double chunk_sum(const float *p) {
    double s = 0.0;
    const float4 *q = reinterpret_cast<const float4 *>(p);
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        const float4 x = q[i];
        s += (double)x.x;
        s += (double)x.y;
        s += (double)x.z;
        s += (double)x.w;
    }
    return s;
}
__device__ __forceinline__ double chunk_sum(const double *p) {
    double s = 0.0;
    const double2 *q = reinterpret_cast<const double2 *>(p);
#pragma unroll
    for (int i = 0; i < 16; ++i) {
        const double2 x = q[i];
        s += x.x;
        s += x.y;
    }
    return s;
}

// the sum of one block of kFan entries: each lane's chunk in order, then the warp scan; lane 31 holds it
template <typename T>
__device__ __forceinline__ double block_sum(const T *blk, int lane) {
    return warp_scan(chunk_sum(blk + 32 * lane), lane);
}

// first lane with a non-zero share whose inclusive prefix exceeds t; where rounding leaves none, the last lane with a
// non-zero share (for t >= 0 a zero share never comes first: its prefix equals the one before it)
__device__ __forceinline__ int pick_lane(double t, double incl, double own) {
    const unsigned nz = __ballot_sync(0xffffffffu, own > 0.0), hit = __ballot_sync(0xffffffffu, t < incl) & nz;
    return hit ? __ffs(hit) - 1 : (nz ? 31 - __clz(nz) : 0);
}

// Descends one block: the chunk whose prefix range holds t, then the entry within it.  t leaves as the residual
// inside the chosen entry.  Never returns an entry of zero priority while the block has a non-zero one.
template <typename T>
__device__ __forceinline__ int descend(const T *blk, double &t, int lane) {
    const double c = chunk_sum(blk + 32 * lane), S = warp_scan(c, lane);
    const double Su = __shfl_up_sync(0xffffffffu, S, 1);   // lane l > 0: the prefix before chunk l
    const int L = pick_lane(t, S, c);
    t = t - (L ? __shfl_sync(0xffffffffu, Su, L) : 0.0);
    const double v = (double)blk[32 * L + lane], V = warp_scan(v, lane);
    const double Vu = __shfl_up_sync(0xffffffffu, V, 1);
    const int I = pick_lane(t, V, v);
    t = t - (I ? __shfl_sync(0xffffffffu, Vu, I) : 0.0);
    return 32 * L + I;
}

// Level sums of the blocks that hold changed entries: warp w recomputes parent block idx[w] >> shift (idx != NULL;
// indices outside the ring are skipped) or b0 + w.  Two warps may recompute one block: they write the same value.
template <typename T>
__global__ void __launch_bounds__(kPerThreads) per_sum_kernel(const T *__restrict__ child, double *__restrict__ parent,
                                                              const long long *__restrict__ idx, long long n, int shift,
                                                              long long b0, long long mem_size) {
    const long long w = ((long long)blockIdx.x * kPerThreads + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (w >= n) return;   // whole warps
    long long b;
    if (idx) {
        const long long j = idx[w];
        if (j < 0 || j >= mem_size) return;
        b = j >> shift;
    } else {
        b = b0 + w;
    }
    const double s = block_sum(child + b * kFan, lane);
    if (lane == 31) parent[b] = s;
}

__global__ void __launch_bounds__(kPerThreads) per_fill_kernel(float *__restrict__ leaves,
                                                               const float *__restrict__ max_priority, long long slot0,
                                                               long long n) {
    const float p = *max_priority;
    for (long long i = (long long)blockIdx.x * kPerThreads + threadIdx.x; i < n; i += (long long)gridDim.x * kPerThreads)
        leaves[slot0 + i] = p;
}

// The new priority of batch row j, or -1 for a row that must not be applied (index outside the ring, a TD error that
// is negative or NaN -- td holds absolute errors -- or a priority that is not finite): the row is flagged.
__device__ __forceinline__ float row_priority(const long long *idx, const float *td, long long j, long long mem_size,
                                              double alpha, float eps, int *bad) {
    const long long i = idx[j];
    const float d = td[j];
    const float p = (float)pow((double)(d + eps), alpha);
    if (i < 0 || i >= mem_size || !(d >= 0.f) || !(p >= 0.f && p <= FLT_MAX)) {
        *bad = 1;
        return -1.f;
    }
    return p;
}

// update, pass 1: the leaves of the batch's slots to 0, so that pass 2's maximum sees only this batch's rows
__global__ void __launch_bounds__(kPerThreads) per_clear_kernel(float *__restrict__ leaves,
                                                                const long long *__restrict__ idx,
                                                                const float *__restrict__ td, long long batch,
                                                                long long mem_size, double alpha, float eps, int *bad) {
    for (long long j = (long long)blockIdx.x * kPerThreads + threadIdx.x; j < batch; j += (long long)gridDim.x * kPerThreads)
        if (row_priority(idx, td, j, mem_size, alpha, eps, bad) >= 0.f) leaves[idx[j]] = 0.f;
}

// update, pass 2: leaf idx[j] = max over the batch rows j that drew it of (td[j] + eps)^alpha, and max_priority up
// to the batch maximum: atomicMax on the bit patterns of non-negative floats, which order as the values do
__global__ void __launch_bounds__(kPerThreads) per_raise_kernel(float *__restrict__ leaves,
                                                                const long long *__restrict__ idx,
                                                                const float *__restrict__ td, long long batch,
                                                                long long mem_size, double alpha, float eps, int *bad,
                                                                float *max_priority) {
    for (long long j0 = (long long)blockIdx.x * kPerThreads; j0 < batch; j0 += (long long)gridDim.x * kPerThreads) {
        const long long j = j0 + threadIdx.x;
        const float p = j < batch ? row_priority(idx, td, j, mem_size, alpha, eps, bad) : -1.f;
        if (p >= 0.f) atomicMax(reinterpret_cast<int *>(leaves + idx[j]), __float_as_int(p));
        const unsigned m = __reduce_max_sync(0xffffffffu, p >= 0.f ? __float_as_uint(p) : 0u);
        if ((threadIdx.x & 31) == 0 && m) atomicMax(reinterpret_cast<int *>(max_priority), (int)m);
    }
}

// Stratified draw of batch row j (one warp per row): u from Philox(counter = (j, counter), key = seed) in the
// kStreamPer domain, t = ((j + u) / batch) total, then the descent from the top level to a leaf.  Writes the leaf to
// idx_out[j] and its priority to p_out[j]; the smallest drawn priority goes to *min_bits.  With `targets`
// (boatper_find) row j descends to targets[j] instead and only the leaf is written.
__global__ void __launch_bounds__(kPerThreads) per_sample_kernel(const __grid_constant__ PerTree tree, long long batch,
                                                                 unsigned long long seed, unsigned long long counter,
                                                                 const double *__restrict__ targets,
                                                                 long long *__restrict__ idx_out,
                                                                 float *__restrict__ p_out, unsigned *min_bits) {
    const long long j = ((long long)blockIdx.x * kPerThreads + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (j >= batch) return;   // whole warps
    double t;
    if (targets) {
        t = targets[j];
    } else {
        const Philox4 r = philox4x32_10((uint32_t)j, (uint32_t)((unsigned long long)j >> 32), (uint32_t)counter,
                                        kStreamPer | (uint32_t)((counter >> 32) & 0x0fffffffu), (uint32_t)seed,
                                        (uint32_t)(seed >> 32));
        // 53 random bits: (x >> 5) 2^26 + (y >> 6), over 2^53
        const double u =
            (double)((unsigned long long)(r.x >> 5) * 67108864ULL + (r.y >> 6)) * (1.0 / 9007199254740992.0);
        t = (((double)j + u) / (double)batch) * tree.sums[tree.n_levels - 1][0];
    }
    long long b = 0;
#pragma unroll
    for (int k = kMaxLevels - 1; k >= 1; --k)   // unrolled: the level pointers stay in the parameter bank
        if (k <= tree.n_levels - 2) b = b * kFan + descend(tree.sums[k] + b * kFan, t, lane);
    const long long leaf = b * kFan + descend(tree.leaves + b * kFan, t, lane);
    if (lane == 0) {
        const float p = tree.leaves[leaf];
        idx_out[j] = leaf;
        if (p_out) {
            p_out[j] = p;
            atomicMin(min_bits, __float_as_uint(p));
        }
    }
}

// w_j = (n P(j))^-beta / max_i (n P(i))^-beta = (p_min / p_j)^beta, in place over the drawn priorities
__global__ void __launch_bounds__(kPerThreads) per_weight_kernel(float *__restrict__ w, long long batch, double beta,
                                                                 const unsigned *__restrict__ min_bits) {
    const double pmin = (double)__uint_as_float(*min_bits);
    for (long long j = (long long)blockIdx.x * kPerThreads + threadIdx.x; j < batch; j += (long long)gridDim.x * kPerThreads)
        w[j] = (float)pow(pmin / (double)w[j], beta);
}

unsigned grid_for(long long threads) {
    return (unsigned)std::max(1LL, std::min((threads + kPerThreads - 1) / kPerThreads, 148LL * 64));
}

// sums of levels 1.. over the blocks holding slots [a, e) (e > a, no wrap), or over the slots idx[0 .. n)
cudaError_t resum(boatper_t p, long long a, long long e, const long long *idx, long long n, cudaStream_t st) {
    for (int k = 1; k < p->n_levels; ++k) {
        const int shift = kFanLog * k;
        const long long b0 = idx ? 0 : a >> shift, nb = idx ? n : ((e - 1) >> shift) - b0 + 1;
        const unsigned grid = (unsigned)((nb * 32 + kPerThreads - 1) / kPerThreads);
        if (k == 1)
            per_sum_kernel<float><<<grid, kPerThreads, 0, st>>>(p->leaves, p->sums[1], idx, nb, shift, b0, p->mem_size);
        else
            per_sum_kernel<double><<<grid, kPerThreads, 0, st>>>(p->sums[k - 1], p->sums[k], idx, nb, shift, b0,
                                                                 p->mem_size);
        count_launch();
        const cudaError_t err = cudaGetLastError();
        if (err != cudaSuccess) return err;
    }
    return cudaSuccess;
}

long long padded(long long n) { return (n + kFan - 1) / kFan * kFan; }

PerTree tree_of(boatper_t p) {
    PerTree t;
    std::memset(&t, 0, sizeof(t));
    t.leaves = p->leaves;
    for (int k = 1; k < p->n_levels; ++k) t.sums[k] = p->sums[k];
    t.n_levels = p->n_levels;
    return t;
}

}  // namespace

extern "C" {

int boatper_create(int64_t mem_size, int device, boatper_t *out) {
    if (!out || mem_size <= 0) return BOATENV_EINVAL;
    *out = nullptr;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0 || device < 0 || device >= ndev) return BOATENV_ENODEVICE;
    boatenv::DeviceGuard _guard(device);
    if (!_guard.ok()) return (int)_guard.error();
    boatper_handle *p = new (std::nothrow) boatper_handle();
    if (!p) return BOATENV_EINVAL;
    std::memset(p, 0, sizeof(*p));
    p->mem_size = mem_size;
    p->device = device;
    p->count[0] = mem_size;
    p->n_levels = 1;
    do {
        p->count[p->n_levels] = (p->count[p->n_levels - 1] + kFan - 1) / kFan;
        ++p->n_levels;
    } while (p->count[p->n_levels - 1] > 1 && p->n_levels < kMaxLevels);
    cudaError_t e = cudaSuccess;
    auto alloc = [&](void **q, size_t bytes) {
        if (e == cudaSuccess) e = cudaMalloc(q, bytes);
        if (e == cudaSuccess) e = cudaMemset(*q, 0, bytes);
    };
    alloc((void **)&p->leaves, (size_t)padded(mem_size) * sizeof(float));
    for (int k = 1; k < p->n_levels; ++k) alloc((void **)&p->sums[k], (size_t)padded(p->count[k]) * sizeof(double));
    alloc((void **)&p->max_priority, sizeof(float));
    alloc((void **)&p->min_bits, sizeof(unsigned));
    alloc((void **)&p->bad, sizeof(int));
    const float one = 1.f;
    if (e == cudaSuccess) e = cudaMemcpy(p->max_priority, &one, sizeof(float), cudaMemcpyHostToDevice);
    if (e != cudaSuccess) {
        boatper_destroy(p);
        return (int)e;
    }
    *out = p;
    return BOATENV_OK;
}

int boatper_destroy(boatper_t p) {
    if (!p) return BOATENV_EINVAL;
    boatenv::DeviceGuard _guard(p->device);
    cudaFree(p->leaves);
    for (int k = 1; k < kMaxLevels; ++k) cudaFree(p->sums[k]);
    cudaFree(p->max_priority);
    cudaFree(p->min_bits);
    cudaFree(p->bad);
    delete p;
    return BOATENV_OK;
}

int boatper_fill_new(boatper_t p, int64_t first_row, int64_t n_rows, void *stream) {
    if (!p || first_row < 0 || n_rows < 0) return BOATENV_EINVAL;
    if (n_rows == 0) return BOATENV_OK;
    if (n_rows > p->mem_size) {   // only the last mem_size rows are still in the ring
        first_row += n_rows - p->mem_size;
        n_rows = p->mem_size;
    }
    GUARD_DEVICE(p);
    const cudaStream_t st = (cudaStream_t)stream;
    long long row = first_row, left = n_rows;
    while (left > 0) {   // split at the ring's wrap point
        const long long slot0 = row % p->mem_size, n = std::min(left, p->mem_size - slot0);
        per_fill_kernel<<<grid_for(n), kPerThreads, 0, st>>>(p->leaves, p->max_priority, slot0, n);
        count_launch();
        CUDA_TRY(cudaGetLastError());
        CUDA_TRY(resum(p, slot0, slot0 + n, nullptr, 0, st));
        row += n;
        left -= n;
    }
    p->filled = std::min((long long)p->mem_size, std::max(p->filled, (long long)(first_row + n_rows)));
    return BOATENV_OK;
}

int boatper_sample(boatper_t p, int64_t batch, uint64_t seed, uint64_t counter, double beta, int64_t *idx_out,
                   float *weight_out, void *stream) {
    if (!p || batch <= 0 || !idx_out || !weight_out || !(beta >= 0.0)) return BOATENV_EINVAL;
    if (p->filled <= 0) return BOATENV_EINVAL;
    GUARD_DEVICE(p);
    const cudaStream_t st = (cudaStream_t)stream;
    CUDA_TRY(cudaMemsetAsync(p->min_bits, 0xff, sizeof(unsigned), st));
    per_sample_kernel<<<(unsigned)((batch * 32 + kPerThreads - 1) / kPerThreads), kPerThreads, 0, st>>>(
        tree_of(p), batch, seed, counter, nullptr, (long long *)idx_out, weight_out, p->min_bits);
    count_launch();
    CUDA_TRY(cudaGetLastError());
    per_weight_kernel<<<grid_for(batch), kPerThreads, 0, st>>>(weight_out, batch, beta, p->min_bits);
    count_launch();
    CUDA_TRY(cudaGetLastError());
    return BOATENV_OK;
}

int boatper_find(boatper_t p, int64_t n, const double *targets, int64_t *idx_out, void *stream) {
    if (!p || n <= 0 || !targets || !idx_out) return BOATENV_EINVAL;
    if (p->filled <= 0) return BOATENV_EINVAL;
    GUARD_DEVICE(p);
    per_sample_kernel<<<(unsigned)((n * 32 + kPerThreads - 1) / kPerThreads), kPerThreads, 0, (cudaStream_t)stream>>>(
        tree_of(p), n, 0, 0, targets, (long long *)idx_out, nullptr, nullptr);
    count_launch();
    CUDA_TRY(cudaGetLastError());
    return BOATENV_OK;
}

int boatper_update(boatper_t p, int64_t batch, const int64_t *idx, const float *td, double alpha, double eps,
                   void *stream) {
    if (!p || batch <= 0 || !idx || !td || !(alpha >= 0.0) || !(eps > 0.0)) return BOATENV_EINVAL;
    if (p->filled <= 0) return BOATENV_EINVAL;
    GUARD_DEVICE(p);
    const cudaStream_t st = (cudaStream_t)stream;
    const long long *ix = (const long long *)idx;
    per_clear_kernel<<<grid_for(batch), kPerThreads, 0, st>>>(p->leaves, ix, td, batch, p->mem_size, alpha, (float)eps,
                                                              p->bad);
    count_launch();
    CUDA_TRY(cudaGetLastError());
    per_raise_kernel<<<grid_for(batch), kPerThreads, 0, st>>>(p->leaves, ix, td, batch, p->mem_size, alpha, (float)eps,
                                                              p->bad, p->max_priority);
    count_launch();
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(resum(p, 0, 0, ix, batch, st));
    return BOATENV_OK;
}

int boatper_check(boatper_t p, void *stream) {
    if (!p) return BOATENV_EINVAL;
    GUARD_DEVICE(p);
    const cudaStream_t st = (cudaStream_t)stream;
    int bad = 0;
    CUDA_TRY(cudaMemcpyAsync(&bad, p->bad, sizeof(int), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    if (!bad) return BOATENV_OK;
    CUDA_TRY(cudaMemsetAsync(p->bad, 0, sizeof(int), st));
    return BOATENV_EINVAL;
}

int64_t boatper_level_size(boatper_t p, int32_t level) {
    if (!p || level < 0 || level >= p->n_levels) return BOATENV_EINVAL;
    return p->count[level];
}

int64_t boatper_filled(boatper_t p) { return p ? p->filled : BOATENV_EINVAL; }

int boatper_read(boatper_t p, int32_t level, void *out, void *stream) {
    if (!p || !out || level < -1 || level >= p->n_levels) return BOATENV_EINVAL;
    GUARD_DEVICE(p);
    const void *src = level < 0 ? (const void *)p->max_priority : level == 0 ? (const void *)p->leaves : p->sums[level];
    const size_t bytes = level < 0 ? sizeof(float) : (size_t)p->count[level] * (level == 0 ? sizeof(float) : sizeof(double));
    CUDA_TRY(cudaMemcpyAsync(out, src, bytes, cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
    return BOATENV_OK;
}

int boatper_load(boatper_t p, const float *leaves, int64_t n, const float *max_priority, int64_t filled, void *stream) {
    if (!p || n < 0 || n > p->mem_size || (n && !leaves) || !max_priority || filled < 0 || filled > p->mem_size)
        return BOATENV_EINVAL;
    GUARD_DEVICE(p);
    const cudaStream_t st = (cudaStream_t)stream;
    CUDA_TRY(cudaMemsetAsync(p->leaves, 0, (size_t)padded(p->mem_size) * sizeof(float), st));
    if (n) CUDA_TRY(cudaMemcpyAsync(p->leaves, leaves, (size_t)n * sizeof(float), cudaMemcpyDeviceToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(p->max_priority, max_priority, sizeof(float), cudaMemcpyDeviceToDevice, st));
    CUDA_TRY(resum(p, 0, p->mem_size, nullptr, 0, st));
    p->filled = filled;
    return BOATENV_OK;
}

}  // extern "C"
