// learner.cu -- one SAC-v1 update (SACLearner.update, continuous_agent.py) of each of 1 to 16 independent BoatEnv
// agents (11 observations, one action, 256-wide layers) in two kernels, with the 256 x 256 products on the tensor cores
// (tcgen05, bf16 operands, fp32 accumulation in TMEM) and everything else in fp32.  Member m of a launch runs on
// blockIdx.y = m with its own arguments, workspace slice and step counter:
//
//   sac_rows_kernel   one CTA per 128-row tile of the batch, one row per thread (= TMEM lane).  Runs the forward and
//                     backward passes of the five networks for its rows in the dependency order of the update and
//                     writes what the weight gradients need (layer inputs, pre-activation gradients, the heads'
//                     inputs and output gradients) and the tile's loss sums to the workspace.
//   sac_params_kernel reduces the gradients over the batch in a fixed order (tcgen05 for the four fc2 weights, one
//                     warp per hidden unit for the rest), writes them to the parameters' .grad tensors, applies Adam
//                     and the Polyak average (agent_math.cuh, as adam_polyak_kernel) and sums the loss partials.  Its
//                     gradients-only instantiation (boatagent_sac_gradients_members) writes the gradients and the
//                     losses times grad_scale and leaves the parameters and the optimiser state alone, so that the
//                     gradients of several replicas can be all-reduced before one Adam step ...
//   adam_polyak_members_kernel  ... boatagent_adam_polyak_members: adam_polyak_kernel's chunk body (agent_math.cuh).
//
// boatagent_sac_update and boatagent_sac_gradients are the one-member case of boatagent_sac_update_members and
// boatagent_sac_gradients_members.
//
// SAC-v2 (boatagent_sac2_update_members: twin target critics, no value network, a learned temperature) reuses the
// building blocks in three launches: sac2_rows_kernel (the row pass of sac2_rows_tile, six stagings as in v1),
// sac2_params_kernel (the gradients-only parameter body over its three trained networks, plus the log alpha gradient)
// and adam_polyak_members_kernel over its 21 slots.
//
// Prioritized replay (boatagent_sac[2]_update_prioritized_members) runs the kPer instantiation of either row pass
// (sac_rows_prioritized_kernel, sac2_rows_prioritized_kernel: importance-weighted critic rows and per-row TD errors)
// and the same parameter and Adam kernels.
//
// Operands in shared memory and in the workspace use the 8x8 core-matrix layout of actor_tc.cuh: element (r, c) of
// an R-row matrix at (c / 8) * (R * 16) + r * 16 + (c % 8) * 2.  The same bytes are a K-major operand with rows = M/N
// (LBO = R * 16, SBO = 128) and an MN-major operand with rows = K (LBO = 128, SBO = R * 16): so W2 [out][in] is the B
// operand of both H1 . W2^T (forward) and dZ2 . W2 (input gradient), and the workspace tiles of dZ2 and H1 [rows][256]
// are the A and B operands of dW2 = dZ2^T . H1 without a transpose.
#include <cstdint>
#include <cstring>
#include <type_traits>
#include <cuda_bf16.h>
#include <cuda_runtime.h>

#include "../../include/boatenv.h"
#include "actor_tc.cuh"
#include "agent_math.cuh"
#include "launch.h"

namespace boatenv {
namespace {

constexpr int kObs = 11, kRows = 128, kLThreads = 128;
constexpr int kNets = 4;                       // trained networks, in workspace order: actor, critic 1, critic 2, value
constexpr int kSlots = 26;                     // DeviceAdam's tensors: actor 8, critic 1 6, critic 2 6, value 6
constexpr int kSmall = 16;                     // per row and network: inputs x[0..11], head output gradients [12..13]

// workspace per (tile, network), bytes
constexpr size_t kWsH1 = 0;                                  // bf16 core [128][256]: layer-2 input
constexpr size_t kWsDz2b = kWsH1 + kRows * kHidden * 2;      // bf16 core [128][256]: layer-2 pre-activation gradient
constexpr size_t kWsDz1 = kWsDz2b + kRows * kHidden * 2;     // fp32 [256][128] (column-major): layer-1 pre-act. grad
constexpr size_t kWsDz2 = kWsDz1 + kRows * kHidden * 4;      // fp32 [256][128]
constexpr size_t kWsH2 = kWsDz2 + kRows * kHidden * 4;       // fp32 [256][128]: the heads' input
constexpr size_t kWsSmall = kWsH2 + kRows * kHidden * 4;     // fp32 [16][128]
constexpr size_t kWsNet = kWsSmall + kSmall * kRows * 4;
constexpr size_t kWsLoss = 4;                                // per tile: sum (V - vt)^2, sum (lp2 - minQ), sum (q_k - q_hat)^2
constexpr size_t ws_bytes(long long tiles, int nets = kNets) { return (size_t)tiles * (nets * kWsNet + 16 * kWsLoss); }

// SAC-v2 (boatagent_sac2_update_members): three trained networks in workspace order actor, critic 1, critic 2, and 21
// slots -- actor 8, critic 1 6, critic 2 6 (their targets the target critics), log alpha 1.  slot_of and the first 20
// slots' shapes are v1's.  Loss partials per tile: sum (lp + target_entropy), sum (alpha lp - minQ), sum (q_k - y)^2.
constexpr int kNets2 = 3, kSlots2 = 21;

// shared memory of the row kernel
constexpr int kLW1 = 0;                                 // bf16 core [256][16]
constexpr int kLW2 = kLW1 + kHidden * kK1 * 2;          // bf16 core [256][256]
constexpr int kLA = kLW2 + kHidden * kHidden * 2;       // bf16 core [128][256]: H1 (forward) / dZ2 (backward)
constexpr int kLA0 = kLA + kRows * kHidden * 2;         // bf16 core [128][16]
constexpr int kLB1 = kLA0 + kRows * kK1 * 2;            // fp32 [256]
constexpr int kLB2 = kLB1 + kHidden * 4;
constexpr int kLW3 = kLB2 + kHidden * 4;                // fp32 [2][256]
constexpr int kLWa = kLW3 + 2 * kHidden * 4;            // fp32 [256]: fc1's action column (critics)
constexpr int kLB3 = kLWa + kHidden * 4;                // fp32 [2]
constexpr int kLRed = kLB3 + 16;                        // fp32 [4 warps][4]
constexpr int kLBar = kLRed + 4 * 4 * 4;
constexpr int kLSmem = kLBar + 16;
static_assert(kLSmem <= 227 * 1024, "shared memory budget");

// shared memory of the parameter kernel (fc2 blocks): one 128-row K chunk of dZ2 (128 of its columns) and H1
constexpr int kPA = 0, kPB = kRows * 128 * 2, kPBar = kPB + kRows * kHidden * 2, kPSmem = kPBar + 16;
constexpr int kPThreads = 256;

__host__ __device__ constexpr uint32_t idesc_mn(int m, int n, bool a_mn, bool b_mn) {
    return umma_idesc(m, n) | (a_mn ? 1u << 15 : 0u) | (b_mn ? 1u << 16 : 0u);
}

struct Net {   // fp32 parameters of one network (nn.Linear layout [out][in])
    const float *w1, *b1, *w2, *b2, *w3[2], *b3[2];
    int in, nh;
};

struct RowArgs {
    const float *state, *action, *reward, *new_state, *eps, *max_action;
    const uint8_t *done;
    long long batch;
    float gamma, scale;
    Net net[5];   // actor, critic 1, critic 2, value, target value
    unsigned char *ws;
};

struct ParamArgs {
    boatagent_adam_slot slot[kSlots];
    float beta1, beta2, eps, tau;
    long long batch;
    const unsigned char *ws;
    long long *state;   // [steps taken, ticket]
    float *losses;
    float grad_scale;   // gradients-only instantiation: factor on the written gradients and losses
};

// Every member's arguments, member m on blockIdx.y = m.  Both tables travel as kernel parameters, within the
// 32,764-byte limit of CUDA 12.1+.
struct MemberRowArgs {
    RowArgs m[BOATAGENT_SAC_MAX_MEMBERS];
};
struct MemberParamArgs {
    ParamArgs m[BOATAGENT_SAC_MAX_MEMBERS];
};
static_assert(sizeof(MemberRowArgs) <= 32764, "kernel parameter limit");
static_assert(sizeof(MemberParamArgs) <= 32764, "kernel parameter limit");

// SAC-v2 row arguments: net[] = actor, critic 1, critic 2, target critic 1, target critic 2
struct Row2Args {
    RowArgs r;
    const float *log_alpha;
    float target_entropy;
};
struct MemberRow2Args {
    Row2Args m[BOATAGENT_SAC_MAX_MEMBERS];
};
static_assert(sizeof(MemberRow2Args) <= 32764, "kernel parameter limit");

// prioritized replay: the row arguments with each row's importance weight and TD-error output
struct PerRowArgs {
    RowArgs r;
    const float *weights;
    float *td;
};
struct MemberPerRowArgs {
    PerRowArgs m[BOATAGENT_SAC_MAX_MEMBERS];
};
struct PerRow2Args {
    Row2Args r;
    const float *weights;
    float *td;
};
struct MemberPerRow2Args {
    PerRow2Args m[BOATAGENT_SAC_MAX_MEMBERS];
};
static_assert(sizeof(MemberPerRowArgs) <= 32764, "kernel parameter limit");
static_assert(sizeof(MemberPerRow2Args) <= 32764, "kernel parameter limit");

__device__ __forceinline__ uint32_t core_off(int r, int c, int rows) { return (uint32_t)((c >> 3) * (rows * 16) + r * 16 + (c & 7) * 2); }

// Sum over the 128 threads of the CTA, fixed order (butterfly within warps, then warps 0..3).
__device__ __forceinline__ void cta_sum4(float (&v)[4], float *red) {
#pragma unroll
    for (int q = 0; q < 4; ++q)
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v[q] += __shfl_xor_sync(0xffffffffu, v[q], o);
    const int warp = threadIdx.x >> 5;
    if ((threadIdx.x & 31) == 0)
#pragma unroll
        for (int q = 0; q < 4; ++q) red[warp * 4 + q] = v[q];
    __syncthreads();
#pragma unroll
    for (int q = 0; q < 4; ++q) v[q] = ((red[q] + red[4 + q]) + red[8 + q]) + red[12 + q];
}

struct Rows {
    unsigned char *smem;
    uint32_t sbase, tmem, lane_base;   // lane_base: this warp's TMEM lanes
    uint64_t *bar;
    uint32_t phase;
    int tid;

    // the CTA's barrier and its 512 TMEM columns (warp 0 allocates into *slot)
    __device__ __forceinline__ void open(unsigned char *s, uint32_t *slot, int t) {
        smem = s;
        sbase = smem_u32(s);
        bar = reinterpret_cast<uint64_t *>(s + kLBar);
        phase = 0;
        tid = t;
        if (t == 0) {
            mbar_init(bar, 1);
            mbar_fence_init();
        }
        if ((t >> 5) == 0) {
            asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 512;" ::"r"(smem_u32(slot)) : "memory");
            asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
        }
        tc_fence_before();
        __syncthreads();
        tc_fence_after();
        tmem = *slot;
        lane_base = tmem + ((uint32_t)((t >> 5) * 32) << 16);
    }
    __device__ __forceinline__ void close() {
        tc_fence_before();
        __syncthreads();
        if ((tid >> 5) == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 512;" ::"r"(tmem) : "memory");
    }

    // the hand-off from the threads' shared-memory / TMEM writes to one MMA batch, issued by thread 0
    __device__ __forceinline__ void mma_sync() {
        fence_proxy_async_smem();
        tc_fence_before();
        __syncthreads();
        tc_fence_after();
    }
    __device__ __forceinline__ void mma_wait() {
        mbar_wait(bar, phase);
        phase ^= 1u;
        tc_fence_after();
    }

    // fp32 parameters -> shared memory (weights as bf16 operands, the rest fp32).  The previous network's MMAs are done.
    __device__ void stage(const Net &n) {
        __syncthreads();
        // 64 rows of 8 weights per thread: unrolled so that several L2 loads are in flight at once
#pragma unroll 8
        for (int i = tid; i < kHidden * (kHidden / 8); i += kLThreads) {   // row = i % 256, 8-column group = i / 256
            const int r = i & 255, kc = i >> 8;
            const float4 x = __ldg(reinterpret_cast<const float4 *>(n.w2 + r * kHidden + kc * 8));
            const float4 y = __ldg(reinterpret_cast<const float4 *>(n.w2 + r * kHidden + kc * 8 + 4));
            *reinterpret_cast<uint4 *>(smem + kLW2 + core_off(r, kc * 8, kHidden)) =
                make_uint4(pack_bf16(x.x, x.y), pack_bf16(x.z, x.w), pack_bf16(y.x, y.y), pack_bf16(y.z, y.w));
        }
#pragma unroll
        for (int i = tid; i < kHidden * 2; i += kLThreads) {
            const int r = i & 255, kc = i >> 8;
            float w[8];
#pragma unroll
            for (int q = 0; q < 8; ++q) w[q] = kc * 8 + q < n.in ? __ldg(n.w1 + r * n.in + kc * 8 + q) : 0.f;
            *reinterpret_cast<uint4 *>(smem + kLW1 + core_off(r, kc * 8, kHidden)) =
                make_uint4(pack_bf16(w[0], w[1]), pack_bf16(w[2], w[3]), pack_bf16(w[4], w[5]), pack_bf16(w[6], w[7]));
        }
        float *b1 = reinterpret_cast<float *>(smem + kLB1), *b2 = reinterpret_cast<float *>(smem + kLB2),
              *w3 = reinterpret_cast<float *>(smem + kLW3), *wa = reinterpret_cast<float *>(smem + kLWa),
              *b3 = reinterpret_cast<float *>(smem + kLB3);
        for (int j = tid; j < kHidden; j += kLThreads) {
            b1[j] = __ldg(n.b1 + j);
            b2[j] = __ldg(n.b2 + j);
            w3[j] = __ldg(n.w3[0] + j);
            w3[kHidden + j] = n.nh > 1 ? __ldg(n.w3[1] + j) : 0.f;
            wa[j] = __ldg(n.w1 + j * n.in + n.in - 1);
        }
        if (tid < 2) b3[tid] = tid < n.nh ? __ldg(n.b3[tid]) : 0.f;
        __syncthreads();
    }

    // Forward pass of the staged network on this thread's row x[0..15] (zero padded).  Returns the head outputs
    // (bias included) and the ReLU masks; with `ws` set, writes H1 (bf16) and h2 (fp32) of the row there.
    __device__ void forward(const float (&x)[kK1], float (&y)[2], uint32_t (&m1)[8], uint32_t (&m2)[8],
                            unsigned char *ws) {
#pragma unroll
        for (int j = 0; j < 2; ++j)
            *reinterpret_cast<uint4 *>(smem + kLA0 + core_off(tid, 8 * j, kRows)) =
                make_uint4(pack_bf16(x[8 * j], x[8 * j + 1]), pack_bf16(x[8 * j + 2], x[8 * j + 3]),
                           pack_bf16(x[8 * j + 4], x[8 * j + 5]), pack_bf16(x[8 * j + 6], x[8 * j + 7]));
        mma_sync();
        if (tid == 0) {   // layer 1: D[0..255] = A0 . W1^T, K = 16
            umma_bf16(tmem, umma_desc(sbase + kLA0, kRows * 16, 128), umma_desc(sbase + kLW1, kHidden * 16, 128),
                      umma_idesc(kRows, kHidden), 0u);
            umma_commit(bar);
        }
        mma_wait();
        const float *b1 = reinterpret_cast<const float *>(smem + kLB1);
#pragma unroll 1
        for (int c = 0; c < 8; ++c) {   // + bias, ReLU, bf16 -> the A operand of layer 2
            uint32_t r[32];
            tmem_ld32_issue(lane_base + 32u * c, r);
            tmem_ld_wait(r);
            uint32_t mask = 0, p[16];
#pragma unroll
            for (int q = 0; q < 16; ++q) {
                const float h0 = fmaxf(__uint_as_float(r[2 * q]) + b1[32 * c + 2 * q], 0.f);
                const float h1 = fmaxf(__uint_as_float(r[2 * q + 1]) + b1[32 * c + 2 * q + 1], 0.f);
                mask |= (h0 > 0.f ? 1u : 0u) << (2 * q) | (h1 > 0.f ? 1u : 0u) << (2 * q + 1);
                p[q] = pack_bf16(h0, h1);
            }
            m1[c] = mask;
#pragma unroll
            for (int g = 0; g < 4; ++g) {
                const uint4 v = make_uint4(p[4 * g], p[4 * g + 1], p[4 * g + 2], p[4 * g + 3]);
                const uint32_t off = core_off(tid, 32 * c + 8 * g, kRows);
                *reinterpret_cast<uint4 *>(smem + kLA + off) = v;
                if (ws) *reinterpret_cast<uint4 *>(ws + kWsH1 + off) = v;
            }
        }
        mma_sync();
        if (tid == 0) {   // layer 2: D[256..511] = H1 . W2^T
#pragma unroll 1
            for (int k = 0; k < kHidden / 16; ++k)
                umma_bf16(tmem + 256u, umma_desc(sbase + kLA + k * 2 * (kRows * 16), kRows * 16, 128),
                          umma_desc(sbase + kLW2 + k * 2 * (kHidden * 16), kHidden * 16, 128), umma_idesc(kRows, kHidden),
                          k > 0 ? 1u : 0u);
            umma_commit(bar);
        }
        mma_wait();
        const float *b2 = reinterpret_cast<const float *>(smem + kLB2), *w3 = reinterpret_cast<const float *>(smem + kLW3);
        y[0] = y[1] = 0.f;
        float *h2out = ws ? reinterpret_cast<float *>(ws + kWsH2) : nullptr;
#pragma unroll 1
        for (int c = 0; c < 8; ++c) {   // + bias, ReLU, the fp32 heads
            uint32_t r[32];
            tmem_ld32_issue(lane_base + 256u + 32u * c, r);
            tmem_ld_wait(r);
            uint32_t mask = 0;
#pragma unroll
            for (int q = 0; q < 32; ++q) {
                const int j = 32 * c + q;
                const float h = fmaxf(__uint_as_float(r[q]) + b2[j], 0.f);
                mask |= (h > 0.f ? 1u : 0u) << q;
                y[0] = fmaf(h, w3[j], y[0]);
                y[1] = fmaf(h, w3[kHidden + j], y[1]);
                if (h2out) h2out[j * kRows + tid] = h;
            }
            m2[c] = mask;
        }
        const float *b3 = reinterpret_cast<const float *>(smem + kLB3);
        y[0] += b3[0];
        y[1] += b3[1];
    }

    // Backward pass of the staged network from the head output gradients dy (nh of them) with the masks of its
    // forward pass.  With `ws` set, writes dZ2 (bf16 and fp32) and dZ1 (fp32) there.  Returns d out / d x[in - 1]
    // (the critics' action input): sum_j dZ1[j] W1[j][in - 1] in fp32.
    __device__ float backward(const float (&dy)[2], const uint32_t (&m1)[8], const uint32_t (&m2)[8], unsigned char *ws) {
        const float *w3 = reinterpret_cast<const float *>(smem + kLW3);
        float *dz2f = ws ? reinterpret_cast<float *>(ws + kWsDz2) : nullptr;
#pragma unroll 1
        for (int c = 0; c < 8; ++c) {
            uint32_t p[16];
#pragma unroll
            for (int q = 0; q < 16; ++q) {
                float d[2];
#pragma unroll
                for (int e = 0; e < 2; ++e) {
                    const int j = 32 * c + 2 * q + e;
                    const float g = fmaf(dy[1], w3[kHidden + j], dy[0] * w3[j]);
                    d[e] = (m2[c] >> (2 * q + e)) & 1u ? g : 0.f;
                    if (dz2f) dz2f[j * kRows + tid] = d[e];
                }
                p[q] = pack_bf16(d[0], d[1]);
            }
#pragma unroll
            for (int g = 0; g < 4; ++g) {
                const uint4 v = make_uint4(p[4 * g], p[4 * g + 1], p[4 * g + 2], p[4 * g + 3]);
                const uint32_t off = core_off(tid, 32 * c + 8 * g, kRows);
                *reinterpret_cast<uint4 *>(smem + kLA + off) = v;
                if (ws) *reinterpret_cast<uint4 *>(ws + kWsDz2b + off) = v;
            }
        }
        mma_sync();
        if (tid == 0) {   // dH1: D[0..255] = dZ2 . W2  (W2 as an MN-major B operand: N = in, K = out)
#pragma unroll 1
            for (int k = 0; k < kHidden / 16; ++k)
                umma_bf16(tmem, umma_desc(sbase + kLA + k * 2 * (kRows * 16), kRows * 16, 128),
                          umma_desc(sbase + kLW2 + k * 16 * 16, 128, kHidden * 16), idesc_mn(kRows, kHidden, false, true),
                          k > 0 ? 1u : 0u);
            umma_commit(bar);
        }
        mma_wait();
        const float *wa = reinterpret_cast<const float *>(smem + kLWa);
        float *dz1 = ws ? reinterpret_cast<float *>(ws + kWsDz1) : nullptr;
        float dx = 0.f;
#pragma unroll 1
        for (int c = 0; c < 8; ++c) {
            uint32_t r[32];
            tmem_ld32_issue(lane_base + 32u * c, r);
            tmem_ld_wait(r);
#pragma unroll
            for (int q = 0; q < 32; ++q) {
                const int j = 32 * c + q;
                const float d = (m1[c] >> q) & 1u ? __uint_as_float(r[q]) : 0.f;
                dx = fmaf(d, wa[j], dx);
                if (dz1) dz1[j * kRows + tid] = d;
            }
        }
        return dx;
    }
};

__device__ __forceinline__ void put_small(unsigned char *ws, int tid, const float (&x)[kK1], float dy0, float dy1) {
    float *s = reinterpret_cast<float *>(ws + kWsSmall);
#pragma unroll
    for (int q = 0; q < 12; ++q) s[q * kRows + tid] = x[q];
    s[12 * kRows + tid] = dy0;
    s[13 * kRows + tid] = dy1;
}

// min(a, b)'s gradient share of a, as torch's backward of torch.min(a, b): ties split the gradient in halves
__device__ __forceinline__ float min_share(float a, float b) { return a < b ? 1.f : (a == b ? 0.5f : 0.f); }

// The row pass of one 128-row tile.  blockIdx.x is the tile and gridDim.x the tile count of ONE update: the members
// are on blockIdx.y, so both stay per member.  kPer (prioritized replay): row i's critic output gradient and critic
// loss partial are scaled by weights[i], and td_out[i] receives its TD error 0.5 (|q1 - q_hat| + |q2 - q_hat|).
template <bool kPer>
__device__ __forceinline__ void sac_rows_tile(const RowArgs &args, const float *weights, float *td_out, const int tid) {
    extern __shared__ __align__(1024) unsigned char smem[];
    __shared__ uint32_t tmem_slot;
    Rows R;
    R.open(smem, &tmem_slot, tid);

    const long long B = args.batch, row = (long long)blockIdx.x * kRows + tid;
    const float invB = 1.0f / (float)B;
    unsigned char *ws_tile = args.ws + (size_t)blockIdx.x * kNets * kWsNet;
    unsigned char *ws_net[kNets];
#pragma unroll
    for (int k = 0; k < kNets; ++k) ws_net[k] = ws_tile + (size_t)k * kWsNet;
    float *loss_part = reinterpret_cast<float *>(args.ws + (size_t)gridDim.x * kNets * kWsNet) + blockIdx.x * kWsLoss;

    float s[kK1], s2[kK1];
#pragma unroll
    for (int q = 0; q < kK1; ++q) {
        s[q] = q < kObs ? __ldg(args.state + row * kObs + q) : 0.f;
        s2[q] = q < kObs ? __ldg(args.new_state + row * kObs + q) : 0.f;
    }
    const float a_batch = __ldg(args.action + row), rew = __ldg(args.reward + row);
    const bool done = __ldg(args.done + row) != 0;
    const float e0 = __ldg(args.eps + row), e1 = __ldg(args.eps + B + row), ma = __ldg(args.max_action);
    const float w_row = kPer ? __ldg(weights + row) : 1.f;
    float y[2];
    uint32_t m1[8], m2[8];

    // target value on new_state: q_hat = scale r + gamma value_ (value_ = 0 where done)
    R.stage(args.net[4]);
    R.forward(s2, y, m1, m2, nullptr);
    const float q_hat = args.scale * rew + args.gamma * (done ? 0.f : y[0]);

    // actor forward on state; both draws use it
    uint32_t am1[8], am2[8];
    R.stage(args.net[0]);
    R.forward(s, y, am1, am2, ws_net[0]);
    const float mean = y[0], raw_std = y[1];
    float a1, a2;
    const float lp1 = gaussian_head_fwd(mean, raw_std, e0, ma, a1);
    const float lp2 = gaussian_head_fwd(mean, raw_std, e1, ma, a2);

    // the critics: Q at (s, a1) for the value target, Q and dQ/da at (s, a2) for the actor, the trained pass at (s, a)
    float q_a1[2], q_a2[2], dq_a2[2], q_sa[2];
#pragma unroll 1
    for (int k = 0; k < 2; ++k) {
        R.stage(args.net[1 + k]);
        float x[kK1];
#pragma unroll
        for (int q = 0; q < kK1; ++q) x[q] = s[q];
        x[kObs] = a1;
        R.forward(x, y, m1, m2, nullptr);
        q_a1[k] = y[0];
        x[kObs] = a2;
        R.forward(x, y, m1, m2, nullptr);
        q_a2[k] = y[0];
        const float one[2] = {1.f, 0.f};
        dq_a2[k] = R.backward(one, m1, m2, nullptr);
        x[kObs] = a_batch;
        R.forward(x, y, m1, m2, ws_net[1 + k]);
        q_sa[k] = y[0];
        const float dq[2] = {kPer ? (q_sa[k] - q_hat) * w_row * invB : (q_sa[k] - q_hat) * invB, 0.f};
        R.backward(dq, m1, m2, ws_net[1 + k]);
        put_small(ws_net[1 + k], tid, x, dq[0], 0.f);
    }

    // value: dV = (V - value_target) / B, value_target = min(Q1, Q2)(s, a1) - log_prob1
    R.stage(args.net[3]);
    R.forward(s, y, m1, m2, ws_net[3]);
    const float vt = fminf(q_a1[0], q_a1[1]) - lp1;
    const float dv[2] = {(y[0] - vt) * invB, 0.f};
    R.backward(dv, m1, m2, ws_net[3]);
    put_small(ws_net[3], tid, s, dv[0], 0.f);
    const float v_err = y[0] - vt;

    // actor: loss mean(log_prob2 - min(Q1, Q2)(s, a2)); the critics' gradients of this loss are discarded
    const float w1 = min_share(q_a2[0], q_a2[1]), w2 = min_share(q_a2[1], q_a2[0]);
    const float grad_action = -(w1 * dq_a2[0] + w2 * dq_a2[1]) * invB;
    float dyh[2];
    gaussian_head_bwd(mean, raw_std, e1, ma, grad_action, invB, dyh[0], dyh[1]);
    R.stage(args.net[0]);
    R.backward(dyh, am1, am2, ws_net[0]);
    put_small(ws_net[0], tid, s, dyh[0], dyh[1]);

    float part[4] = {v_err * v_err, lp2 - fminf(q_a2[0], q_a2[1]), (q_sa[0] - q_hat) * (q_sa[0] - q_hat),
                     (q_sa[1] - q_hat) * (q_sa[1] - q_hat)};
    if constexpr (kPer) {
        part[2] = w_row * part[2];
        part[3] = w_row * part[3];
        td_out[row] = 0.5f * (fabsf(q_sa[0] - q_hat) + fabsf(q_sa[1] - q_hat));
    }
    cta_sum4(part, reinterpret_cast<float *>(smem + kLRed));
    if (tid < 4) loss_part[tid] = part[tid];
    R.close();
}

// member blockIdx.y, its tiles on blockIdx.x
__global__ void __launch_bounds__(kLThreads, 1) sac_rows_kernel(const __grid_constant__ MemberRowArgs args) {
    sac_rows_tile<false>(args.m[blockIdx.y], nullptr, nullptr, threadIdx.x);
}

__global__ void __launch_bounds__(kLThreads, 1) sac_rows_prioritized_kernel(
    const __grid_constant__ MemberPerRowArgs args) {
    const PerRowArgs &a = args.m[blockIdx.y];
    sac_rows_tile<true>(a.r, a.weights, a.td, threadIdx.x);
}

// The SAC-v2 row pass of one 128-row tile, with alpha = exp(log_alpha) read before the update:
//   y = scale r + gamma (1 - done) (min(Qt1, Qt2)(s', a') - alpha lp'),   a', lp' = actor(s', eps[0])
//   critics: 0.5 mse(Q_k(s, a), y);  actor: mean(alpha lp - min(Q1, Q2)(s, a~)),   a~, lp = actor(s, eps[1])
// Six stagings, as in v1: actor, the two target critics, the two critics, the actor again for its backward pass.
// kPer: importance weights and TD errors as in sac_rows_tile, with y in place of q_hat.
template <bool kPer>
__device__ __forceinline__ void sac2_rows_tile(const Row2Args &a2, const float *weights, float *td_out, const int tid) {
    extern __shared__ __align__(1024) unsigned char smem[];
    __shared__ uint32_t tmem_slot;
    const RowArgs &args = a2.r;
    Rows R;
    R.open(smem, &tmem_slot, tid);

    const long long B = args.batch, row = (long long)blockIdx.x * kRows + tid;
    const float invB = 1.0f / (float)B;
    unsigned char *ws_tile = args.ws + (size_t)blockIdx.x * kNets2 * kWsNet;
    unsigned char *ws_net[kNets2];
#pragma unroll
    for (int k = 0; k < kNets2; ++k) ws_net[k] = ws_tile + (size_t)k * kWsNet;
    float *loss_part = reinterpret_cast<float *>(args.ws + (size_t)gridDim.x * kNets2 * kWsNet) + blockIdx.x * kWsLoss;

    float s[kK1], s2[kK1];
#pragma unroll
    for (int q = 0; q < kK1; ++q) {
        s[q] = q < kObs ? __ldg(args.state + row * kObs + q) : 0.f;
        s2[q] = q < kObs ? __ldg(args.new_state + row * kObs + q) : 0.f;
    }
    const float a_batch = __ldg(args.action + row), rew = __ldg(args.reward + row);
    const bool done = __ldg(args.done + row) != 0;
    const float e0 = __ldg(args.eps + row), e1 = __ldg(args.eps + B + row), ma = __ldg(args.max_action);
    const float alpha = expf(__ldg(a2.log_alpha));
    const float w_row = kPer ? __ldg(weights + row) : 1.f;
    float y[2];
    uint32_t m1[8], m2[8];

    // actor: the target's draw on new_state, then the trained pass on state (its activations to the workspace)
    uint32_t am1[8], am2[8];
    R.stage(args.net[0]);
    R.forward(s2, y, m1, m2, nullptr);
    float a_next, a_pi;
    const float lp_next = gaussian_head_fwd(y[0], y[1], e0, ma, a_next);
    R.forward(s, y, am1, am2, ws_net[0]);
    const float mean = y[0], raw_std = y[1];
    const float lp = gaussian_head_fwd(mean, raw_std, e1, ma, a_pi);

    // target critics at (s', a')
    float qt[2];
#pragma unroll 1
    for (int k = 0; k < 2; ++k) {
        R.stage(args.net[3 + k]);
        float x[kK1];
#pragma unroll
        for (int q = 0; q < kK1; ++q) x[q] = s2[q];
        x[kObs] = a_next;
        R.forward(x, y, m1, m2, nullptr);
        qt[k] = y[0];
    }
    const float q_hat = args.scale * rew + args.gamma * (done ? 0.f : fminf(qt[0], qt[1]) - alpha * lp_next);

    // the critics: Q and dQ/da at (s, a~) for the actor, the trained pass at (s, a)
    float q_pi[2], dq_pi[2], q_sa[2];
#pragma unroll 1
    for (int k = 0; k < 2; ++k) {
        R.stage(args.net[1 + k]);
        float x[kK1];
#pragma unroll
        for (int q = 0; q < kK1; ++q) x[q] = s[q];
        x[kObs] = a_pi;
        R.forward(x, y, m1, m2, nullptr);
        q_pi[k] = y[0];
        const float one[2] = {1.f, 0.f};
        dq_pi[k] = R.backward(one, m1, m2, nullptr);
        x[kObs] = a_batch;
        R.forward(x, y, m1, m2, ws_net[1 + k]);
        q_sa[k] = y[0];
        const float dq[2] = {kPer ? (q_sa[k] - q_hat) * w_row * invB : (q_sa[k] - q_hat) * invB, 0.f};
        R.backward(dq, m1, m2, ws_net[1 + k]);
        put_small(ws_net[1 + k], tid, x, dq[0], 0.f);
    }

    // actor: d loss / d lp = alpha / B; the critics' gradients of this loss are discarded
    const float w1 = min_share(q_pi[0], q_pi[1]), w2 = min_share(q_pi[1], q_pi[0]);
    const float grad_action = -(w1 * dq_pi[0] + w2 * dq_pi[1]) * invB;
    float dyh[2];
    gaussian_head_bwd(mean, raw_std, e1, ma, grad_action, alpha * invB, dyh[0], dyh[1]);
    R.stage(args.net[0]);
    R.backward(dyh, am1, am2, ws_net[0]);
    put_small(ws_net[0], tid, s, dyh[0], dyh[1]);

    float part[4] = {lp + a2.target_entropy, alpha * lp - fminf(q_pi[0], q_pi[1]),
                     (q_sa[0] - q_hat) * (q_sa[0] - q_hat), (q_sa[1] - q_hat) * (q_sa[1] - q_hat)};
    if constexpr (kPer) {
        part[2] = w_row * part[2];
        part[3] = w_row * part[3];
        td_out[row] = 0.5f * (fabsf(q_sa[0] - q_hat) + fabsf(q_sa[1] - q_hat));
    }
    cta_sum4(part, reinterpret_cast<float *>(smem + kLRed));
    if (tid < 4) loss_part[tid] = part[tid];
    R.close();
}

__global__ void __launch_bounds__(kLThreads, 1) sac2_rows_kernel(const __grid_constant__ MemberRow2Args args) {
    sac2_rows_tile<false>(args.m[blockIdx.y], nullptr, nullptr, threadIdx.x);
}

__global__ void __launch_bounds__(kLThreads, 1) sac2_rows_prioritized_kernel(
    const __grid_constant__ MemberPerRow2Args args) {
    const PerRow2Args &a = args.m[blockIdx.y];
    sac2_rows_tile<true>(a.r, a.weights, a.td, threadIdx.x);
}

// slot of tensor `t` (0 w1, 1 b1, 2 w2, 3 b2, 4 / 6 head weights, 5 / 7 head biases) of trained network `n`
__device__ __forceinline__ int slot_of(int n, int t) { return n == 0 ? t : 8 + 6 * (n - 1) + t; }

// kAdam: write the gradients, apply Adam + Polyak and count the step; else write grad_scale times the gradients only.
// blockIdx.x is the CTA and gridDim.x the CTA count of ONE update (member = blockIdx.y), so the step-counter ticket
// counts one member's CTAs.  kN: the trained networks of the workspace, kNets (SAC-v1) or kNets2 (SAC-v2, whose last
// CTA also writes the log alpha gradient).
template <bool kAdam, int kN = kNets>
__device__ __forceinline__ void sac_params_block(const ParamArgs &args, const int tid) {
    extern __shared__ __align__(1024) unsigned char smem[];
    __shared__ uint32_t tmem_slot;
    __shared__ float s_bc1, s_bc2_sqrt;
    const int warp = tid >> 5, lane = tid & 31;
    const long long B = args.batch, tiles = B / kRows;
    if constexpr (kAdam) {
        if (tid == 0) adam_bias_corrections(*reinterpret_cast<volatile long long *>(args.state) + 1, args.beta1,
                                            args.beta2, s_bc1, s_bc2_sqrt);
        __syncthreads();
    }
    const float bc2_sqrt = s_bc2_sqrt;
    auto adam = [&](int k, long long i, float g) {
        const boatagent_adam_slot &sl = args.slot[k];
        if constexpr (kAdam) {
            const_cast<float *>(sl.grad)[i] = g;
            adam_polyak_element(sl, i, g, args.beta1, args.beta2, args.eps, args.tau, sl.lr / s_bc1, bc2_sqrt);
        } else {
            const_cast<float *>(sl.grad)[i] = g * args.grad_scale;
        }
    };
    const int blk = blockIdx.x;
    if (blk < 2 * kN) {
        // ---- fc2 weight gradient of network blk / 2, output rows 128 (blk % 2) .. + 127: dW2 = dZ2^T . H1 on tcgen05
        const int n = blk >> 1, half = blk & 1;
        uint64_t *bar = reinterpret_cast<uint64_t *>(smem + kPBar);
        if (tid == 0) {
            mbar_init(bar, 1);
            mbar_fence_init();
        }
        if (warp == 0) {
            asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 256;" ::"r"(smem_u32(&tmem_slot)) : "memory");
            asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
        }
        tc_fence_before();
        __syncthreads();
        tc_fence_after();
        const uint32_t tmem = tmem_slot, sbase = smem_u32(smem);
        for (long long t = 0; t < tiles; ++t) {   // K = the batch, one 128-row tile at a time
            const unsigned char *w = args.ws + ((size_t)t * kN + n) * kWsNet;
            const uint4 *srcA = reinterpret_cast<const uint4 *>(w + kWsDz2b + (size_t)half * (kRows * 128 * 2));
            const uint4 *srcB = reinterpret_cast<const uint4 *>(w + kWsH1);
#pragma unroll
            for (int i = tid; i < kRows * 128 * 2 / 16; i += kPThreads) reinterpret_cast<uint4 *>(smem + kPA)[i] = srcA[i];
#pragma unroll
            for (int i = tid; i < kRows * kHidden * 2 / 16; i += kPThreads) reinterpret_cast<uint4 *>(smem + kPB)[i] = srcB[i];
            fence_proxy_async_smem();
            tc_fence_before();
            __syncthreads();
            tc_fence_after();
            if (tid == 0) {
#pragma unroll 1
                for (int k = 0; k < kRows / 16; ++k)   // A: dZ2 columns as M, rows as K; B: H1 columns as N, rows as K
                    umma_bf16(tmem, umma_desc(sbase + kPA + k * 16 * 16, 128, kRows * 16),
                              umma_desc(sbase + kPB + k * 16 * 16, 128, kRows * 16), idesc_mn(128, kHidden, true, true),
                              (t > 0 || k > 0) ? 1u : 0u);
                umma_commit(bar);
            }
            mbar_wait(bar, (uint32_t)(t & 1));
            tc_fence_after();
        }
        // epilogue: warp w reads TMEM lanes 32 (w % 4) .. (output row), columns 128 (w / 4) .. + 127 (input)
        const int m = half * 128 + (warp & 3) * 32 + lane;
        const int k = slot_of(n, 2);
#pragma unroll 1
        for (int c = 0; c < 4; ++c) {
            const int col = (warp >> 2) * 128 + 32 * c;
            uint32_t r[32];
            tmem_ld32_issue(tmem + ((uint32_t)((warp & 3) * 32) << 16) + (uint32_t)col, r);
            tmem_ld_wait(r);
#pragma unroll 4
            for (int q = 0; q < 32; ++q) adam(k, (long long)m * kHidden + col + q, __uint_as_float(r[q]));
        }
        tc_fence_before();
        __syncthreads();
        if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 256;" ::"r"(tmem) : "memory");
    } else if (blk < 2 * kN + kN * (kHidden / 8)) {
        // ---- one warp per hidden unit j of network n: fc1 weights and bias, fc2 bias, head weights (+ head biases at
        // j = 0), reduced over the batch in a fixed order (rows strided over the lanes, then a butterfly)
        const int u = (blk - 2 * kN) * 8 + warp, n = u / kHidden, j = u % kHidden;
        const int in = n == 1 || n == 2 ? kObs + 1 : kObs, nh = n == 0 ? 2 : 1;
        float acc[18];
#pragma unroll
        for (int q = 0; q < 18; ++q) acc[q] = 0.f;
        for (long long t = 0; t < tiles; ++t) {
            const unsigned char *w = args.ws + ((size_t)t * kN + n) * kWsNet;
            const float *dz1 = reinterpret_cast<const float *>(w + kWsDz1) + j * kRows;
            const float *dz2 = reinterpret_cast<const float *>(w + kWsDz2) + j * kRows;
            const float *h2 = reinterpret_cast<const float *>(w + kWsH2) + j * kRows;
            const float *sm = reinterpret_cast<const float *>(w + kWsSmall);
#pragma unroll
            for (int rr = 0; rr < kRows / 32; ++rr) {
                const int r = rr * 32 + lane;
                const float d1 = dz1[r], d2 = dz2[r], h = h2[r];
#pragma unroll
                for (int q = 0; q < 12; ++q) acc[q] = fmaf(d1, sm[q * kRows + r], acc[q]);
                acc[12] += d1;
                acc[13] += d2;
                const float g0 = sm[12 * kRows + r], g1 = sm[13 * kRows + r];
                acc[14] = fmaf(g0, h, acc[14]);
                acc[15] = fmaf(g1, h, acc[15]);
                acc[16] += g0;
                acc[17] += g1;
            }
        }
#pragma unroll
        for (int q = 0; q < 18; ++q)
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) acc[q] += __shfl_xor_sync(0xffffffffu, acc[q], o);
        float g = 0.f;   // lane l applies Adam to one element (no dynamic register indexing)
#pragma unroll
        for (int q = 0; q < 18; ++q) g = lane == q ? acc[q] : g;
        if (lane < in) adam(slot_of(n, 0), (long long)j * in + lane, g);
        else if (lane == 12) adam(slot_of(n, 1), j, g);
        else if (lane == 13) adam(slot_of(n, 3), j, g);
        else if (lane == 14) adam(slot_of(n, 4), j, g);
        else if (lane == 15 && nh > 1) adam(slot_of(n, 6), j, g);
        else if (lane == 16 && j == 0) adam(slot_of(n, 5), 0, g);
        else if (lane == 17 && j == 0 && nh > 1) adam(slot_of(n, 7), 0, g);
    } else if (tid == 0) {
        // ---- the three losses from the tiles' partial sums, in tile order
        const float *p = reinterpret_cast<const float *>(args.ws + (size_t)tiles * kN * kWsNet);
        float s[4] = {0.f, 0.f, 0.f, 0.f};
        for (long long t = 0; t < tiles; ++t)
            for (int q = 0; q < 4; ++q) s[q] += p[t * kWsLoss + q];
        const float invB = 1.0f / (float)B;
        if constexpr (kN == kNets2) {
            // temperature loss -log_alpha mean(lp + target_entropy), lp detached: its log alpha gradient is -mean(...)
            const float ent = s[0] * invB;
            adam(kSlots2 - 1, 0, -ent);
            args.losses[0] = (-args.slot[kSlots2 - 1].param[0] * ent) * args.grad_scale;
            args.losses[1] = (s[1] * invB) * args.grad_scale;
            args.losses[2] = (0.5f * (s[2] * invB) + 0.5f * (s[3] * invB)) * args.grad_scale;
        } else if constexpr (kAdam) {
            args.losses[0] = 0.5f * (s[0] * invB);
            args.losses[1] = s[1] * invB;
            args.losses[2] = 0.5f * (s[2] * invB) + 0.5f * (s[3] * invB);
        } else {
            args.losses[0] = (0.5f * (s[0] * invB)) * args.grad_scale;
            args.losses[1] = (s[1] * invB) * args.grad_scale;
            args.losses[2] = (0.5f * (s[2] * invB) + 0.5f * (s[3] * invB)) * args.grad_scale;
        }
    }
    if constexpr (kAdam) {
        __syncthreads();
        if (tid == 0) {   // the last CTA to finish publishes the new step count
            __threadfence();
            const unsigned long long done = atomicAdd(reinterpret_cast<unsigned long long *>(args.state + 1), 1ULL) + 1ULL;
            if (done == gridDim.x) {
                args.state[1] = 0;
                args.state[0] += 1;
            }
        }
    }
}

// member blockIdx.y; threadIdx.x is read here, where the launch bounds bound it
template <bool kAdam>
__global__ void __launch_bounds__(kPThreads) sac_params_kernel(const __grid_constant__ MemberParamArgs args) {
    sac_params_block<kAdam>(args.m[blockIdx.y], threadIdx.x);
}

// SAC-v2 gradients of every member (Adam follows as adam_polyak_members_kernel over the 21 slots)
__global__ void __launch_bounds__(kPThreads) sac2_params_kernel(const __grid_constant__ MemberParamArgs args) {
    sac_params_block<false, kNets2>(args.m[blockIdx.y], threadIdx.x);
}

// Adam + Polyak step (boatagent_adam_polyak_members): member blockIdx.y, its chunks on blockIdx.x
__global__ void __launch_bounds__(kAdamThreads) adam_polyak_members_kernel(const __grid_constant__ MemberParamArgs args) {
    const ParamArgs &a = args.m[blockIdx.y];
    adam_polyak_chunk(a.slot, kSlots, a.beta1, a.beta2, a.eps, a.tau, a.state, blockIdx.x, gridDim.x, threadIdx.x);
}

constexpr int kParamBlocks = 2 * kNets + kNets * (kHidden / 8) + 1;
constexpr int kParamBlocks2 = 2 * kNets2 + kNets2 * (kHidden / 8) + 1;

// numel of slot k, in DeviceAdam's order (actor: fc1 w, b, fc2 w, b, mean w, b, std w, b; critics and value: fc1 w, b,
// fc2 w, b, head w, b)
constexpr long long expected_numel(int k) {
    const int t = k < 8 ? k : (k - 8) % 6, in = (k >= 8 && k < 20) ? kObs + 1 : kObs;
    return t == 0 ? (long long)kHidden * in : t == 2 ? (long long)kHidden * kHidden : (t == 5 || t == 7) ? 1 : kHidden;
}

// numel of SAC-v2 slot k: v1's actor and critics, then log alpha
constexpr long long expected_numel2(int k) { return k < kSlots2 - 1 ? expected_numel(k) : 1; }

// the CTAs of one agent's Adam step: the chunks of its 26 (v2: 21) slots, as boatagent_adam_polyak_step counts them
constexpr int adam_chunks(bool v2 = false) {
    long long n = 0;
    for (int k = 0; k < (v2 ? kSlots2 : kSlots); ++k)
        n += ((v2 ? expected_numel2(k) : expected_numel(k)) + kAdamChunk - 1) / kAdamChunk;
    return (int)n;
}

}  // namespace
}  // namespace boatenv

using namespace boatenv;

extern "C" int64_t boatagent_sac_update_workspace_bytes(int64_t batch) {
    if (batch <= 0 || batch % kRows != 0) return BOATENV_EINVAL;
    return (int64_t)ws_bytes(batch / kRows);
}

extern "C" int64_t boatagent_sac2_update_workspace_bytes(int64_t batch) {
    if (batch <= 0 || batch % kRows != 0) return BOATENV_EINVAL;
    return (int64_t)ws_bytes(batch / kRows, kNets2);
}

namespace {

// The 26 slots of one agent in DeviceAdam's order: every pointer set, the agent's shapes, a target on the value
// network's tensors and only on them, 16-byte aligned parameters.  v2: the 21 slots, targets on the critics' tensors
// and only on them.
int check_slots(const boatagent_adam_slot *slots, bool v2 = false) {
    for (int k = 0; k < (v2 ? kSlots2 : kSlots); ++k) {
        const boatagent_adam_slot &s = slots[k];
        if (!s.param || !s.grad || !s.exp_avg || !s.exp_avg_sq || s.numel != (v2 ? expected_numel2(k) : expected_numel(k)))
            return BOATENV_EINVAL;
        if ((v2 ? k >= 8 && k < 20 : k >= 20) != (s.target != nullptr)) return BOATENV_EINVAL;
        if ((reinterpret_cast<uintptr_t>(s.param) & 15u) != 0) return BOATENV_EALIGN;
    }
    return 0;
}

MemberRowArgs &member_rows() {   // ~32 KB together: kept off the stack
    static thread_local MemberRowArgs ra;
    return ra;
}
MemberParamArgs &member_params() {
    static thread_local MemberParamArgs pa;
    return pa;
}
MemberRow2Args &member_rows2() {
    static thread_local MemberRow2Args ra;
    return ra;
}
template <class RowTable>
RowTable &member_rows_of() {   // the prioritized tables
    static thread_local RowTable ra;
    return ra;
}

const boatagent_sac_member &base_of(const boatagent_sac_member &e) { return e; }
const boatagent_sac_member &base_of(const boatagent_sac2_member &e) { return e.base; }
const boatagent_sac_member &base_of(const boatagent_sac_prioritized_member &e) { return e.base; }
const boatagent_sac_member &base_of(const boatagent_sac2_prioritized_member &e) { return e.base.base; }
float entropy_of(const boatagent_sac2_member &e) { return e.target_entropy; }
float entropy_of(const boatagent_sac2_prioritized_member &e) { return e.base.target_entropy; }
RowArgs &rows_of(RowArgs &r) { return r; }
RowArgs &rows_of(Row2Args &r) { return r.r; }
RowArgs &rows_of(PerRowArgs &r) { return r.r; }
RowArgs &rows_of(PerRow2Args &r) { return r.r.r; }
Row2Args &row2_of(Row2Args &r) { return r; }
Row2Args &row2_of(PerRow2Args &r) { return r.r; }

// The member tables of the kernels of SAC-v1 (Entry boatagent_sac_member, rows MemberRowArgs) or SAC-v2
// (boatagent_sac2_member, MemberRow2Args), or of their prioritized updates (boatagent_sac[2]_prioritized_member,
// MemberPerRow[2]Args): every member checked as documented in boatenv.h (its adam_state only with `adam`) before
// anything is launched.
template <class Entry, class RowTable>
int member_tables(const Entry *members_host, int32_t n_members, int64_t batch, void *workspace,
                  int64_t workspace_bytes, bool adam, float beta1, float beta2, float adam_eps, float grad_scale,
                  RowTable &ra, MemberParamArgs &pa) {
    constexpr bool v2 = std::is_same<Entry, boatagent_sac2_member>::value ||
                        std::is_same<Entry, boatagent_sac2_prioritized_member>::value;
    constexpr bool per = std::is_same<Entry, boatagent_sac_prioritized_member>::value ||
                         std::is_same<Entry, boatagent_sac2_prioritized_member>::value;
    if (!members_host || n_members < 1 || n_members > BOATAGENT_SAC_MAX_MEMBERS || !workspace) return BOATENV_EINVAL;
    if (batch <= 0 || batch % kRows != 0) return BOATENV_EINVAL;
    // a multiple of 16: every slice stays 16-byte aligned
    const size_t slice = ws_bytes(batch / kRows, v2 ? kNets2 : kNets);
    if (workspace_bytes < 0 || (uint64_t)workspace_bytes < slice * (uint64_t)n_members) return BOATENV_EINVAL;
    if ((reinterpret_cast<uintptr_t>(workspace) & 15u) != 0) return BOATENV_EALIGN;
    std::memset(&ra, 0, sizeof(ra));
    std::memset(&pa, 0, sizeof(pa));
    for (int m = 0; m < n_members; ++m) {
        const boatagent_sac_member &b = base_of(members_host[m]);
        if ((adam && !b.adam_state) || !b.state || !b.action || !b.reward || !b.new_state || !b.done || !b.eps ||
            !b.max_action || !b.slots || !b.losses || b.n_slots != (v2 ? kSlots2 : kSlots))
            return BOATENV_EINVAL;
        const int rc = check_slots(b.slots, v2);
        if (rc != 0) return rc;
        if constexpr (per) {
            if (!members_host[m].weights || !members_host[m].td_out) return BOATENV_EINVAL;
            ra.m[m].weights = members_host[m].weights;
            ra.m[m].td = members_host[m].td_out;
        }
        unsigned char *ws = static_cast<unsigned char *>(workspace) + slice * (size_t)m;

        RowArgs &r = rows_of(ra.m[m]);
        r.state = b.state;
        r.action = b.action;
        r.reward = b.reward;
        r.new_state = b.new_state;
        r.eps = b.eps;
        r.max_action = b.max_action;
        r.done = b.done;
        r.batch = batch;
        r.gamma = b.gamma;
        r.scale = b.reward_scale;
        r.ws = ws;
        auto net = [&](int k0, int in, bool actor, bool target) {
            Net n;
            const boatagent_adam_slot *s = b.slots + k0;
            auto p = [&](int t) { return (const float *)(target ? s[t].target : s[t].param); };
            n.w1 = p(0); n.b1 = p(1); n.w2 = p(2); n.b2 = p(3);
            n.w3[0] = p(4); n.b3[0] = p(5);
            n.w3[1] = actor ? p(6) : nullptr; n.b3[1] = actor ? p(7) : nullptr;
            n.in = in;
            n.nh = actor ? 2 : 1;
            return n;
        };
        r.net[0] = net(0, kObs, true, false);
        r.net[1] = net(8, kObs + 1, false, false);
        r.net[2] = net(14, kObs + 1, false, false);
        if constexpr (v2) {
            r.net[3] = net(8, kObs + 1, false, true);
            r.net[4] = net(14, kObs + 1, false, true);
            row2_of(ra.m[m]).log_alpha = b.slots[kSlots2 - 1].param;
            row2_of(ra.m[m]).target_entropy = entropy_of(members_host[m]);
        } else {
            r.net[3] = net(20, kObs, false, false);
            r.net[4] = net(20, kObs, false, true);
        }

        ParamArgs &p = pa.m[m];   // v2: slots 21.. stay zero
        std::memcpy(p.slot, b.slots, sizeof(boatagent_adam_slot) * (v2 ? kSlots2 : kSlots));
        p.beta1 = beta1;
        p.beta2 = beta2;
        p.eps = adam_eps;
        p.tau = b.tau;
        p.batch = batch;
        p.ws = ws;
        p.state = (long long *)b.adam_state;
        p.losses = b.losses;
        p.grad_scale = grad_scale;
    }
    return 0;
}

// the dynamic shared memory opt-in of every learner kernel, once per device
int set_smem_attributes() {
    static std::mutex mu;
    static bool set_of[64] = {false};
    int dev = 0;
    CUDA_TRY(cudaGetDevice(&dev));
    if (dev < 0 || dev >= 64) return (int)cudaErrorInvalidDevice;
    std::lock_guard<std::mutex> lock(mu);
    if (!set_of[dev]) {
        CUDA_TRY(cudaFuncSetAttribute(sac_rows_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kLSmem));
        CUDA_TRY(cudaFuncSetAttribute(sac_params_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kPSmem));
        CUDA_TRY(cudaFuncSetAttribute(sac_params_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, kPSmem));
        CUDA_TRY(cudaFuncSetAttribute(sac2_rows_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kLSmem));
        CUDA_TRY(cudaFuncSetAttribute(sac2_params_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kPSmem));
        CUDA_TRY(cudaFuncSetAttribute(sac_rows_prioritized_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kLSmem));
        CUDA_TRY(cudaFuncSetAttribute(sac2_rows_prioritized_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kLSmem));
        set_of[dev] = true;
    }
    return 0;
}

// the row pass of a member table
void launch_rows(const MemberRowArgs &ra, dim3 grid, cudaStream_t s) { sac_rows_kernel<<<grid, kLThreads, kLSmem, s>>>(ra); }
void launch_rows(const MemberPerRowArgs &ra, dim3 grid, cudaStream_t s) {
    sac_rows_prioritized_kernel<<<grid, kLThreads, kLSmem, s>>>(ra);
}
void launch_rows(const MemberRow2Args &ra, dim3 grid, cudaStream_t s) { sac2_rows_kernel<<<grid, kLThreads, kLSmem, s>>>(ra); }
void launch_rows(const MemberPerRow2Args &ra, dim3 grid, cudaStream_t s) {
    sac2_rows_prioritized_kernel<<<grid, kLThreads, kLSmem, s>>>(ra);
}

template <class RowTable>
int launch(bool adam, int32_t n_members, int64_t batch, const RowTable &ra, const MemberParamArgs &pa, void *stream) {
    const int rc = set_smem_attributes();
    if (rc != 0) return rc;
    const cudaStream_t s = (cudaStream_t)stream;
    launch_rows(ra, dim3((unsigned)(batch / kRows), (unsigned)n_members), s);
    boatenv::count_launch();
    CUDA_TRY(cudaGetLastError());
    const dim3 grid(kParamBlocks, (unsigned)n_members);
    if (adam)
        sac_params_kernel<true><<<grid, kPThreads, kPSmem, s>>>(pa);
    else
        sac_params_kernel<false><<<grid, kPThreads, kPSmem, s>>>(pa);
    boatenv::count_launch();
    return (int)cudaGetLastError();
}

// SAC-v2: the row pass, the gradients, then one coalesced Adam + Polyak launch over the 21 slots (the
// adam_polyak_members_kernel of v1's split update, on the v2 chunk count; slots 21.. of the table are empty).
template <class RowTable>
int launch2(int32_t n_members, int64_t batch, const RowTable &ra, const MemberParamArgs &pa, void *stream) {
    const int rc = set_smem_attributes();
    if (rc != 0) return rc;
    const cudaStream_t s = (cudaStream_t)stream;
    launch_rows(ra, dim3((unsigned)(batch / kRows), (unsigned)n_members), s);
    boatenv::count_launch();
    CUDA_TRY(cudaGetLastError());
    sac2_params_kernel<<<dim3(kParamBlocks2, (unsigned)n_members), kPThreads, kPSmem, s>>>(pa);
    boatenv::count_launch();
    CUDA_TRY(cudaGetLastError());
    adam_polyak_members_kernel<<<dim3(adam_chunks(true), (unsigned)n_members), kAdamThreads, 0, s>>>(pa);
    boatenv::count_launch();
    return (int)cudaGetLastError();
}

}  // namespace

extern "C" int boatagent_sac2_update_members(const boatagent_sac2_member *members_host, int32_t n_members,
                                             int64_t batch, float beta1, float beta2, float adam_eps, void *workspace,
                                             int64_t workspace_bytes, void *stream) {
    MemberRow2Args &ra = member_rows2();
    MemberParamArgs &pa = member_params();
    const int rc = member_tables(members_host, n_members, batch, workspace, workspace_bytes, true, beta1, beta2,
                                 adam_eps, 1.0f, ra, pa);
    if (rc != 0) return rc;
    return launch2(n_members, batch, ra, pa, stream);
}

extern "C" int boatagent_sac_update_prioritized_members(const boatagent_sac_prioritized_member *members_host,
                                                        int32_t n_members, int64_t batch, float beta1, float beta2,
                                                        float adam_eps, void *workspace, int64_t workspace_bytes,
                                                        void *stream) {
    MemberPerRowArgs &ra = member_rows_of<MemberPerRowArgs>();
    MemberParamArgs &pa = member_params();
    const int rc = member_tables(members_host, n_members, batch, workspace, workspace_bytes, true, beta1, beta2,
                                 adam_eps, 1.0f, ra, pa);
    if (rc != 0) return rc;
    return launch(true, n_members, batch, ra, pa, stream);
}

extern "C" int boatagent_sac2_update_prioritized_members(const boatagent_sac2_prioritized_member *members_host,
                                                         int32_t n_members, int64_t batch, float beta1, float beta2,
                                                         float adam_eps, void *workspace, int64_t workspace_bytes,
                                                         void *stream) {
    MemberPerRow2Args &ra = member_rows_of<MemberPerRow2Args>();
    MemberParamArgs &pa = member_params();
    const int rc = member_tables(members_host, n_members, batch, workspace, workspace_bytes, true, beta1, beta2,
                                 adam_eps, 1.0f, ra, pa);
    if (rc != 0) return rc;
    return launch2(n_members, batch, ra, pa, stream);
}

extern "C" int boatagent_sac_update_members(const boatagent_sac_member *members_host, int32_t n_members, int64_t batch,
                                            float beta1, float beta2, float adam_eps, void *workspace,
                                            int64_t workspace_bytes, void *stream) {
    MemberRowArgs &ra = member_rows();
    MemberParamArgs &pa = member_params();
    const int rc = member_tables(members_host, n_members, batch, workspace, workspace_bytes, true, beta1, beta2,
                                 adam_eps, 1.0f, ra, pa);
    if (rc != 0) return rc;
    return launch(true, n_members, batch, ra, pa, stream);
}

extern "C" int boatagent_sac_gradients_members(const boatagent_sac_member *members_host, int32_t n_members,
                                               int64_t batch, float grad_scale, void *workspace,
                                               int64_t workspace_bytes, void *stream) {
    MemberRowArgs &ra = member_rows();
    MemberParamArgs &pa = member_params();
    const int rc = member_tables(members_host, n_members, batch, workspace, workspace_bytes, false, 0.f, 0.f, 0.f,
                                 grad_scale, ra, pa);
    if (rc != 0) return rc;
    return launch(false, n_members, batch, ra, pa, stream);
}

extern "C" int boatagent_sac_update(const float *state, const float *action, const float *reward, const float *new_state,
                                    const uint8_t *done, const float *eps, const float *max_action, int64_t batch,
                                    float gamma, float reward_scale, const boatagent_adam_slot *slots_host,
                                    int32_t n_slots, float beta1, float beta2, float adam_eps, float tau,
                                    int64_t *adam_state, float *losses_out, void *workspace, int64_t workspace_bytes,
                                    void *stream) {
    const boatagent_sac_member m = {state, action, reward, new_state, done, eps, max_action, slots_host, n_slots,
                                    gamma, reward_scale, tau, adam_state, losses_out};
    return boatagent_sac_update_members(&m, 1, batch, beta1, beta2, adam_eps, workspace, workspace_bytes, stream);
}

extern "C" int boatagent_sac_gradients(const float *state, const float *action, const float *reward,
                                       const float *new_state, const uint8_t *done, const float *eps,
                                       const float *max_action, int64_t batch, float gamma, float reward_scale,
                                       const boatagent_adam_slot *slots_host, int32_t n_slots, float grad_scale,
                                       float *losses_out, void *workspace, int64_t workspace_bytes, void *stream) {
    const boatagent_sac_member m = {state, action, reward, new_state, done, eps, max_action, slots_host, n_slots,
                                    gamma, reward_scale, 0.f, nullptr, losses_out};
    return boatagent_sac_gradients_members(&m, 1, batch, grad_scale, workspace, workspace_bytes, stream);
}

extern "C" int boatagent_adam_polyak_members(const boatagent_sac_member *members_host, int32_t n_members, float beta1,
                                             float beta2, float adam_eps, void *stream) {
    if (!members_host || n_members < 1 || n_members > BOATAGENT_SAC_MAX_MEMBERS) return BOATENV_EINVAL;
    MemberParamArgs &pa = member_params();
    std::memset(&pa, 0, sizeof(pa));
    for (int m = 0; m < n_members; ++m) {
        const boatagent_sac_member &b = members_host[m];
        if (!b.adam_state || !b.slots || b.n_slots != kSlots) return BOATENV_EINVAL;
        const int rc = check_slots(b.slots);
        if (rc != 0) return rc;
        std::memcpy(pa.m[m].slot, b.slots, sizeof(pa.m[m].slot));
        pa.m[m].beta1 = beta1;
        pa.m[m].beta2 = beta2;
        pa.m[m].eps = adam_eps;
        pa.m[m].tau = b.tau;
        pa.m[m].state = (long long *)b.adam_state;
    }
    adam_polyak_members_kernel<<<dim3(adam_chunks(), (unsigned)n_members), kAdamThreads, 0, (cudaStream_t)stream>>>(pa);
    boatenv::count_launch();
    return (int)cudaGetLastError();
}
