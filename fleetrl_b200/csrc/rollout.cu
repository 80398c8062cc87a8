// rollout.cu — device RolloutBuffer: SB3 2.3.2's PPO rollout storage (stable_baselines3/common/buffers.py, RolloutBuffer)
// behind include/fleetstep.h, over caller-owned [T][E]... float32 arrays (FleetRolloutBuf).  The library keeps no state.
//
//   rollout_add_kernel     RolloutBuffer.add: one slot t of every array (flat copies of [E][D], [E][N] and [E]); 16-byte
//                          vectors where both views are 16-byte aligned, 4-byte words otherwise.
//   rollout_gae_kernel     compute_returns_and_advantage: one thread per env scans t = T-1 .. 0 with SB3's float32
//                          operations in SB3's order (explicit _rn intrinsics, so no contraction flag can change them),
//                          loading kAhead steps of its [T][E] rows (coalesced across the warp) before the dependent chain.
//   rollout_gather_kernel  _get_samples after swap_and_flatten without the flatten: flat sample k (env-major, env k / T,
//                          step k % T) is row (k % T) * E + k / T of the [T][E] storage.  One warp per sample row issues
//                          all loads of a segment before its stores; one launch writes the six minibatch tensors.
// No atomics: every output element has one writer, so all three are deterministic.  Offsets are 64-bit throughout.
#include <cuda_runtime.h>
#include <stdint.h>

#include <algorithm>
#include <string>

#include "fleetstep.h"

namespace {

constexpr int kThreads = 256;
constexpr int kAhead = 16;        // GAE steps loaded ahead of the dependent arithmetic
constexpr int kSegment = 4;       // loads a lane issues before its stores in the row copies
constexpr int kAddMaxBlocks = 8192;

thread_local std::string g_err;

int fail(int code, const std::string& msg) {
    g_err = msg;
    return code;
}

#define ROLL_TRY(expr)                                                                  \
    do {                                                                                \
        cudaError_t _e = (expr);                                                        \
        if (_e != cudaSuccess) return fail(FLEET_E_CUDA, std::string(#expr) + ": " + cudaGetErrorString(_e)); \
    } while (0)

bool aligned16(const void* p) { return ((uintptr_t)p & 15u) == 0; }

// dst[i] = src[i] for i < n, grid-stride, kSegment loads in flight per thread.
template <typename V>
__device__ __forceinline__ void copy_flat(const V* __restrict__ src, V* __restrict__ dst, int64_t n) {
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += kSegment * stride) {
        if (i + (kSegment - 1) * stride < n) {
            V v[kSegment];
#pragma unroll
            for (int u = 0; u < kSegment; u++) v[u] = src[i + u * stride];
#pragma unroll
            for (int u = 0; u < kSegment; u++) dst[i + u * stride] = v[u];
        } else {
            for (int64_t j = i; j < n; j += stride) dst[j] = src[j];
        }
    }
}

__device__ __forceinline__ void copy_words(const float* src, float* dst, int64_t n, bool vec) {
    if (vec) {
        const int64_t n4 = n >> 2;
        copy_flat(reinterpret_cast<const float4*>(src), reinterpret_cast<float4*>(dst), n4);
        copy_flat(src + 4 * n4, dst + 4 * n4, n - 4 * n4);
    } else {
        copy_flat(src, dst, n);
    }
}

struct AddParams {
    const float* obs; float* obs_dst; int64_t n_obs; int obs_vec;
    const float* act; float* act_dst; int64_t n_act; int act_vec;
    const float* rew; float* rew_dst;
    const uint8_t* start; float* start_dst;
    const float* val; float* val_dst;
    const float* logp; float* logp_dst;
    int64_t E;
};

__global__ void __launch_bounds__(kThreads) rollout_add_kernel(AddParams p) {
    if (p.obs) copy_words(p.obs, p.obs_dst, p.n_obs, p.obs_vec);
    if (p.act) copy_words(p.act, p.act_dst, p.n_act, p.act_vec);
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < p.E; e += stride) {
        if (p.rew) p.rew_dst[e] = p.rew[e];
        if (p.start) p.start_dst[e] = p.start[e] ? 1.0f : 0.0f;
        if (p.val) p.val_dst[e] = p.val[e];
        if (p.logp) p.logp_dst[e] = p.logp[e];
    }
}

// RolloutBuffer.compute_returns_and_advantage (buffers.py), per env e:
//   t = T-1:  nnt = 1 - float32(dones[e]);      nv = last_values[e]
//   t < T-1:  nnt = 1 - episode_starts[t+1][e]; nv = values[t+1][e]
//   delta = (rewards[t][e] + (g * nv) * nnt) - values[t][e];   lgl = delta + (gl * nnt) * lgl   (lgl = 0 before T-1)
//   advantages[t][e] = lgl;   returns[t][e] = lgl + values[t][e]
__global__ void __launch_bounds__(kThreads) rollout_gae_kernel(
        const float* __restrict__ rewards, const float* __restrict__ values, const float* __restrict__ starts,
        const float* __restrict__ last_values, const uint8_t* __restrict__ dones, float* __restrict__ adv,
        float* __restrict__ ret, int T, int64_t E, float g, float gl) {
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= E) return;
    float nv = last_values[e];
    float nnt = __fsub_rn(1.0f, (float)dones[e]);
    float lgl = 0.0f;
    for (int t0 = T - 1; t0 >= 0; t0 -= kAhead) {
        float r[kAhead], v[kAhead], s[kAhead];
#pragma unroll
        for (int k = 0; k < kAhead; k++) {
            const int t = t0 - k;
            if (t >= 0) {
                const int64_t o = (int64_t)t * E + e;
                r[k] = rewards[o];
                v[k] = values[o];
                s[k] = t > 0 ? starts[o] : 0.0f;   // episode_starts[t] is the non-terminal flag of step t-1
            }
        }
#pragma unroll
        for (int k = 0; k < kAhead; k++) {
            const int t = t0 - k;
            if (t >= 0) {
                const float delta = __fsub_rn(__fadd_rn(r[k], __fmul_rn(__fmul_rn(g, nv), nnt)), v[k]);
                lgl = __fadd_rn(delta, __fmul_rn(__fmul_rn(gl, nnt), lgl));
                const int64_t o = (int64_t)t * E + e;
                adv[o] = lgl;
                ret[o] = __fadd_rn(lgl, v[k]);
                nv = v[k];
                nnt = __fsub_rn(1.0f, s[k]);
            }
        }
    }
}

// One row of n elements of V, copied by the 32 lanes of a warp, kSegment loads per lane before its stores.
template <typename V>
__device__ __forceinline__ void copy_row(const V* __restrict__ src, V* __restrict__ dst, int n, int lane) {
    for (int j0 = lane; j0 < n; j0 += 32 * kSegment) {
        V v[kSegment];
#pragma unroll
        for (int u = 0; u < kSegment; u++)
            if (j0 + 32 * u < n) v[u] = src[j0 + 32 * u];
#pragma unroll
        for (int u = 0; u < kSegment; u++)
            if (j0 + 32 * u < n) dst[j0 + 32 * u] = v[u];
    }
}

struct GatherParams {
    const float* obs; const float* act; const float* val; const float* logp; const float* adv; const float* ret;
    const int64_t* idx;
    float* obs_out; float* act_out; float* val_out; float* logp_out; float* adv_out; float* ret_out;
    int64_t count, E, total;
    int T, D, N, obs_vec;
};

__global__ void __launch_bounds__(kThreads) rollout_gather_kernel(GatherParams p) {
    const int lane = threadIdx.x & 31;
    const int64_t i = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (i >= p.count) return;
    const int64_t k = p.idx[i];
    if (k < 0 || k >= p.total) return;   // out-of-range indices write nothing (the Python side range-checks them)
    const int64_t row = (k % p.T) * p.E + k / p.T;
    const int D = p.D, N = p.N;
    if (lane < 4) {   // the four per-sample scalars: one lane each, loaded with the rows
        const float* src = lane == 0 ? p.val : lane == 1 ? p.logp : lane == 2 ? p.adv : p.ret;
        float* dst = lane == 0 ? p.val_out : lane == 1 ? p.logp_out : lane == 2 ? p.adv_out : p.ret_out;
        dst[i] = src[row];
    }
    if (p.obs_vec)
        copy_row(reinterpret_cast<const float4*>(p.obs + row * D), reinterpret_cast<float4*>(p.obs_out + i * D), D >> 2,
                 lane);
    else
        copy_row(p.obs + row * D, p.obs_out + i * D, D, lane);
    copy_row(p.act + row * N, p.act_out + i * N, N, lane);
}

int check_buf(const FleetRolloutBuf* b) {
    if (!b) return fail(FLEET_E_INVALID, "buffer descriptor is NULL");
    if (b->buffer_size < 1 || b->num_envs < 1 || b->obs_dim < 1 || b->action_dim < 1)
        return fail(FLEET_E_INVALID, "buffer_size, num_envs, obs_dim and action_dim must be >= 1");
    if (!b->observations || !b->actions || !b->rewards || !b->episode_starts || !b->values || !b->log_probs ||
        !b->advantages || !b->returns)
        return fail(FLEET_E_INVALID, "a storage pointer of the buffer is NULL");
    return FLEET_OK;
}

}  // namespace

int fleet_rollout_add(const FleetRolloutBuf* b, int32_t slot, const float* obs, const float* action, const float* reward,
                      const uint8_t* episode_start, const float* value, const float* log_prob, void* stream) {
    int rc = check_buf(b);
    if (rc) return rc;
    if (slot < 0 || slot >= b->buffer_size)
        return fail(FLEET_E_INVALID, "slot " + std::to_string(slot) + " outside [0, " + std::to_string(b->buffer_size) + ")");
    const int64_t E = b->num_envs, D = b->obs_dim, N = b->action_dim, t = slot;
    AddParams p;
    p.obs = obs; p.obs_dst = b->observations + t * E * D; p.n_obs = E * D;
    p.obs_vec = aligned16(obs) && aligned16(p.obs_dst);
    p.act = action; p.act_dst = b->actions + t * E * N; p.n_act = E * N;
    p.act_vec = aligned16(action) && aligned16(p.act_dst);
    p.rew = reward; p.rew_dst = b->rewards + t * E;
    p.start = episode_start; p.start_dst = b->episode_starts + t * E;
    p.val = value; p.val_dst = b->values + t * E;
    p.logp = log_prob; p.logp_dst = b->log_probs + t * E;
    p.E = E;
    if (!obs && !action && !reward && !episode_start && !value && !log_prob) return FLEET_OK;
    int64_t work = E;
    if (obs) work = std::max(work, p.obs_vec ? p.n_obs / 4 : p.n_obs);
    if (action) work = std::max(work, p.act_vec ? p.n_act / 4 : p.n_act);
    const int64_t blocks = std::min<int64_t>(kAddMaxBlocks, (work + kThreads - 1) / kThreads);
    rollout_add_kernel<<<(unsigned)blocks, kThreads, 0, (cudaStream_t)stream>>>(p);
    ROLL_TRY(cudaGetLastError());
    return FLEET_OK;
}

int fleet_rollout_gae(const FleetRolloutBuf* b, double gamma, double gae_lambda, const float* last_values,
                      const uint8_t* dones, void* stream) {
    int rc = check_buf(b);
    if (rc) return rc;
    if (!(gamma >= 0.0 && gamma <= 1.0)) return fail(FLEET_E_INVALID, "gamma must be in [0, 1]");
    if (!(gae_lambda >= 0.0 && gae_lambda <= 1.0)) return fail(FLEET_E_INVALID, "gae_lambda must be in [0, 1]");
    if (!last_values || !dones) return fail(FLEET_E_INVALID, "last_values and dones are required");
    const int64_t E = b->num_envs;
    // NumPy 2 promotes the Python float gamma to float32 against the float32 arrays; gamma * gae_lambda is a Python
    // (double) product, rounded to float32 where it meets next_non_terminal.
    const float g = (float)gamma, gl = (float)(gamma * gae_lambda);
    rollout_gae_kernel<<<(unsigned)((E + kThreads - 1) / kThreads), kThreads, 0, (cudaStream_t)stream>>>(
        b->rewards, b->values, b->episode_starts, last_values, dones, b->advantages, b->returns, b->buffer_size, E, g, gl);
    ROLL_TRY(cudaGetLastError());
    return FLEET_OK;
}

int fleet_rollout_gather(const FleetRolloutBuf* b, const int64_t* flat_idx_dev, int64_t count, float* obs_out,
                         float* actions_out, float* values_out, float* log_probs_out, float* advantages_out,
                         float* returns_out, void* stream) {
    int rc = check_buf(b);
    if (rc) return rc;
    if (count < 0) return fail(FLEET_E_INVALID, "count must be >= 0");
    if (count == 0) return FLEET_OK;
    if (!flat_idx_dev || !obs_out || !actions_out || !values_out || !log_probs_out || !advantages_out || !returns_out)
        return fail(FLEET_E_INVALID, "flat_idx_dev and the six outputs are required");
    GatherParams p;
    p.obs = b->observations; p.act = b->actions; p.val = b->values; p.logp = b->log_probs;
    p.adv = b->advantages; p.ret = b->returns;
    p.idx = flat_idx_dev;
    p.obs_out = obs_out; p.act_out = actions_out; p.val_out = values_out; p.logp_out = log_probs_out;
    p.adv_out = advantages_out; p.ret_out = returns_out;
    p.count = count; p.E = b->num_envs; p.total = (int64_t)b->buffer_size * b->num_envs;
    p.T = b->buffer_size; p.D = b->obs_dim; p.N = b->action_dim;
    p.obs_vec = b->obs_dim % 4 == 0 && aligned16(b->observations) && aligned16(obs_out);
    const int64_t warps_per_block = kThreads / 32;
    const int64_t blocks = (count + warps_per_block - 1) / warps_per_block;
    if (blocks > 0x7fffffff) return fail(FLEET_E_INVALID, "count too large for one launch");
    rollout_gather_kernel<<<(unsigned)blocks, kThreads, 0, (cudaStream_t)stream>>>(p);
    ROLL_TRY(cudaGetLastError());
    return FLEET_OK;
}

const char* fleet_rollout_last_error(void) { return g_err.c_str(); }
