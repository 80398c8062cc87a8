// vecnorm.cu — device VecNormalize: SB3 2.3.2's running observation / return normalisation behind include/fleetstep.h
// (stable_baselines3/common/vec_env/vec_normalize.py, common/running_mean_std.py), for any [E][D] float32 batch.
//
// Two launches per training step, on the caller's stream, no host synchronisation:
//   norm_moments_kernel  one read of the batch.  Envs are cut into chunks of kChunk rows (independent of the SM count);
//                        a CTA sums one chunk x 32 columns of (x - K) and (x - K)^2 in float64, K = the running mean, and
//                        for column tile 0 also the chunk's new returns (returns*gamma + reward, not written back).  The
//                        last CTA of each column tile adds the chunk partials in chunk order into the caller's moments
//                        vector.  No floating-point atomics: the result is bit-identical for any grid.  Because every
//                        rank holds the same K, the shifted sums of several ranks simply add (one all-reduce).
//   norm_apply_kernel    one read and one write of the batch: RunningMeanStd.update_from_moments in float64 (CTA (0,0)
//                        commits it to the other half of a ping-pong state buffer, every CTA recomputes the statistics
//                        of its own columns), then VecNormalize._normalize_obs / _normalize_reward with an IEEE divide
//                        and sqrt (no reciprocal): with identical statistics the outputs equal the NumPy formula bit
//                        for bit.  Terminal rows of finished envs use the updated statistics; returns[done] = 0.
// Loads are 4-byte scalars, coalesced across the 32 columns a warp covers, so any view alignment and any D work.
#include <cuda_runtime.h>
#include <stdint.h>

#include <string>

#include "fleetstep.h"

namespace {

constexpr int kNormThreads = 256;
constexpr int kNormWarps = kNormThreads / 32;
constexpr int kCols = 32;          // columns per CTA: one per lane
constexpr int kChunk = 512;        // envs per chunk: fixes the summation order
constexpr int kSlice = 32;         // chunk partials staged in shared memory per pass of the final reduction
constexpr int kFinal = 2 * kCols + 2;   // values a column tile reduces: S1, S2 of its columns (+ the returns' two)

// State buffer layout (float64, 2D+4): obs mean [D], obs var [D], obs count, ret mean, ret var, ret count.
// Moments vector layout (float64, 2D+4): obs n, S1 [D], S2 [D], ret n, ret S1, ret S2.
// Chunk partial row (float64, 2D+2): S1 [D], S2 [D], ret S1, ret S2.

__device__ __forceinline__ double clip(double v, double c) {   // np.clip: NaN passes through
    v = v < -c ? -c : v;
    return v > c ? c : v;
}

// RunningMeanStd.update_from_moments (running_mean_std.py) with the batch given as shifted sums about K = mean.
__device__ __forceinline__ void merge(double mean, double var, double count, double n, double s1, double s2,
                                      double* new_mean, double* new_var, double* new_count) {
    const double delta = s1 / n;                     // batch_mean - mean
    double m2b = s2 - s1 * delta;                    // sum of squared deviations from the batch mean
    if (m2b < 0.0) m2b = 0.0;                        // rounding
    const double batch_var = m2b / n;
    const double tot = count + n;
    *new_mean = mean + delta * n / tot;
    const double m_a = var * count;
    const double m_b = batch_var * n;
    const double m_2 = m_a + m_b + delta * delta * count * n / tot;
    *new_var = m_2 / tot;
    *new_count = n + count;
}

__global__ void __launch_bounds__(kNormThreads) norm_moments_kernel(
        const float* __restrict__ x, const float* __restrict__ rew, const double* __restrict__ ret,
        const double* __restrict__ st, double* __restrict__ part, unsigned* __restrict__ tickets, double* __restrict__ out,
        int64_t E, int D, int nchunks, double gamma) {
    __shared__ double wsum[kNormWarps][2][kCols];
    __shared__ double rsum[kNormWarps][2];
    __shared__ double stage[kSlice][kFinal];
    __shared__ int is_last;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int c = blockIdx.x, tile = blockIdx.y;
    const int d = tile * kCols + lane;
    const int64_t e0 = (int64_t)c * kChunk, e1 = min(E, e0 + kChunk);
    const int64_t rs = 2 * (int64_t)D + 2;
    double* prow = part + (int64_t)c * rs;

    if (x) {   // column sums: warp w takes rows e0+w, e0+w+8, ... in order
        double s1 = 0.0, s2 = 0.0;
        if (d < D) {
            const double K = st[d];
            for (int64_t e = e0 + warp; e < e1; e += 4 * kNormWarps) {
                float v[4];
#pragma unroll
                for (int u = 0; u < 4; u++) {
                    const int64_t ee = e + u * kNormWarps;
                    v[u] = ee < e1 ? x[ee * D + d] : 0.0f;
                }
#pragma unroll
                for (int u = 0; u < 4; u++) {
                    if (e + u * kNormWarps < e1) {
                        const double t = (double)v[u] - K;
                        s1 += t;
                        s2 += t * t;
                    }
                }
            }
        }
        wsum[warp][0][lane] = s1;
        wsum[warp][1][lane] = s2;
    }
    if (rew && tile == 0) {   // the chunk's new returns (VecNormalize._update_reward) about K = ret mean
        const double K = st[2 * D + 1];
        double r1 = 0.0, r2 = 0.0;
        for (int64_t e = e0 + threadIdx.x; e < e1; e += kNormThreads) {
            const double r = ret[e] * gamma + (double)rew[e];
            const double t = r - K;
            r1 += t;
            r2 += t * t;
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            r1 += __shfl_down_sync(0xffffffffu, r1, o);
            r2 += __shfl_down_sync(0xffffffffu, r2, o);
        }
        if (lane == 0) { rsum[warp][0] = r1; rsum[warp][1] = r2; }
    }
    __syncthreads();
    if (x && warp == 0 && d < D) {
        double s1 = 0.0, s2 = 0.0;
        for (int w = 0; w < kNormWarps; w++) { s1 += wsum[w][0][lane]; s2 += wsum[w][1][lane]; }
        prow[d] = s1;
        prow[D + d] = s2;
    }
    if (rew && tile == 0 && threadIdx.x == 32) {
        double r1 = 0.0, r2 = 0.0;
        for (int w = 0; w < kNormWarps; w++) { r1 += rsum[w][0]; r2 += rsum[w][1]; }
        prow[2 * D] = r1;
        prow[2 * D + 1] = r2;
    }
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) is_last = atomicAdd(&tickets[tile], 1u) == (unsigned)(nchunks - 1);
    __syncthreads();
    if (!is_last) return;
    __threadfence();

    // Last CTA of this column tile: add the chunk partials in chunk order.  Thread k < kFinal owns value k:
    // k < 32 S1 of column tile*32+k, k < 64 S2 of column tile*32+k-32, 64 / 65 the returns' S1 / S2 (tile 0).
    const int k = threadIdx.x;
    int64_t src = -1;
    if (k < kFinal) {
        if (k < 2 * kCols) {
            const int dk = tile * kCols + (k & 31);
            if (x && dk < D) src = (k < kCols ? 0 : D) + dk;
        } else if (rew && tile == 0) {
            src = 2 * (int64_t)D + (k - 2 * kCols);
        }
    }
    double acc = 0.0;
    for (int c0 = 0; c0 < nchunks; c0 += kSlice) {
        const int nc = min(kSlice, nchunks - c0);
        for (int i = threadIdx.x; i < nc * kFinal; i += kNormThreads) {   // stage: every thread loads, independently
            const int cc = i / kFinal, kk = i - cc * kFinal;
            int64_t s = -1;
            if (kk < 2 * kCols) {
                const int dk = tile * kCols + (kk & 31);
                if (x && dk < D) s = (kk < kCols ? 0 : D) + dk;
            } else if (rew && tile == 0) {
                s = 2 * (int64_t)D + (kk - 2 * kCols);
            }
            stage[cc][kk] = s >= 0 ? __ldcg(part + (int64_t)(c0 + cc) * rs + s) : 0.0;
        }
        __syncthreads();
        if (src >= 0)
            for (int cc = 0; cc < nc; cc++) acc += stage[cc][k];
        __syncthreads();
    }
    if (src >= 0) {
        if (k < 2 * kCols) out[1 + src] = acc;                       // S1 at 1+d, S2 at 1+D+d
        else out[2 * (int64_t)D + 2 + (k - 2 * kCols)] = acc;        // ret S1, ret S2
    }
    if (tile == 0 && threadIdx.x == 0) {
        out[0] = x ? (double)E : 0.0;
        out[2 * (int64_t)D + 1] = rew ? (double)E : 0.0;
        if (!rew) out[2 * (int64_t)D + 2] = out[2 * (int64_t)D + 3] = 0.0;
    }
    if (threadIdx.x == 0) tickets[tile] = 0;   // ready for the next call on the stream
}

struct ApplyParams {
    const double* st;       // running statistics before this step
    double* st_new;         // written by CTA (0,0) when mom != NULL
    const double* mom;      // NULL: normalise only
    const float* x; float* y;
    const float* rew; float* rew_out;
    const uint8_t* done;
    const float* term; float* term_out;
    double* ret;
    int64_t rows;
    int D, norm_obs, norm_reward;
    double clip_obs, clip_reward, gamma, eps;
};

// Running statistics of column d (d == D: the returns) after merging the moments, as update_from_moments leaves them.
__device__ __forceinline__ void stats_after(const ApplyParams& p, int d, double* mean, double* var, double* count) {
    const int D = p.D;
    const bool is_ret = d == D;
    const double* st = p.st;
    double m = is_ret ? st[2 * D + 1] : st[d];
    double v = is_ret ? st[2 * D + 2] : st[D + d];
    double cnt = is_ret ? st[2 * D + 3] : st[2 * D];
    if (p.mom) {
        const double n = is_ret ? p.mom[2 * D + 1] : p.mom[0];
        if (n > 0.0) {
            const double s1 = is_ret ? p.mom[2 * D + 2] : p.mom[1 + d];
            const double s2 = is_ret ? p.mom[2 * D + 3] : p.mom[1 + D + d];
            merge(m, v, cnt, n, s1, s2, &m, &v, &cnt);
        }
    }
    *mean = m; *var = v; *count = cnt;
}

__global__ void __launch_bounds__(kNormThreads) norm_apply_kernel(ApplyParams p) {
    __shared__ double s_mean[kCols], s_den[kCols];
    __shared__ double s_ret_den;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int tile = blockIdx.y, D = p.D;
    const int64_t e0 = (int64_t)blockIdx.x * kChunk, e1 = min(p.rows, e0 + kChunk);

    if (p.mom && blockIdx.x == 0 && blockIdx.y == 0) {   // commit the merged statistics
        for (int d = threadIdx.x; d <= D; d += kNormThreads) {
            double m, v, cnt;
            stats_after(p, d, &m, &v, &cnt);
            if (d < D) {
                p.st_new[d] = m;
                p.st_new[D + d] = v;
                if (d == 0) p.st_new[2 * D] = cnt;
            } else {
                p.st_new[2 * D + 1] = m;
                p.st_new[2 * D + 2] = v;
                p.st_new[2 * D + 3] = cnt;
            }
        }
    }
    if (warp == 0) {
        const int d = tile * kCols + lane;
        if (p.x && d < D) {
            double m, v, cnt;
            stats_after(p, d, &m, &v, &cnt);
            s_mean[lane] = m;
            s_den[lane] = sqrt(v + p.eps);
        }
    } else if (threadIdx.x == 32 && tile == 0 && p.rew) {
        double m, v, cnt;
        stats_after(p, D, &m, &v, &cnt);
        s_ret_den = sqrt(v + p.eps);
    }
    __syncthreads();

    if (p.x) {   // observations and terminal rows: warp w takes rows e0+w, e0+w+8, ...
        const int d = tile * kCols + lane;
        if (d < D) {
            const double m = s_mean[lane], den = s_den[lane], c = p.clip_obs;
            const int64_t stride = (int64_t)kNormWarps * D;   // elements between the rows of one warp
            int64_t off = (e0 + warp) * D + d;
            for (int64_t e = e0 + warp; e < e1; e += 4 * kNormWarps, off += 4 * stride) {
                const int nu = (int)min((int64_t)4, (e1 - e + kNormWarps - 1) / kNormWarps);
                float v[4];
#pragma unroll
                for (int u = 0; u < 4; u++) v[u] = u < nu ? p.x[off + u * stride] : 0.0f;
#pragma unroll
                for (int u = 0; u < 4; u++)
                    if (u < nu) p.y[off + u * stride] = p.norm_obs ? (float)clip(__ddiv_rn((double)v[u] - m, den), c) : v[u];
            }
            if (p.term) {
                off = (e0 + warp) * D + d;
                for (int64_t e = e0 + warp; e < e1; e += kNormWarps, off += stride) {
                    if (!p.done[e]) continue;
                    const float t = p.term[off];
                    p.term_out[off] = p.norm_obs ? (float)clip(__ddiv_rn((double)t - m, den), c) : t;
                }
            }
        }
    }
    if (p.rew && tile == 0) {   // rewards and returns
        const bool commit = p.mom && p.mom[2 * D + 1] > 0.0;
        const double den = s_ret_den, c = p.clip_reward;
        for (int64_t e = e0 + threadIdx.x; e < e1; e += kNormThreads) {
            const float r = p.rew[e];
            if (commit || p.done) {
                double g = p.ret[e];
                if (commit) g = g * p.gamma + (double)r;
                if (p.done && p.done[e]) g = 0.0;
                p.ret[e] = g;
            }
            p.rew_out[e] = p.norm_reward ? (float)clip(__ddiv_rn((double)r, den), c) : r;
        }
    } else if (p.done && tile == 0) {   // returns[done] = 0 without rewards
        for (int64_t e = e0 + threadIdx.x; e < e1; e += kNormThreads)
            if (p.done[e]) p.ret[e] = 0.0;
    }
}

}  // namespace

struct FleetNorm {
    int device = 0;
    int64_t E = 0;
    int D = 0;
    double clip_obs = 10.0, clip_reward = 10.0, gamma = 0.99, eps = 1e-8;
    int training = 1, norm_obs = 1, norm_reward = 1;
    double* st[2] = {nullptr, nullptr};   // ping-pong running statistics (layout above)
    int cur = 0;
    double* ret = nullptr;                // VecNormalize.returns [E]
    double* part = nullptr;               // chunk partials [nchunks][2D+2]
    unsigned* tickets = nullptr;          // per column tile
    int nchunks = 0, ntiles = 0;
    std::string err;
};

namespace {

int nfail(FleetNorm* n, int code, const std::string& msg) {
    if (n) n->err = msg;
    return code;
}

#define NORM_TRY(n, expr)                                                                              \
    do {                                                                                               \
        cudaError_t _e = (expr);                                                                       \
        if (_e != cudaSuccess)                                                                         \
            return nfail(n, FLEET_E_CUDA, std::string(#expr) + ": " + cudaGetErrorString(_e));         \
    } while (0)

int64_t state_len(const FleetNorm* n) { return 2 * (int64_t)n->D + 4; }

}  // namespace

int fleet_norm_create(int32_t num_envs, int32_t obs_dim, int32_t device, double clip_obs, double clip_reward, double gamma,
                      double epsilon, FleetNorm** out) {
    if (!out) return FLEET_E_INVALID;
    FleetNorm* n = new FleetNorm();
    *out = n;   // returned even on failure so that fleet_norm_last_error works; caller destroys it
    if (num_envs < 1 || obs_dim < 1) return nfail(n, FLEET_E_INVALID, "num_envs and obs_dim must be >= 1");
    if (!(clip_obs > 0.0) || !(clip_reward > 0.0)) return nfail(n, FLEET_E_INVALID, "clip_obs and clip_reward must be > 0");
    if (!(gamma >= 0.0 && gamma <= 1.0)) return nfail(n, FLEET_E_INVALID, "gamma must be in [0, 1]");
    if (!(epsilon >= 0.0)) return nfail(n, FLEET_E_INVALID, "epsilon must be >= 0");
    n->device = device;
    n->E = num_envs;
    n->D = obs_dim;
    n->clip_obs = clip_obs; n->clip_reward = clip_reward; n->gamma = gamma; n->eps = epsilon;
    n->nchunks = (int)((n->E + kChunk - 1) / kChunk);
    n->ntiles = (obs_dim + kCols - 1) / kCols;
    cudaError_t ce = cudaSetDevice(device);
    if (ce != cudaSuccess) return nfail(n, FLEET_E_CUDA, std::string("cudaSetDevice: ") + cudaGetErrorString(ce));
    const int64_t L = state_len(n);
    const size_t bytes[5] = {L * sizeof(double), L * sizeof(double), n->E * sizeof(double),
                             (size_t)n->nchunks * (2 * (size_t)obs_dim + 2) * sizeof(double), n->ntiles * sizeof(unsigned)};
    void** ptrs[5] = {(void**)&n->st[0], (void**)&n->st[1], (void**)&n->ret, (void**)&n->part, (void**)&n->tickets};
    for (int i = 0; i < 5; i++) {
        ce = cudaMalloc(ptrs[i], bytes[i]);
        if (ce != cudaSuccess) {
            *ptrs[i] = nullptr;
            return nfail(n, FLEET_E_NOMEM, "cudaMalloc of " + std::to_string(bytes[i]) + " bytes failed: " + cudaGetErrorString(ce));
        }
    }
    NORM_TRY(n, cudaMemset(n->ret, 0, bytes[2]));
    NORM_TRY(n, cudaMemset(n->tickets, 0, bytes[4]));
    // RunningMeanStd(epsilon=1e-4): mean 0, var 1, count 1e-4, for the observations and the returns
    double* h = new double[L];
    for (int64_t i = 0; i < L; i++) h[i] = 0.0;
    for (int d = 0; d < obs_dim; d++) h[obs_dim + d] = 1.0;
    h[2 * obs_dim] = 1e-4;
    h[2 * obs_dim + 2] = 1.0;
    h[2 * obs_dim + 3] = 1e-4;
    ce = cudaMemcpy(n->st[0], h, bytes[0], cudaMemcpyHostToDevice);
    delete[] h;
    if (ce != cudaSuccess) return nfail(n, FLEET_E_CUDA, std::string("cudaMemcpy: ") + cudaGetErrorString(ce));
    return FLEET_OK;
}

int fleet_norm_destroy(FleetNorm* n) {
    if (!n) return FLEET_E_INVALID;
    cudaSetDevice(n->device);
    cudaFree(n->st[0]); cudaFree(n->st[1]); cudaFree(n->ret); cudaFree(n->part); cudaFree(n->tickets);
    delete n;
    return FLEET_OK;
}

int fleet_norm_set_flags(FleetNorm* n, int32_t training, int32_t norm_obs, int32_t norm_reward) {
    if (!n) return FLEET_E_INVALID;
    n->training = training != 0;
    n->norm_obs = norm_obs != 0;
    n->norm_reward = norm_reward != 0;
    return FLEET_OK;
}

int fleet_norm_moments_len(const FleetNorm* n) { return n ? (int)state_len(n) : FLEET_E_INVALID; }

int fleet_norm_moments(FleetNorm* n, const float* obs_dev, const float* reward_dev, double* moments_dev, void* stream) {
    if (!n) return FLEET_E_INVALID;
    if (!moments_dev) return nfail(n, FLEET_E_INVALID, "moments_dev is NULL");
    NORM_TRY(n, cudaSetDevice(n->device));
    cudaStream_t s = (cudaStream_t)stream;
    const float* x = n->training && n->norm_obs ? obs_dev : nullptr;
    const float* r = n->training ? reward_dev : nullptr;
    if (!x) NORM_TRY(n, cudaMemsetAsync(moments_dev, 0, state_len(n) * sizeof(double), s));
    if (!x && !r) return FLEET_OK;
    const dim3 grid((unsigned)n->nchunks, x ? (unsigned)n->ntiles : 1u);
    norm_moments_kernel<<<grid, kNormThreads, 0, s>>>(x, r, n->ret, n->st[n->cur], n->part, n->tickets, moments_dev, n->E,
                                                       n->D, n->nchunks, n->gamma);
    NORM_TRY(n, cudaGetLastError());
    return FLEET_OK;
}

int fleet_norm_apply(FleetNorm* n, const double* moments_dev, int64_t rows, const float* obs_dev, float* obs_out_dev,
                     const float* reward_dev, float* reward_out_dev, const uint8_t* done_dev, const float* terminal_obs_dev,
                     float* terminal_obs_out_dev, void* stream) {
    if (!n) return FLEET_E_INVALID;
    const double* mom = n->training ? moments_dev : nullptr;
    if (rows < 1) return nfail(n, FLEET_E_INVALID, "rows must be >= 1");
    if ((mom || done_dev) && rows != n->E) return nfail(n, FLEET_E_INVALID, "a statistics update or done flags need rows == num_envs");
    if (!obs_dev != !obs_out_dev) return nfail(n, FLEET_E_INVALID, "obs_dev and obs_out_dev must both be given or both be NULL");
    if (!reward_dev != !reward_out_dev) return nfail(n, FLEET_E_INVALID, "reward_dev and reward_out_dev must both be given or both be NULL");
    if (!terminal_obs_dev != !terminal_obs_out_dev) return nfail(n, FLEET_E_INVALID, "terminal_obs_dev and terminal_obs_out_dev must both be given or both be NULL");
    if (terminal_obs_dev && (!done_dev || !obs_dev)) return nfail(n, FLEET_E_INVALID, "terminal rows need done_dev and obs_dev");
    NORM_TRY(n, cudaSetDevice(n->device));
    ApplyParams p;
    p.st = n->st[n->cur];
    p.st_new = n->st[n->cur ^ 1];
    p.mom = mom;
    p.x = obs_dev; p.y = obs_out_dev;
    p.rew = reward_dev; p.rew_out = reward_out_dev;
    p.done = done_dev;
    p.term = terminal_obs_dev; p.term_out = terminal_obs_out_dev;
    p.ret = n->ret;
    p.rows = rows;
    p.D = n->D; p.norm_obs = n->norm_obs; p.norm_reward = n->norm_reward;
    p.clip_obs = n->clip_obs; p.clip_reward = n->clip_reward; p.gamma = n->gamma; p.eps = n->eps;
    if (!obs_dev && !reward_dev && !done_dev && !mom) return FLEET_OK;
    const dim3 grid((unsigned)((rows + kChunk - 1) / kChunk), obs_dev ? (unsigned)n->ntiles : 1u);
    norm_apply_kernel<<<grid, kNormThreads, 0, (cudaStream_t)stream>>>(p);
    NORM_TRY(n, cudaGetLastError());
    if (mom) n->cur ^= 1;
    return FLEET_OK;
}

int fleet_norm_reset_returns(FleetNorm* n, void* stream) {
    if (!n) return FLEET_E_INVALID;
    NORM_TRY(n, cudaSetDevice(n->device));
    NORM_TRY(n, cudaMemsetAsync(n->ret, 0, n->E * sizeof(double), (cudaStream_t)stream));
    return FLEET_OK;
}

int fleet_norm_get_state(FleetNorm* n, double* obs_mean, double* obs_var, double* obs_count, double* ret_mean,
                         double* ret_var, double* ret_count, double* returns, void* stream) {
    if (!n) return FLEET_E_INVALID;
    NORM_TRY(n, cudaSetDevice(n->device));
    cudaStream_t s = (cudaStream_t)stream;
    const int D = n->D;
    const double* st = n->st[n->cur];
    double* dst[7] = {obs_mean, obs_var, obs_count, ret_mean, ret_var, ret_count, returns};
    const double* src[7] = {st, st + D, st + 2 * D, st + 2 * D + 1, st + 2 * D + 2, st + 2 * D + 3, n->ret};
    const int64_t cnt[7] = {D, D, 1, 1, 1, 1, n->E};
    for (int i = 0; i < 7; i++)
        if (dst[i]) NORM_TRY(n, cudaMemcpyAsync(dst[i], src[i], cnt[i] * sizeof(double), cudaMemcpyDeviceToHost, s));
    NORM_TRY(n, cudaStreamSynchronize(s));
    return FLEET_OK;
}

int fleet_norm_set_state(FleetNorm* n, const double* obs_mean, const double* obs_var, const double* obs_count,
                         const double* ret_mean, const double* ret_var, const double* ret_count, const double* returns,
                         void* stream) {
    if (!n) return FLEET_E_INVALID;
    NORM_TRY(n, cudaSetDevice(n->device));
    cudaStream_t s = (cudaStream_t)stream;
    const int D = n->D;
    double* st = n->st[n->cur];
    const double* src[7] = {obs_mean, obs_var, obs_count, ret_mean, ret_var, ret_count, returns};
    double* dst[7] = {st, st + D, st + 2 * D, st + 2 * D + 1, st + 2 * D + 2, st + 2 * D + 3, n->ret};
    const int64_t cnt[7] = {D, D, 1, 1, 1, 1, n->E};
    for (int i = 0; i < 7; i++)
        if (src[i]) NORM_TRY(n, cudaMemcpyAsync(dst[i], src[i], cnt[i] * sizeof(double), cudaMemcpyHostToDevice, s));
    NORM_TRY(n, cudaStreamSynchronize(s));
    return FLEET_OK;
}

const char* fleet_norm_last_error(const FleetNorm* n) { return n ? n->err.c_str() : "null handle"; }
