// ppo.cu — the per-minibatch loss of SB3 2.3.2's PPO.train (stable_baselines3/ppo/ppo.py) with the diagonal Gaussian of
// common/distributions.py (DiagGaussianDistribution), forward and backward, behind include/fleetstep.h.  The library
// keeps no state: the caller owns the minibatch (FleetPpoBatch), the per-sample coefficients the forward pass saves for
// the backward pass, the float64 statistics accumulator and a workspace of fleet_ppo_workspace_bytes(B, N).
//
//   ppo_log_prob_kernel  log_prob of every row: one warp per row, lanes over the action dimensions.
//   ppo_rows_kernel      forward 1/2: log_prob, ratio, value loss, clip fraction and approx_kl of every row, and the
//                        advantages' moments; the last CTA combines the chunk partials (mean and unbiased std).
//   ppo_policy_kernel    forward 2/2: normalised advantage, clipped surrogate, d loss / d log_prob of every row; the last
//                        CTA writes the loss and adds the five statistics to the accumulator.
//   ppo_backward_kernel  grad_mean, grad_values, and the column sums of grad_log_std; the last CTA combines them.
//
// Every reduction runs in float64 over chunks of a fixed number of rows, and the last CTA of a launch (integer ticket,
// as in vecnorm.cu) adds the chunk partials in an order that depends on B and N only: no floating-point atomics, so
// every output is bit-identical from call to call.  Offsets are 64-bit throughout.
#include <cuda_runtime.h>
#include <stdint.h>

#include <cmath>
#include <string>

#include "fleetstep.h"

namespace {

constexpr int kThreads = 256;
constexpr int kWarps = kThreads / 32;
constexpr int kRowsPerWarp = 16;
constexpr int kRows = kWarps * kRowsPerWarp;   // rows per CTA of the row kernels: fixes every summation order
constexpr int kPolicyRows = kThreads;          // rows per CTA of ppo_policy_kernel
constexpr int kPart1 = 6;                      // ppo_rows_kernel's chunk partial: n, mean(A), M2(A), sum vl, clips, kl

thread_local std::string g_err;

int fail(int code, const std::string& msg) {
    g_err = msg;
    return code;
}

#define PPO_TRY(expr)                                                                   \
    do {                                                                                \
        cudaError_t _e = (expr);                                                        \
        if (_e != cudaSuccess) return fail(FLEET_E_CUDA, std::string(#expr) + ": " + cudaGetErrorString(_e)); \
    } while (0)

// Workspace layout.  The tickets must be zero before the first call (a zero-filled allocation); every launch returns
// its ticket to zero.
struct WsHead {
    unsigned tickets[4];
    float adv_mean, adv_std;     // rounded to float32, written by ppo_rows_kernel's last CTA
    double sums[3];              // sum over the batch of value-loss terms, clipped rows, approx_kl terms
    double pad[2];
};
static_assert(sizeof(WsHead) == 64, "WsHead is 64 bytes");

inline int64_t align256(int64_t x) { return (x + 255) & ~(int64_t)255; }
inline int64_t chunks(int64_t B, int rows) { return (B + rows - 1) / rows; }

struct WsLayout {
    int64_t ratio, part1, part2, part3, total;
};

WsLayout ws_layout(int64_t B, int64_t N) {
    WsLayout l;
    l.ratio = align256(sizeof(WsHead));
    l.part1 = l.ratio + align256(B * 4);
    l.part2 = l.part1 + align256(chunks(B, kRows) * kPart1 * 8);
    l.part3 = l.part2 + align256(chunks(B, kPolicyRows) * 8);
    l.total = l.part3 + align256(chunks(B, kRows) * N * 8);
    return l;
}

// One term of Normal.log_prob (torch/distributions/normal.py) in float32, in torch's order:
//   -((value - loc) ** 2) / (2 * var) - log_scale - math.log(math.sqrt(2 * math.pi)),   var = scale ** 2
__device__ __forceinline__ float lp_term(float a, float mu, float two_var, float log_sig, float lsp) {
    const float d = __fsub_rn(a, mu);
    const float t = __fdiv_rn(-__fmul_rn(d, d), two_var);
    return __fsub_rn(__fsub_rn(t, log_sig), lsp);
}

// sigma = exp(log_std), log(sigma): what Normal(mean, ones_like(mean) * log_std.exp()) computes.
__device__ __forceinline__ void column(const float* log_std, int n, float& var, float& log_sig) {
    const float sig = expf(log_std[n]);
    var = __fmul_rn(sig, sig);
    log_sig = logf(sig);
}

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);   // every lane ends with the same bits
    return v;
}

// Sum of v over the CTA in a fixed order (warp butterflies, then warps 0..7).  Every thread gets the result.
__device__ __forceinline__ double block_sum(double v, double* sm) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    v = warp_sum(v);
    __syncthreads();
    if (lane == 0) sm[warp] = v;
    __syncthreads();
    double s = 0.0;
#pragma unroll
    for (int w = 0; w < kWarps; w++) s += sm[w];
    return s;
}

// The log_prob of the kRowsPerWarp rows row0 .. row0+15 of this warp (rows >= B are skipped), summed over the action
// dimensions: lane l adds its columns l, l+32, ... in order in float64, then a butterfly over the lanes; rounded to
// float32 once.  Shared by the log_prob and the loss kernels, so both give the same bits for the same inputs.
__device__ __forceinline__ void warp_log_probs(const float* __restrict__ mean, const float* __restrict__ act,
                                               const float* __restrict__ log_std, int64_t row0, int64_t B, int N,
                                               float lsp, float out[kRowsPerWarp]) {
    const int lane = threadIdx.x & 31;
    double acc[kRowsPerWarp];
#pragma unroll
    for (int r = 0; r < kRowsPerWarp; r++) acc[r] = 0.0;
    for (int n = lane; n < N; n += 32) {
        float var, log_sig;
        column(log_std, n, var, log_sig);
        const float two_var = __fmul_rn(2.0f, var);
        float mu[kRowsPerWarp], a[kRowsPerWarp];
#pragma unroll
        for (int r = 0; r < kRowsPerWarp; r++) {
            if (row0 + r < B) {
                const int64_t o = (row0 + r) * N + n;
                mu[r] = mean[o];
                a[r] = act[o];
            }
        }
#pragma unroll
        for (int r = 0; r < kRowsPerWarp; r++)
            if (row0 + r < B) acc[r] += (double)lp_term(a[r], mu[r], two_var, log_sig, lsp);
    }
#pragma unroll
    for (int r = 0; r < kRowsPerWarp; r++) out[r] = __double2float_rn(warp_sum(acc[r]));
}

__global__ void __launch_bounds__(kThreads) ppo_log_prob_kernel(const float* __restrict__ mean,
                                                                const float* __restrict__ act,
                                                                const float* __restrict__ log_std,
                                                                float* __restrict__ out, int64_t B, int N, float lsp) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t row0 = (int64_t)blockIdx.x * kRows + warp * kRowsPerWarp;
    float lp[kRowsPerWarp];
    warp_log_probs(mean, act, log_std, row0, B, N, lsp, lp);
#pragma unroll
    for (int r = 0; r < kRowsPerWarp; r++)
        if (lane == r && row0 + r < B) out[row0 + r] = lp[r];
}

struct LossArgs {
    FleetPpoBatch b;
    float clip_lo, clip_hi, clip_eps;   // float32(1 - clip_range), float32(1 + clip_range), float32(clip_range)
    float vf_lo, vf_hi;                 // float32(-clip_range_vf), float32(clip_range_vf)
    float lsp;                          // float32(math.log(math.sqrt(2 * math.pi)))
    int clip_vf, normalize;
    double ent_coef, vf_coef;
    float* coef;                        // [2][B]: d loss / d log_prob, d loss / d values
    double* stats;
    float* loss_out;
    WsHead* head;
    float* ratio;
    double* part1;
    double* part2;
    double* part3;
};

// Arrive at the launch's ticket after this CTA's partials are written; true in the last CTA to arrive.
__device__ __forceinline__ bool last_cta(unsigned* ticket, int* flag) {
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) *flag = atomicAdd(ticket, 1u) == gridDim.x - 1;
    __syncthreads();
    if (!*flag) return false;
    __threadfence();
    return true;
}

// Chan et al.'s pairwise combination of (count, mean, M2).
__device__ __forceinline__ void chan(double& n, double& m, double& m2, double nb, double mb, double m2b) {
    if (nb == 0.0) return;
    const double nt = n + nb, d = mb - m;
    m2 = m2 + m2b + d * d * (n * nb / nt);
    m = m + d * (nb / nt);
    n = nt;
}

__global__ void __launch_bounds__(kThreads) ppo_rows_kernel(LossArgs p) {
    __shared__ float s_lp[kRows];
    __shared__ double sm[kWarps];
    __shared__ double tree[4][kThreads];
    __shared__ int is_last;
    const FleetPpoBatch& b = p.b;
    const int64_t B = b.batch_size;
    const int N = b.action_dim;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t c0 = (int64_t)blockIdx.x * kRows;
    {
        float lp[kRowsPerWarp];
        warp_log_probs(b.mean, b.actions, b.log_std, c0 + warp * kRowsPerWarp, B, N, p.lsp, lp);
#pragma unroll
        for (int r = 0; r < kRowsPerWarp; r++)
            if (lane == r) s_lp[warp * kRowsPerWarp + r] = lp[r];
    }
    __syncthreads();

    // Per row (thread t < kRows owns row c0 + t): ratio, value loss, clip fraction, approx_kl.
    const int64_t i = c0 + threadIdx.x;
    const bool valid = threadIdx.x < kRows && i < B;
    double adv = 0.0, vl = 0.0, clip = 0.0, kl = 0.0;
    if (valid) {
        const float log_ratio = __fsub_rn(s_lp[threadIdx.x], b.old_log_prob[i]);
        const float r = expf(log_ratio);
        p.ratio[i] = r;
        clip = fabsf(__fsub_rn(r, 1.0f)) > p.clip_eps ? 1.0 : 0.0;
        kl = ((double)r - 1.0) - (double)log_ratio;
        const float v = b.values[i];
        float vp = v, mask = 1.0f;
        if (p.clip_vf) {
            const float ov = b.old_values[i];
            const float dv = __fsub_rn(v, ov);
            vp = __fadd_rn(ov, fminf(fmaxf(dv, p.vf_lo), p.vf_hi));
            mask = (dv >= p.vf_lo && dv <= p.vf_hi) ? 1.0f : 0.0f;   // clamp passes the gradient at its bounds
        }
        const float e = __fsub_rn(b.returns[i], vp);
        vl = (double)e * (double)e;
        // F.mse_loss(returns, values_pred): d / d values_pred = 2 * (values_pred - returns) / B
        p.coef[B + i] = (float)(p.vf_coef * 2.0 * -(double)e / (double)B) * mask;
        adv = (double)b.advantages[i];
    }
    const double cnt = (double)(valid ? 1 : 0);
    const double n_c = block_sum(cnt, sm);
    const double mean_c = block_sum(adv, sm) / fmax(n_c, 1.0);
    const double dev = valid ? adv - mean_c : 0.0;
    const double m2_c = block_sum(dev * dev, sm);
    const double vl_c = block_sum(vl, sm), clip_c = block_sum(clip, sm), kl_c = block_sum(kl, sm);
    if (threadIdx.x == 0) {
        double* q = p.part1 + (int64_t)blockIdx.x * kPart1;
        q[0] = n_c; q[1] = mean_c; q[2] = m2_c; q[3] = vl_c; q[4] = clip_c; q[5] = kl_c;
    }
    if (!last_cta(&p.head->tickets[0], &is_last)) return;

    // Last CTA: thread t folds chunks t, t + 256, ... in order, then a fixed pairwise tree over the threads.
    double n = 0.0, m = 0.0, m2 = 0.0, s_vl = 0.0, s_clip = 0.0, s_kl = 0.0;
    for (int64_t c = threadIdx.x; c < gridDim.x; c += kThreads) {
        const double* q = p.part1 + c * kPart1;
        chan(n, m, m2, __ldcg(q), __ldcg(q + 1), __ldcg(q + 2));
        s_vl += __ldcg(q + 3);
        s_clip += __ldcg(q + 4);
        s_kl += __ldcg(q + 5);
    }
    for (int s = kThreads / 2; s > 0; s >>= 1) {
        tree[0][threadIdx.x] = n; tree[1][threadIdx.x] = m; tree[2][threadIdx.x] = m2;
        tree[3][threadIdx.x] = s_vl;
        __syncthreads();
        if (threadIdx.x < s) {
            const int o = threadIdx.x + s;
            chan(n, m, m2, tree[0][o], tree[1][o], tree[2][o]);
            s_vl += tree[3][o];
        }
        __syncthreads();
        tree[0][threadIdx.x] = s_clip; tree[1][threadIdx.x] = s_kl;
        __syncthreads();
        if (threadIdx.x < s) {
            s_clip += tree[0][threadIdx.x + s];
            s_kl += tree[1][threadIdx.x + s];
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        // advantages.mean() and advantages.std() (unbiased), reduced in float64 and rounded to float32
        p.head->adv_mean = __double2float_rn(m);
        p.head->adv_std = __double2float_rn(n > 1.0 ? sqrt(m2 / (n - 1.0)) : 0.0);
        p.head->sums[0] = s_vl;
        p.head->sums[1] = s_clip;
        p.head->sums[2] = s_kl;
        p.head->tickets[0] = 0;   // ready for the next call on the stream
    }
}

__global__ void __launch_bounds__(kThreads) ppo_policy_kernel(LossArgs p) {
    __shared__ double sm[kWarps];
    __shared__ double tree[kThreads];
    __shared__ int is_last;
    const FleetPpoBatch& b = p.b;
    const int64_t B = b.batch_size;
    const int64_t i = (int64_t)blockIdx.x * kPolicyRows + threadIdx.x;
    double term = 0.0;
    if (i < B) {
        float a = b.advantages[i];
        if (p.normalize) a = __fdiv_rn(__fsub_rn(a, p.head->adv_mean), __fadd_rn(p.head->adv_std, 1e-8f));
        const float r = __ldcg(p.ratio + i);
        const float rc = fminf(fmaxf(r, p.clip_lo), p.clip_hi);
        const float l1 = __fmul_rn(a, r), l2 = __fmul_rn(a, rc);
        term = (double)fminf(l1, l2);
        // torch's minimum sends the gradient to the smaller side and half to each on a tie; clamp passes it on
        // [lo, hi] inclusive.  d ratio / d log_prob = ratio.
        const float pass = (r >= p.clip_lo && r <= p.clip_hi) ? 1.0f : 0.0f;
        const float w = l1 < l2 ? 1.0f : l1 > l2 ? pass : 0.5f + 0.5f * pass;
        p.coef[i] = (float)(-((double)a * (double)w) * (double)r / (double)B);
    }
    const double part = block_sum(term, sm);
    if (threadIdx.x == 0) p.part2[blockIdx.x] = part;
    if (!last_cta(&p.head->tickets[1], &is_last)) return;

    double s = 0.0;
    for (int64_t c = threadIdx.x; c < gridDim.x; c += kThreads) s += __ldcg(p.part2 + c);
    // entropy of one row: sum_n 0.5 + 0.5 * log(2 pi) + log(sigma_n) (Normal.entropy), the same for every row
    double ent = 0.0;
    for (int n = threadIdx.x; n < b.action_dim; n += kThreads) {
        float var, log_sig;
        column(b.log_std, n, var, log_sig);
        ent += 0.5 + 0.5 * log(2.0 * M_PI) + (double)log_sig;
    }
    for (int k = kThreads / 2; k > 0; k >>= 1) {
        tree[threadIdx.x] = s;
        __syncthreads();
        if (threadIdx.x < k) s += tree[threadIdx.x + k];
        __syncthreads();
        tree[threadIdx.x] = ent;
        __syncthreads();
        if (threadIdx.x < k) ent += tree[threadIdx.x + k];
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        const double Bd = (double)B;
        const double policy_loss = -s / Bd;
        const double value_loss = __ldcg(&p.head->sums[0]) / Bd;
        const double entropy_loss = -ent;
        *p.loss_out = __double2float_rn(policy_loss + p.ent_coef * entropy_loss + p.vf_coef * value_loss);
        p.stats[0] += policy_loss;
        p.stats[1] += value_loss;
        p.stats[2] += entropy_loss;
        p.stats[3] += __ldcg(&p.head->sums[1]) / Bd;
        p.stats[4] += __ldcg(&p.head->sums[2]) / Bd;
        p.head->tickets[1] = 0;
    }
}

struct BackArgs {
    FleetPpoBatch b;
    const float* grad_loss;
    const float* coef;
    float* grad_mean;
    float* grad_log_std;
    float* grad_values;
    double ent_coef;
    WsHead* head;
    double* part3;
};

__global__ void __launch_bounds__(kThreads) ppo_backward_kernel(BackArgs p) {
    __shared__ double s_col[kWarps][32];
    __shared__ int is_last;
    const FleetPpoBatch& b = p.b;
    const int64_t B = b.batch_size;
    const int N = b.action_dim;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t c0 = (int64_t)blockIdx.x * kRows;
    const int64_t row0 = c0 + warp * kRowsPerWarp;
    const float gl = *p.grad_loss;
    if (threadIdx.x < kRows && c0 + threadIdx.x < B)
        p.grad_values[c0 + threadIdx.x] = __fmul_rn(gl, p.coef[B + c0 + threadIdx.x]);
    float g[kRowsPerWarp];
#pragma unroll
    for (int r = 0; r < kRowsPerWarp; r++) g[r] = row0 + r < B ? __fmul_rn(gl, p.coef[row0 + r]) : 0.0f;

    // Column segments of 32: every warp takes its 16 rows; the 8 warps' sums are added in warp order.
    for (int n0 = 0; n0 < N; n0 += 32) {
        const int n = n0 + lane;
        double acc = 0.0;
        if (n < N) {
            float var, log_sig;
            column(b.log_std, n, var, log_sig);
            float mu[kRowsPerWarp], a[kRowsPerWarp];
#pragma unroll
            for (int r = 0; r < kRowsPerWarp; r++) {
                if (row0 + r < B) {
                    const int64_t o = (row0 + r) * N + n;
                    mu[r] = b.mean[o];
                    a[r] = b.actions[o];
                }
            }
#pragma unroll
            for (int r = 0; r < kRowsPerWarp; r++) {
                if (row0 + r < B) {
                    // d log_prob / d mean = (a - mu) / var;  d log_prob / d log_std = (a - mu)^2 / var - 1
                    const float d = __fsub_rn(a[r], mu[r]);
                    p.grad_mean[(row0 + r) * N + n] = __fmul_rn(g[r], __fdiv_rn(d, var));
                    const float q = __fdiv_rn(__fmul_rn(d, d), var);
                    acc += (double)g[r] * ((double)q - 1.0);
                }
            }
        }
        s_col[warp][lane] = acc;
        __syncthreads();
        if (warp == 0 && n < N) {
            double s = 0.0;
#pragma unroll
            for (int w = 0; w < kWarps; w++) s += s_col[w][lane];
            p.part3[(int64_t)blockIdx.x * N + n] = s;
        }
        __syncthreads();
    }
    if (!last_cta(&p.head->tickets[2], &is_last)) return;

    // Last CTA: warp w adds chunks w, w + 8, ... of each column in order; then the warps in order.
    for (int n0 = 0; n0 < N; n0 += 32) {
        const int n = n0 + lane;
        double acc = 0.0;
        if (n < N) {
            int64_t c = warp;
            for (; c + 3 * kWarps < gridDim.x; c += 4 * kWarps) {
                double v[4];
#pragma unroll
                for (int u = 0; u < 4; u++) v[u] = __ldcg(p.part3 + (c + u * kWarps) * N + n);
#pragma unroll
                for (int u = 0; u < 4; u++) acc += v[u];
            }
            for (; c < gridDim.x; c += kWarps) acc += __ldcg(p.part3 + c * N + n);
        }
        s_col[warp][lane] = acc;
        __syncthreads();
        if (warp == 0 && n < N) {
            double s = 0.0;
#pragma unroll
            for (int w = 0; w < kWarps; w++) s += s_col[w][lane];
            // entropy_loss = -mean(sum_n log sigma_n + const): d / d log_std_n = -1
            p.grad_log_std[n] = __double2float_rn(s - (double)gl * p.ent_coef);
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) p.head->tickets[2] = 0;
}

int check_batch(const FleetPpoBatch* b) {
    if (!b) return fail(FLEET_E_INVALID, "batch descriptor is NULL");
    if (b->batch_size < 1 || b->action_dim < 1) return fail(FLEET_E_INVALID, "batch_size and action_dim must be >= 1");
    if (!b->mean || !b->log_std || !b->actions) return fail(FLEET_E_INVALID, "mean, log_std and actions are required");
    if (chunks(b->batch_size, kRows) > 0x7fffffff) return fail(FLEET_E_INVALID, "batch_size too large for one launch");
    return FLEET_OK;
}

int check_loss_inputs(const FleetPpoBatch* b, const FleetPpoParams* p, const void* ws, int64_t ws_bytes) {
    int rc = check_batch(b);
    if (rc) return rc;
    if (!b->values || !b->old_log_prob || !b->advantages || !b->returns)
        return fail(FLEET_E_INVALID, "values, old_log_prob, advantages and returns are required");
    if (!p) return fail(FLEET_E_INVALID, "params is NULL");
    if (!(p->clip_range > 0.0)) return fail(FLEET_E_INVALID, "clip_range must be > 0");
    if (p->clip_range_vf >= 0.0 && !b->old_values)
        return fail(FLEET_E_INVALID, "old_values is required when clip_range_vf is set");
    if (!ws) return fail(FLEET_E_INVALID, "workspace is NULL");
    if (((uintptr_t)ws & 255u) != 0) return fail(FLEET_E_INVALID, "workspace must be 256-byte aligned");
    const int64_t need = ws_layout(b->batch_size, b->action_dim).total;
    if (ws_bytes < need)
        return fail(FLEET_E_INVALID, "workspace of " + std::to_string(ws_bytes) + " bytes is smaller than the " +
                                         std::to_string(need) + " fleet_ppo_workspace_bytes requires");
    return FLEET_OK;
}

float log_sqrt_2pi() { return (float)std::log(std::sqrt(2.0 * M_PI)); }

}  // namespace

int64_t fleet_ppo_workspace_bytes(int64_t batch_size, int32_t action_dim) {
    if (batch_size < 1 || action_dim < 1) return 0;
    return ws_layout(batch_size, action_dim).total;
}

int fleet_ppo_log_prob(const FleetPpoBatch* b, float* log_prob_out, void* stream) {
    int rc = check_batch(b);
    if (rc) return rc;
    if (!log_prob_out) return fail(FLEET_E_INVALID, "log_prob_out is required");
    const int64_t B = b->batch_size;
    ppo_log_prob_kernel<<<(unsigned)chunks(B, kRows), kThreads, 0, (cudaStream_t)stream>>>(
        b->mean, b->actions, b->log_std, log_prob_out, B, b->action_dim, log_sqrt_2pi());
    PPO_TRY(cudaGetLastError());
    return FLEET_OK;
}

int fleet_ppo_loss(const FleetPpoBatch* b, const FleetPpoParams* p, float* loss_out, double* stats_acc,
                   float* sample_coef, void* workspace, int64_t workspace_bytes, void* stream) {
    int rc = check_loss_inputs(b, p, workspace, workspace_bytes);
    if (rc) return rc;
    if (!loss_out || !stats_acc || !sample_coef)
        return fail(FLEET_E_INVALID, "loss_out, stats_acc and sample_coef are required");
    const int64_t B = b->batch_size;
    const WsLayout l = ws_layout(B, b->action_dim);
    char* ws = (char*)workspace;
    LossArgs a;
    a.b = *b;
    // Python computes 1 - clip_range and 1 + clip_range in double; torch rounds the bounds to the tensor's float32.
    a.clip_lo = (float)(1.0 - p->clip_range);
    a.clip_hi = (float)(1.0 + p->clip_range);
    a.clip_eps = (float)p->clip_range;
    a.clip_vf = p->clip_range_vf >= 0.0;
    a.vf_lo = (float)(-p->clip_range_vf);
    a.vf_hi = (float)p->clip_range_vf;
    a.lsp = log_sqrt_2pi();
    a.normalize = p->normalize_advantage && B > 1;
    a.ent_coef = p->ent_coef;
    a.vf_coef = p->vf_coef;
    a.coef = sample_coef;
    a.stats = stats_acc;
    a.loss_out = loss_out;
    a.head = (WsHead*)ws;
    a.ratio = (float*)(ws + l.ratio);
    a.part1 = (double*)(ws + l.part1);
    a.part2 = (double*)(ws + l.part2);
    a.part3 = (double*)(ws + l.part3);
    cudaStream_t s = (cudaStream_t)stream;
    ppo_rows_kernel<<<(unsigned)chunks(B, kRows), kThreads, 0, s>>>(a);
    PPO_TRY(cudaGetLastError());
    ppo_policy_kernel<<<(unsigned)chunks(B, kPolicyRows), kThreads, 0, s>>>(a);
    PPO_TRY(cudaGetLastError());
    return FLEET_OK;
}

int fleet_ppo_loss_backward(const FleetPpoBatch* b, const FleetPpoParams* p, const float* grad_loss,
                            const float* sample_coef, float* grad_mean, float* grad_log_std, float* grad_values,
                            void* workspace, int64_t workspace_bytes, void* stream) {
    int rc = check_loss_inputs(b, p, workspace, workspace_bytes);
    if (rc) return rc;
    if (!grad_loss || !sample_coef || !grad_mean || !grad_log_std || !grad_values)
        return fail(FLEET_E_INVALID, "grad_loss, sample_coef, grad_mean, grad_log_std and grad_values are required");
    const int64_t B = b->batch_size;
    const WsLayout l = ws_layout(B, b->action_dim);
    char* ws = (char*)workspace;
    BackArgs a;
    a.b = *b;
    a.grad_loss = grad_loss;
    a.coef = sample_coef;
    a.grad_mean = grad_mean;
    a.grad_log_std = grad_log_std;
    a.grad_values = grad_values;
    a.ent_coef = p->ent_coef;
    a.head = (WsHead*)ws;
    a.part3 = (double*)(ws + l.part3);
    ppo_backward_kernel<<<(unsigned)chunks(B, kRows), kThreads, 0, (cudaStream_t)stream>>>(a);
    PPO_TRY(cudaGetLastError());
    return FLEET_OK;
}

const char* fleet_ppo_last_error(void) { return g_err.c_str(); }
