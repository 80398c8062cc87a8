// fleetstep.cu — B200 (sm_100a) implementation of the FleetRL environment step behind include/fleetstep.h.
//
// Two launches per fleet_step call, on the caller's stream:
//   step kernel   fleet_step_pf_kernel (persistent, warp-specialised, software-pipelined; auto-reset on, 8 <= N <= 256;
//                 a generic instance and one compiled for the cfg2 fleet shape) or
//                 fleet_step_kernel (generic: any N, frozen envs): EvCharger.charge + LoadCalculation.check_violation +
//                 ScoreConfig penalties + time advance + departure/arrival logic + Observer/Normalization observation
//                 assembly for E envs x N EVs; appends the new soc_deg sample to a small per-env ring and pushes envs that
//                 need more onto a device work list.  The two kernels share the per-vehicle step (ev_slot_step) and
//                 the env-level parts (stage_env_scratch, obs_row_dst, finalise_env); they differ in how inputs are
//                 fetched, how the per-env sums are reduced, how the observation tile is stored and in launch
//                 geometry.
//   post kernel   fleet_post_kernel: incremental rainflow (persistent three-point stack per vehicle) over the ring samples,
//                 at the daily 14:45 trigger RainflowSeiDegradation / EmpiricalDegradation.calculate_degradation, then the
//                 SB3-style auto-reset of finished envs.
//   fleet_reset_kernel  FleetEnv.reset for the masked envs; policy_kernel (rule-based baselines), fleet_log_kernel
//                 (DataLogger rows of selected envs), small gather / scatter / statistics kernels.
// Reference: fleetrl/fleet_env/fleet_environment.py:330-702, utils/ev_charging/ev_charger.py:39-231,
// utils/load_calculation/load_calculation.py:83-94, fleet_env/config/score_config.py:26-41,
// utils/observation/observer_bl_pv.py:12-136, utils/normalization/*.py,
// utils/battery_degradation/rainflow_sei_degradation.py:91-212, empirical_degradation.py:29-99, rainflow 3.2.0.
//
// Mapping (DESIGN.md): a CTA works on tiles of B = floor(256/N) consecutive envs; thread j of the tile owns the
// (env, EV) pair ("slot") j = b*N + n.  All [E][N] state is env-major, so slot j of the tile touches element
// e0*N + j of every array: perfectly coalesced scalar loads/stores with no padding.  Per-env reductions over the
// EVs go through shared memory and are summed in a FIXED order by one lane per (env, quantity) (deterministic run to
// run; a documented re-association of the reference's Python accumulation, DESIGN.md 4).  Everything that depends only
// on the time index (price/tariff factors, PV share, grid margin, the observation header with its look-ahead windows and
// calendar features, the per-(time, EV) schedule record with its auxiliary observation terms) is precomputed once on the
// host in float64 with the reference's operation order and staged in HBM (~64 MB at N=50, T=35040); the kernels gather
// it by time index.
//
// Arithmetic: float64 with -fmad=false (no FMA contraction), operation order of the reference; float32 only where
// the reference casts (observation, reward output) and for hours_left, whose values are exact multiples of dt
// (validated at create time).
//
// The product path has NO CPU fallback: every entry point fails with FLEET_E_CUDA if the device is unusable.
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <string>
#include <vector>

#include "fleetstep.h"

namespace {

constexpr int kThreads = 256;        // threads per CTA
constexpr int kMinCtasPerSm = 4;     // register budget: 64 regs/thread -> 1024 resident threads per SM
constexpr int kStatStripes = 64;     // atomic striping of the statistics vector
// per-slot contributions reduced per env (sequential, car order, one thread per (quantity, env))
constexpr int kNQ = 5;
enum { Q_REWARD = 0, Q_CASH, Q_ATH, Q_MISS, Q_NVIOL };

// per-time flags
constexpr uint32_t TF_TRIGGER = 1u;  // hour == 14 && minute == 45     fleet_environment.py:665
constexpr uint32_t TF_LUNCH = 2u;    // 11 < hour < 15                 fleet_environment.py:538
// StepRow::flags_next carries, above its TF_* bits, the distance from row t to the first 14:45 row at or after t + 2
constexpr int TF_DIST_SHIFT = 8;
constexpr uint32_t TF_DIST_NONE = 0xffffffu;   // no such row (saturated)

// per-env tile flags
//   EF_EVAL_AHEAD   a daily evaluation remains in the episode after this step's (next 14:45 row at or after t + 2 <= t_fin)
constexpr int EF_FROZEN = 1, EF_DONE = 2, EF_TRIGGER = 4, EF_LUNCH = 8, EF_RESET = 16, EF_EVAL_AHEAD = 32;

// One (time, vehicle) schedule record, 32 bytes = one L2 sector: SOC_on_return, time_left, There at this row and
// at the previous row, and the auxiliary observation terms of observer_bl_pv.py:85-91 for the un-raised target
// SOC (pure functions of the schedule row, SURVEY B-4), already normalised when OracleNormalization is on.
struct __align__(16) EvRec {
    double sr;
    float tl;
    uint8_t there, there_prev;
    uint16_t pad;
    float tt, cl, hn, lax;   // target_soc*there, charging_left, hours_needed, laxity (float32 as observed)
};
static_assert(sizeof(EvRec) == 32, "EvRec must be 32 bytes");

// Everything EvCharger.charge / check_violation need that depends only on the time index t (host-precomputed).
struct __align__(16) StepRow {
    double S;         // delu[t]/1000.0 + fixed_markup/1000                       ev_charger.py:145,35,149
    double F_cr;      // ((-1*price_multiplier)*price_reward_curve[t])/1000       ev_charger.py:154-156
    double F_dr;      // ((-1*price_multiplier)*tariff_reward_curve[t])/1000      ev_charger.py:204-206
    double Rfac;      // discharging_eff*tariff[t]/1000*(1-feed_in_deduction)     ev_charger.py:196-199
    double pv_share;  // pv[t]*dt / max(sum(there[:,t]),1)                        ev_charger.py:134-142
    double gml;       // grid_connection - load[t]                                load_calculation.py:93
    double pvv;       // pv[t]
    uint32_t flags;       // TF_* of row t
    uint32_t flags_next;  // TF_* of row t+1 | distance to the first 14:45 row >= t+2 << TF_DIST_SHIFT
};
static_assert(sizeof(StepRow) == 64, "StepRow must be 64 bytes");

struct StepParams {
    // sizes
    int E, N, T, R, Rm, L, D, Ha, Hb, hdr_stride, B;   // R: rows of the soc_deg history ring (power of two), Rm = R - 1
    unsigned long long RN;    // R * N
    unsigned int n_magic;     // ceil(2^32 / N): j / N == __umulhi(j, n_magic) for j < 2^16
    unsigned int h_magic;     // same for the header length Ha+Hb
    int off_contrib, off_obs; // byte offsets of the contribution arrays / obs tile in dynamic shared memory
    // flags
    int is_ct, calc_deg, deg_mode, carry, auto_reset, bulk_ok;
    int rf_on;                // incremental rainflow state is maintained (calc_deg && deg_mode == FLEET_DEG_SEI)
    int start_lo, start_hi;
    unsigned long long seed;
    long long env_id_offset;
    // constants
    double dt, P, eta_c, eta_d, mult, cap0, target, target_lunch, eps, def_soc, min_lax;
    double pen_inv, pen_oc, clip_oc, pen_ovl, full_reward, evse, grid, init_soh, lc_batt_cap, hn_den, price_mult;
    double temperature, max_tl, max_soc, max_hn;
    float dt_f;
    // tables
    const EvRec* ev_rec;      // [T][N]
    const StepRow* step_row;  // [T]
    const float* hdr;         // [T][hdr_stride]
    // state
    int4* env4;               // [E] {t, t_start, ep_count, k_done}: k_done = newest history sample the rainflow state has consumed;
                              // once no daily evaluation remains in the episode the ring may wrap over unconsumed samples
                              // and k_done lag by more than R - 1 (wl_flags): nothing reads them before the reset
    double* soc;              // [E][N]
    float* hl;                // [E][N]
    double* soh;              // [E][N]
    double* hist;             // [E][R][N] ring of soc_deg samples: sample k of the episode lives in row k & Rm
    uint8_t* tflip;           // [E][N] target_soc raised to 0.9 (fleet_environment.py:613-614)
    int* n_flips;             // [1] number of set tflip bytes (0 => the array is never read)
    double* env_f64;          // [6][E] ep_return, last_ep_return, reward64, cashflow, overload, soc_viol
    int* rf_len;              // [E][N] RainflowSeiDegradation.rainflow_length
    double* fd_cyc;           // [E][N]
    double* life;             // [E][N]
    int* n_cycles;            // [E][N]
    double* last_deg;         // [E][N]
    // incremental rainflow (DESIGN.md 3.2): the three-point stack of rainflow.extract_cycles persists per vehicle
    int rf_S, rf_X, rf_P;     // inline stack entries per vehicle, entries per extension slot, number of extension slots
    double* rf_stack;         // [E][N][S] committed reversal points still on the stack (entry 0 = bottom)
    unsigned int* rf_dc;      // [E][N] stack depth | committed cycles of the episode << 16
    double2* rf_acc;          // [E][N] {sum of the means of the committed cycles, stress sum of those at list positions >= rainflow_length-1}
    int* rf_ext;              // [E][N] extension slot holding stack entries >= S, or -1
    int* ext_owner;           // [P] vehicle index owning the slot, or -1
    double* ext_val;          // [P][X]
    double* charge_log;       // [E][N] or nullptr: energy into (+) / out of (-) each battery in the last step
    double* stats;            // [kStatStripes][FLEET_S__COUNT]
    unsigned int* err_flags;  // [1]
    const int* next_start;    // [E] or nullptr
    int2* wl;                 // [E] work list of the post kernel: {env, WL_* flags}
    int4* wl_flush;           // [E] flush-only entries of the post kernel: {env, k_done, k_now, -}
    int* wl_count;            // [8] {entries pushed from the front, next entry to fetch, entries pushed from the back,
                              //      flush-only entries, next flush unit to fetch, -, -, -}
    unsigned int* wl_done;    // [1]
    int* wl_chunks;           // [E] per work-list entry: chunks of it that have finished (self-clearing), or nullptr
    int post_chunks, post_cv; // post kernel: work items per entry, vehicles per item
    // persistent step kernel geometry (host-computed so that the kernel reads it from the constant bank, not registers)
    int pf_B, pf_bulk, pf_ntiles, pf_cslots, pf_cper, pf_pair;      // pf_B: envs per tile = kPfSlots / N
    int pf_pad;                                               // unused: keeps the fields below at their constant-bank offsets
                                                              // (moving them changes how ptxas pairs and schedules their loads)
    unsigned int pf_tile_hist;                               // B * RN: history elements per tile (< 2^32, checked at create)
    int pf_envs_b, pf_contrib_b, pf_obs_b;                    // bytes of one env-scratch / contribution / obs buffer
    int pf_off_contrib, pf_off_sums, pf_off_obs, pf_off_stage;   // shared-memory offsets
    // I/O
    const float* actions;
    float* obs;
    float* reward;
    uint8_t* done;
    float* terminal_obs;
    // reset kernel only
    const int* start_idx;
    const uint8_t* mask;
};

enum { EF_EP_RETURN = 0, EF_LAST_EP_RETURN, EF_REWARD64, EF_CASHFLOW, EF_OVERLOAD, EF_SOC_VIOL, EF__COUNT };

struct EnvS {  // per-env scratch of a tile, shared memory (both step kernels; stage_env_scratch fills it)
    int t, t_start, ep_count, flags;
    double S, F_cr, F_dr, Rfac, pv_share, gml, pvv;
    int k_done, pad;
};

__device__ __forceinline__ unsigned long long mix64(unsigned long long z) {
    z += 0x9E3779B97F4A7C15ull;
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    return z ^ (z >> 31);
}
// Counter-based start-index draw keyed by (seed, global env id, episode number): integer work, bit-exact with
// the oracle's draw_start.  Replaces the reference's unseeded random.choice (random_time_picker.py:31).
__device__ __forceinline__ int draw_start(unsigned long long seed, int start_lo, int start_hi, long long env_id,
                                          int episode_no) {
    unsigned long long h =
        mix64(seed ^ mix64((unsigned long long)env_id * 0xD1B54A32D192ED03ull + (unsigned long long)(unsigned)episode_no));
    unsigned long long span = (unsigned long long)(start_hi - start_lo) + 1ull;
    return start_lo + (int)(h % span);
}
// Start index of env e's next episode: starts[e] when the caller supplies start indices, else the draw for episode
// ep_count (the number of episodes the env has begun so far).
__device__ __forceinline__ int episode_start(const StepParams& p, const int* starts, int e, int ep_count) {
    return starts ? starts[e] : draw_start(p.seed, p.start_lo, p.start_hi, p.env_id_offset + e, ep_count);
}
// env4 and episode return of env e when its next episode begins at time index t0.
__device__ __forceinline__ void begin_episode(const StepParams& p, int e, int t0, int ep_count) {
    p.env4[e] = make_int4(t0, t0, ep_count + 1, 0);
    p.env_f64[(size_t)EF_EP_RETURN * p.E + e] = 0;
}


// L2 residency: the time-indexed tables and the per-env time index are re-read every step by (other) envs, the
// [E][N] state streams through once per step.  Table / env4 accesses carry an evict_last policy, streaming state
// uses evict-first (ld.global.cs / st.global.cs).
__device__ __forceinline__ uint64_t l2_evict_last_policy() {
    uint64_t pol;
    asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(pol));
    return pol;
}
__device__ __forceinline__ int4 ld_keep_v4(const void* ptr, uint64_t pol) {
    int4 v;
    asm volatile("ld.global.L2::cache_hint.v4.s32 {%0,%1,%2,%3}, [%4], %5;"
                 : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(ptr), "l"(pol));
    return v;
}
__device__ __forceinline__ float ld_keep_f32(const float* ptr, uint64_t pol) {
    float v;
    asm volatile("ld.global.L2::cache_hint.f32 %0, [%1], %2;" : "=f"(v) : "l"(ptr), "l"(pol));
    return v;
}
__device__ __forceinline__ void st_keep_v4(void* ptr, int4 v, uint64_t pol) {
    asm volatile("st.global.L2::cache_hint.v4.s32 [%0], {%1,%2,%3,%4}, %5;"
                 :: "l"(ptr), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w), "l"(pol) : "memory");
}

// An EvRec from the two 128-bit halves of its 32-byte sector.
__device__ __forceinline__ EvRec decode_rec(int4 v, int4 w) {
    EvRec r;
    r.sr = __hiloint2double(v.y, v.x);
    r.tl = __int_as_float(v.z);
    r.there = (uint8_t)(v.w & 0xff);
    r.there_prev = (uint8_t)((v.w >> 8) & 0xff);
    r.pad = 0;
    r.tt = __int_as_float(w.x); r.cl = __int_as_float(w.y); r.hn = __int_as_float(w.z); r.lax = __int_as_float(w.w);
    return r;
}

__device__ __forceinline__ EvRec load_rec(const EvRec* ptr) {
    // two 128-bit read-only loads of one 32-byte sector (tables keep the default L2 policy; streaming state uses
    // evict-first loads/stores so the tables stay resident)
    return decode_rec(__ldg(reinterpret_cast<const int4*>(ptr)), __ldg(reinterpret_cast<const int4*>(ptr) + 1));
}

__device__ __forceinline__ EvRec load_rec_keep(const EvRec* ptr, uint64_t pol) {
    return decode_rec(ld_keep_v4(ptr, pol), ld_keep_v4(reinterpret_cast<const int4*>(ptr) + 1, pol));
}

// Auxiliary observation terms for a vehicle whose target SOC was raised to 0.9 (rare; the table holds the values
// for the configured target): observer_bl_pv.py:85-91, oracle_normalization.py:146-150.
template <bool kNorm>
__device__ __noinline__ float4 aux_on_the_fly(double tgt, double sr, float tl, int there, double lc_batt_cap, double hn_den,
                                              double max_soc, double max_hn) {
    const double th = (double)there;
    double tt = tgt * th;
    double cl = tt - sr;
    double hn = cl * lc_batt_cap / hn_den;
    double lax = ((double)tl / (hn + 0.001) - 1) * th;
    lax = lax < 0 ? 0 : (lax > 5 ? 5 : lax);
    if (kNorm) { tt = tt / max_soc; cl = cl / max_soc; hn = hn / max_hn; lax = lax / 5; }
    return make_float4((float)tt, (float)cl, (float)hn, (float)lax);
}

// Per-EV part of the observation row `o` (global or shared memory): simulated soc / hours_left
// (fleet_environment.py:645-649, oracle_normalization.py:65-66) and the auxiliary block.
template <bool kNorm, bool kAux>
__device__ __forceinline__ void write_ev_obs(const StepParams& p, float* __restrict__ o, int n, double soc, float hl,
                                             const EvRec& rec, bool flip) {
    const int N = p.N;
    o[n] = (float)soc;
    o[N + n] = kNorm ? (float)((double)hl / p.max_tl) : hl;
    if (kAux) {
        float4 ax = make_float4(rec.tt, rec.cl, rec.hn, rec.lax);
        if (flip) ax = aux_on_the_fly<kNorm>(0.9, rec.sr, rec.tl, rec.there, p.lc_batt_cap, p.hn_den, p.max_soc, p.max_hn);
        float* a = o + 2 * N + p.Ha;
        a[n] = (float)rec.there;
        a[N + n] = ax.x;
        a[2 * N + n] = ax.y;
        a[3 * N + n] = ax.z;
        a[4 * N + n] = ax.w;
    }
}

// Time-only part of the observation (price/tariff/load/pv windows, evse/grid terms, calendar sin/cos): a host-
// precomputed float32 row of Ha + Hb elements per time index.  Element q of it goes to position hdr_pos(q) of the
// observation row: the first Ha after the per-EV soc / hours_left, the Hb others (aux only) after the auxiliary block.
template <bool kAux>
__device__ __forceinline__ int hdr_pos(int Ha, int N, int q) {
    return q < Ha ? 2 * N + q : 2 * N + Ha + (kAux ? 5 * N : 0) + (q - Ha);
}
// The header row of time t, copied by the env's slot threads.  Without aux Hb is 0 and the bound is written as Ha: as a
// compile-time choice it keeps fleet_reset_kernel one register lower.
template <bool kAux>
__device__ __forceinline__ void copy_hdr(const StepParams& p, float* __restrict__ o, int n, int t) {
    const float* __restrict__ h = p.hdr + (size_t)t * p.hdr_stride;
    for (int q = n; q < (kAux ? p.Ha + p.Hb : p.Ha); q += p.N) o[hdr_pos<kAux>(p.Ha, p.N, q)] = __ldg(h + q);
}

// FleetEnv.reset for one (env, EV) slot: fleet_environment.py:345-348, 371-372, 382-399.
template <bool kNorm, bool kAux>
__device__ __forceinline__ void reset_slot(const StepParams& p, int e, int n, int t0, float* obs_row, bool reinit_deg) {
    const size_t i = (size_t)e * p.N + n;
    const EvRec rec = load_rec(&p.ev_rec[(size_t)t0 * p.N + n]);
    bool flip = false;
    if (reinit_deg) {
        // fresh-object semantics (carry_degradation_state == 0): re-initialise what lives on the reference's
        // env / degradation objects (rainflow_sei_degradation.py:31-34,57-60; fleet_environment.py:263)
        p.rf_len[i] = 1; p.fd_cyc[i] = 0; p.life[i] = 1 - p.init_soh;
        p.tflip[i] = 0;
    } else if (*p.n_flips != 0) {
        flip = p.tflip[i] != 0;
    }
    const double tgt = flip ? 0.9 : p.target;
    const double soh = 1.0 * p.init_soh;
    const double cap = soh * p.cap0;
    double soc = rec.sr;
    const float hl = rec.tl;
    const double time_needed = (tgt - soc) * cap / p.P;
    if (hl > 0.f && p.min_lax * time_needed > (double)hl) soc = tgt - (time_needed * p.P / cap) / p.min_lax;
    const double sdeg = (soc == 0) ? p.def_soc : soc;
    p.soc[i] = soc;
    p.hl[i] = hl;
    p.soh[i] = soh;
    p.hist[((size_t)e * p.R + 0) * p.N + n] = sdeg;                 // LogDataDeg.soc_log restarts with this sample
    if (p.rf_on) {
        // rainflow state of the new episode: the first sample is the first point on the stack, no cycles yet
        // (the rainflow_length / fd_cyc / l members above survive unless reinit_deg)
        const int slot = p.rf_ext[i];
        if (slot >= 0) { atomicExch(&p.ext_owner[slot], -1); p.rf_ext[i] = -1; }
        p.rf_stack[i * (size_t)p.rf_S] = sdeg;
        p.rf_dc[i] = 1u;
        p.rf_acc[i] = make_double2(0.0, 0.0);
    }
    if (obs_row) {
        write_ev_obs<kNorm, kAux>(p, obs_row, n, soc, hl, rec, flip);
        copy_hdr<kAux>(p, obs_row, n, t0);
    }
}

// ------------------------------------------------------------------------------------------------ degradation
// rainflow 3.2.0 extract_cycles (ASTM E1049-85 three-point method) feeding RainflowSeiDegradation.calculate_degradation
// (rainflow_sei_degradation.py:128-206), INCREMENTALLY.
//
// The reference re-runs extract_cycles over the whole soc_log of the episode at every daily evaluation.  Both halves of
// that algorithm are streaming: reversals() is causal except for the provisional last sample, and the three-point stack
// only ever looks at its top three points.  So per vehicle the committed state is kept in HBM between evaluations:
//   * the stack of reversal points that have not been paired off yet (values only; entry 0 = bottom),
//   * c = number of cycles emitted so far (they form a stable prefix of the list the reference would build),
//   * the running sum of their means (the reference averages the means of ALL cycles, :140),
//   * the stress sum of those committed cycles whose list position is >= rainflow_length-1, i.e. the part of the
//     positional slice [rainflow_length-1 : len-1] (:146) that is already final.
// The step kernel only appends soc_deg samples to a small per-env ring (hist).  The post kernel consumes the ring
// (at the daily trigger, or earlier when the ring is about to wrap): reversal detection continues from the last
// consumed sample (the direction of the last non-zero difference is the sign of x_cur - top of stack, because the top
// of the stack is always the most recently yielded reversal), reversals are pushed, closed cycles are committed.
// An evaluation then pushes the provisional end point onto a READ-ONLY view of the stack and counts the residue.
#ifdef POST_TIMING   // diagnostic build: cycles per phase of the post kernel, taken by thread 0 of every CTA (scripts/post_timing.py)
// (slots 1-14: work-list entries; slot 15: flush units, slot 0: their cycles, taken by lane 0 of every warp)
__device__ unsigned long long g_post_clk[16];
#ifdef POST_TIMING_EVAL_ONLY   /* only the entries with a daily evaluation are timed */
#define PT_ON(c_) (c_)
#else
#define PT_ON(c_) true
#endif
#define PT_START2(k_, c_) long long _pt = clock64(); const bool _pt_on = (k_) && PT_ON(c_)
#define PT_START(c_) PT_START2(true, c_)
#define PT_MARK(k) do { if (threadIdx.x == 0 && _pt_on) { const long long _c = clock64(); atomicAdd(&g_post_clk[k], (unsigned long long)(_c - _pt)); _pt = _c; } } while (0)
#define PT_COUNT(k, n) do { if (threadIdx.x == 0 && _pt_on) atomicAdd(&g_post_clk[k], (unsigned long long)(n)); } while (0)
#else
#define PT_START(c_) do {} while (0)
#define PT_START2(k_, c_) do {} while (0)
#define PT_MARK(k) do {} while (0)
#define PT_COUNT(k, n) do {} while (0)
#endif
constexpr int kPostThreads = 64;   // threads per CTA of the post kernel (one work-list env per CTA, one vehicle per thread)
constexpr int kRfBatch = 8;        // history rows in flight per lane while scanning
constexpr int kRfQueue = 12;       // reversal values queued per lane between two runs of the three-point stack
constexpr int kRfPend = 8;         // cycles per lane waiting for their stress evaluation (even)
constexpr int kPostMinCtas = 8;    // resident CTAs per SM of the two-warp post kernel (twice as many of the one-warp one)

// SEI stress of one cycle: rainflow_sei_degradation.py:68-79 with effective DoD = clip(range*count, 0, 1) (:170):
//     S_dod = 1 / (kd1 * dod ** kd2 + kd3)   (:68)      S_soc = exp(k_sigma * (mean - sigma_ref))   (:70)
// with the general-purpose log / exp: dod ** kd2 as exp(kd2 * log(dod)).  Measured against extended precision over 3.5 M
// arguments (tests/test_gpu_parity.py::test_sei_stress_accuracy, which asserts < 5e-14): largest relative error 3.5e-15,
// far inside the 1e-12 stated for fd_cyc against the reference.  dod == 0 gives exp(+inf) = inf -> stress 0.
__device__ __forceinline__ double sei_cycle_stress(double range, double count, double mean, double s_temp) {
    const double k_sigma = 1.04, sigma_ref = 0.5, kd1 = 1.4E5, kd2 = -5.01E-1, kd3 = -1.23E5;
    double eff = range * count;
    eff = eff < 0 ? 0 : (eff > 1 ? 1 : eff);
    // a few ulp off a correctly rounded pow (|kd2 log dod| < 20)
    const double s_dod = 1.0 / (kd1 * exp(kd2 * log(eff)) + kd3);              // :68
    const double s_soc = exp(k_sigma * (mean - sigma_ref));                    // :70
    return s_dod * s_soc * s_temp;                                             // :77-79
}

// diagnostic: the stress function over arrays (accuracy test)
__global__ void debug_stress_kernel(const double* eff, const double* mean, double* out, int n) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = sei_cycle_stress(eff[i], 1.0, mean[i], 1.0);
}

// Claim a stack extension slot for vehicle `vid` (open addressing over the owner table; rare path).
__device__ __noinline__ int rf_ext_alloc(const StepParams& p, size_t vid) {
    const unsigned P = (unsigned)p.rf_P;
    if (P == 0) return -1;
    unsigned q = (unsigned)(mix64((unsigned long long)vid) % P);
    for (unsigned k = 0; k < P; k++) {
        if (atomicCAS(&p.ext_owner[q], -1, (int)vid) == -1) return (int)q;
        if (++q == P) q = 0;
    }
    return -1;
}

// EmpiricalDegradation.calculate_degradation for one vehicle (empirical_degradation.py:60-94).
__device__ __forceinline__ double empirical_eval(double dt, double evse, double old_soc, double new_soc) {
    const double avg_soc = (old_soc + new_soc) / 2;
    const double cs[3] = {0, 40, 90};
    const double ca[3] = {0.0065, 0.0293, 0.065};
    int best = 0;
    double bd = fabs(cs[0] - avg_soc);
#pragma unroll
    for (int k = 1; k < 3; k++) {
        const double d = fabs(cs[k] - avg_soc);
        if (d < bd) { bd = d; best = k; }
    }
    const double cal = ca[best] * dt / 8760;
    const double dod = fabs(new_soc - old_soc);
    const double cyc = (evse <= 22.0) ? dod * 0.000125 / 2 : dod * 0.000167 / 2;
    return cal + cyc;
}

// asynchronous global->shared copies (LDGSTS): no register staging, any number in flight per thread; each carries an L2
// cache policy (createpolicy): evict_first for streamed state, evict_last for the tables
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int kPending>
__device__ __forceinline__ void cp_async_wait_group() { asm volatile("cp.async.wait_group %0;" :: "n"(kPending) : "memory"); }
__device__ __forceinline__ void cp_async4_hint(uint32_t sdst, const void* gsrc, uint64_t pol) {
    asm volatile("cp.async.ca.shared.global.L2::cache_hint [%0], [%1], 4, %2;" :: "r"(sdst), "l"(gsrc), "l"(pol) : "memory");
}
__device__ __forceinline__ void cp_async8_hint(uint32_t sdst, const void* gsrc, uint64_t pol) {
    asm volatile("cp.async.ca.shared.global.L2::cache_hint [%0], [%1], 8, %2;" :: "r"(sdst), "l"(gsrc), "l"(pol) : "memory");
}
__device__ __forceinline__ void cp_async16_hint(uint32_t sdst, const void* gsrc, uint64_t pol) {
    asm volatile("cp.async.cg.shared.global.L2::cache_hint [%0], [%1], 16, %2;" :: "r"(sdst), "l"(gsrc), "l"(pol) : "memory");
}
__device__ __forceinline__ uint64_t l2_evict_first_policy() {
    uint64_t pol;
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
    return pol;
}

// RainflowSeiDegradation.calculate_degradation once the cycle list is known (rainflow_sei_degradation.py:128-206):
// m cycles in the list, msum = sum of their means, fsum = stress of the slice [rainflow_length-1 : m-1].  Updates
// fd_cyc / l / rainflow_length / soh of vehicle i and returns the SOH loss.
__device__ __forceinline__ double sei_fade_update(const StepParams& p, size_t i, int len, int m, int rfl, double msum,
                                                  double fsum, bool big, double s_temp, bool& consumed) {
    const double alpha_sei = 5.75E-2, beta_sei = 121, k_sigma = 1.04, sigma_ref = 0.5, k_dt = 4.14E-10;
    double deg = 0;
    consumed = false;
    p.n_cycles[i] = m;
    if (m > rfl) {                                                                     // :143
        const double battery_age = (double)(len - 1) * p.dt * 3600;                    // :138  max(End) == len-1
        const double mean_soc_cal = msum / (double)m;                                  // :140
        if (big) atomicOr(p.err_flags, 4u);                                            // :164-167
        const double fd_cal = (k_dt * battery_age) * exp(k_sigma * (mean_soc_cal - sigma_ref)) * s_temp;  // :81-83
        const double fd_cyc = p.fd_cyc[i] + fsum;                                      // :174
        p.fd_cyc[i] = fd_cyc;
        const double fd = fd_cyc + fd_cal;
        const double l_old = p.life[i];
        double new_l;
        if (p.init_soh == 1.0) {
            new_l = 1 - alpha_sei * exp(-beta_sei * fd) - (1 - alpha_sei) * exp(-fd);  // :85-86
            if (new_l < 0) atomicOr(p.err_flags, 2u);                                  // :179-180
        } else {
            new_l = 1 - (1 - l_old) * exp(-fd);                                        // :89,186
        }
        deg = new_l - l_old;                                                           // :189
        p.life[i] = new_l;                                                             // :192
        p.rf_len[i] = m;                                                               // :195
        consumed = true;
    }
    p.last_deg[i] = deg;
    p.soh[i] = p.soh[i] - deg;                                                         // :671 (battery_cap is derived, :673)
    return deg;
}

// GENERAL (slow) path for one vehicle: plain serial code straight on the vehicle's stack storage in HBM (inline entries +
// extension slot), any depth up to S + X.  Taken by the few vehicles whose stack is, or becomes, deeper than the
// shared-memory copy of the fast path below.  Same arithmetic, same order of the cycle list.
__device__ __noinline__ double rf_vehicle_slow(const StepParams& p, int e, int n, int k_done, int k_now, bool evaluate,
                                               double s_temp) {
    const int N = p.N, S = p.rf_S, X = p.rf_X, Rm = p.Rm;
    const size_t i = (size_t)e * N + n;
    const unsigned int dc = p.rf_dc[i];
    int depth = (int)(dc & 0xffffu), c = (int)(dc >> 16);
    double2 acc = p.rf_acc[i];
    int slot = p.rf_ext[i];
    const int rfl = p.rf_len[i];
    const double* hcol = p.hist + (size_t)e * p.RN + n;
    double* stk = p.rf_stack + i * (size_t)S;
    double* ext = slot >= 0 ? p.ext_val + (size_t)slot * X : nullptr;
#define RF_GET(s_) ((s_) < S ? stk[(s_)] : ext[(s_) - S])
#define RF_PUT(s_, v_) do { if ((s_) < S) stk[(s_)] = (v_); else ext[(s_) - S] = (v_); } while (0)
    bool bad = false, big = false;
    double x_cur = hcol[(size_t)(k_done & Rm) * N];
    double dsg = x_cur - RF_GET(depth - 1);
    for (int r = k_done + 1; r <= k_now; r++) {
        const double x_next = hcol[(size_t)(r & Rm) * N];
        if (x_next == x_cur) continue;
        const double d = x_next - x_cur;
        if ((dsg < 0 && d > 0) || (dsg > 0 && d < 0)) {      // x_cur is a reversal: push it
            if (depth >= S && !ext) {
                slot = (depth < S + X) ? rf_ext_alloc(p, i) : -1;
                if (slot >= 0) ext = p.ext_val + (size_t)slot * X;
            }
            if (depth >= S + X || (depth >= S && !ext)) bad = true;               // capacity exceeded: dropped, flagged
            else {
                RF_PUT(depth, x_cur); depth++;
                while (depth >= 3) {
                    const double x3 = RF_GET(depth - 1), x2 = RF_GET(depth - 2), x1 = RF_GET(depth - 3);
                    if (fabs(x3 - x2) < fabs(x2 - x1)) break;
                    const double range = fabs(x1 - x2), mean = 0.5 * (x1 + x2);
                    const bool half = depth == 3;
                    acc.x += mean;
                    if (c >= rfl - 1) { acc.y += sei_cycle_stress(range, half ? 0.5 : 1.0, mean, s_temp); big = big || range > 5; }
                    c++;
                    if (half) { RF_PUT(0, x2); RF_PUT(1, x3); depth = 2; }        // popleft
                    else { RF_PUT(depth - 3, x3); depth -= 2; }
                }
            }
        }
        dsg = d; x_cur = x_next;
    }
    if (bad) atomicOr(p.err_flags, 8u);
    double deg = 0;
    if (evaluate) {
        const int len = k_now + 1;
        int m = c, h = depth, lo = 0;
        double msum = acc.x, fs = 0;
        if (len >= 3) {
            auto prov = [&](double xa, double xb, double cnt, bool last) {
                const double range = fabs(xa - xb), mean = 0.5 * (xa + xb);
                msum += mean;
                if (!last && m >= rfl - 1) { fs += sei_cycle_stress(range, cnt, mean, s_temp); big = big || range > 5; }
                m++;
            };
            while (h - lo >= 2) {
                const double x2 = RF_GET(h - 1), x1 = RF_GET(h - 2);
                if (fabs(x_cur - x2) < fabs(x2 - x1)) break;
                if (h - lo == 2) { prov(x1, x2, 0.5, false); lo++; }
                else { prov(x1, x2, 1.0, false); h -= 2; }
            }
            for (int k = lo; k + 1 < h; k++) prov(RF_GET(k), RF_GET(k + 1), 0.5, false);
            prov(RF_GET(h - 1), x_cur, 0.5, true);
        }
        bool consumed;
        deg = sei_fade_update(p, i, len, m, rfl, msum, acc.y + fs, big, s_temp, consumed);
        if (consumed) acc.y = 0;
    }
#undef RF_GET
#undef RF_PUT
    if (slot >= 0 && depth <= S) { atomicExch(&p.ext_owner[slot], -1); slot = -1; }
    p.rf_dc[i] = (unsigned int)depth | ((unsigned int)c << 16);
    p.rf_acc[i] = acc;
    p.rf_ext[i] = slot;
    return deg;
}

// FAST path, one vehicle per lane, WARP-SYNCHRONOUS (all 32 lanes call it; `active` = the lane has a vehicle): consume
// history samples k_done+1 .. k_now, then (kEval && evaluate) run calculate_degradation.  e, k_done and k_now may differ
// from lane to lane (flush units span envs); `evaluate` must be uniform over the warp.
//   smcol   this thread's column of the stack copy: entry s at smcol[s * kPostThreads], s < S (a vehicle whose stack is
//           or gets deeper leaves for rf_vehicle_slow with its HBM state untouched); the top two entries are carried in
//           registers (t1 = top, t2 = below) together with Y = |t1 - t2| (+inf while there is only one point)
//   qcol    its column of the reversal queue
//   pcol    its column of cycles {range * count, mean} waiting for their SEI stress
// The lanes of a warp scan the history rows in lock-step (coalesced loads, eight in flight, branch-free) and queue the
// reversal values; whenever a queue could overflow, and at the end, the queues are emptied by the three-point stack.
// The vehicles of a warp have different numbers of reversals and closures, so the stack is cut into micro-operations
// and every loop iteration performs one per lane: try to place the next reversal, which either lands on the stack (or
// closes a half cycle) and is consumed, or closes one full cycle and stays.  The log/exp of the SEI stress model never
// run inside that loop: cycles that need them are appended to the warp's list, which all 32 lanes evaluate together
// (one cycle per lane, whoever owns it); each owner then adds up its own results in list order (deterministic).
// Returns the SOH loss (0 unless evaluated).
template <int kT, bool kEval>
__device__ __forceinline__ double rf_vehicle(const StepParams& p, int e, int n, bool active, int k_done, int k_now,
                                             bool evaluate, double s_temp, double* __restrict__ smcol,
                                             double* __restrict__ qcol, double2* __restrict__ pcol) {
    const unsigned full = 0xffffffffu;
    const int N = p.N, S = p.rf_S, Rm = p.Rm;
    const double inf = __longlong_as_double(0x7ff0000000000000ll);
    const size_t i = (size_t)e * N + (active ? n : 0);
    const double* __restrict__ hcol = p.hist + (size_t)e * p.RN + (active ? n : 0);   // sample k at hcol[(k & Rm) * N]
    double* __restrict__ stk = p.rf_stack + i * (size_t)S;                            // entry s at stk[s]
    int depth = 1, c = 0, rflm1 = 0;
    double2 acc = make_double2(0.0, 0.0);                    // x: sum of committed means, y: pending stress sum
    double x_cur = 0;
    if (active) {                                            // everything this lane needs, one round trip
        const unsigned int dc = p.rf_dc[i];
        acc = p.rf_acc[i];
        rflm1 = p.rf_len[i] - 1;
        x_cur = __ldcs(hcol + (size_t)(k_done & Rm) * N);
        for (int s = 0; s < S; s += 2) {                     // (S is even; entries >= depth are don't-cares)
            const double2 v2 = *reinterpret_cast<const double2*>(stk + s);
            smcol[s * kT] = v2.x; smcol[(s + 1) * kT] = v2.y;
        }
        depth = (int)(dc & 0xffffu); c = (int)(dc >> 16);
    }
    bool slow = active && depth > S;                         // this lane's vehicle takes the general path
    bool live = active && !slow;
    PT_START2(kEval, evaluate);
    double t1 = 0, t2 = 0, Y = inf;
    if (live) {
        t1 = smcol[(depth - 1) * kT];
        if (depth >= 2) { t2 = smcol[(depth - 2) * kT]; Y = fabs(t1 - t2); }
    }
    double dsg = live ? x_cur - t1 : 0.0;                    // sign of the last non-zero difference (0: none yet)
    bool big = false;
    int np = 0;                                              // this lane's cycles waiting for their stress
    bool has_item = false;
    double item_eff = 0, item_mean = 0;
    // (converged code) a lane's new cycle goes to its own pending column; when a column is full, and at the end, all
    // lanes evaluate their columns together, two cycles per iteration (two independent log/exp chains in flight), and add
    // the results up in list order
#define RF_APPEND(target_)                                                                     \
    do {                                                                                       \
        if (has_item) { pcol[np * kT] = make_double2(item_eff, item_mean); np++; has_item = false; } \
        if (__any_sync(full, np == kRfPend)) RF_DRAIN(target_);                                \
    } while (0)
#define RF_DRAIN(target_)                                                                      \
    do {                                                                                       \
        const int m_ = __reduce_max_sync(full, np);                                            \
        for (int k_ = 0; k_ < m_; k_ += 2) {                                                   \
            const double2 i0_ = pcol[min(k_, kRfPend - 1) * kT];                     \
            const double2 i1_ = pcol[min(k_ + 1, kRfPend - 1) * kT];                 \
            const double s0_ = sei_cycle_stress(i0_.x, 1.0, i0_.y, s_temp);                    \
            const double s1_ = sei_cycle_stress(i1_.x, 1.0, i1_.y, s_temp);                    \
            if (k_ < np) (target_) += s0_;                                                     \
            if (k_ + 1 < np) (target_) += s1_;                                                 \
        }                                                                                      \
        np = 0;                                                                                \
    } while (0)

    // ---- committed part: rainflow.reversals + extract_cycles over the pending samples
    int nq = 0;                                              // queued reversals
    for (int r0 = k_done + 1; ; r0 += kRfBatch) {
        const bool more = r0 <= k_now;                       // (lanes with fewer pending rows run on with d == 0)
        // extract_cycles(): empty the queues when the next batch might not fit, and after the last row
        if (__any_sync(full, more ? nq > kRfQueue - kRfBatch : nq > 0)) {
            PT_MARK(2);
            int q = 0;
            while (__any_sync(full, q < nq)) {
                // One micro-operation per lane, written without branches (the three outcomes would otherwise run one
                // after the other in almost every iteration).  With v the reversal to place and X = |v - t1|:
                //   X < Y                 read the next point: t2 spills to the copy, (t2, t1) <- (t1, v), Y <- X
                //   X >= Y, two points    Y contains the starting point: half cycle (t2, t1), popleft, (t2, t1) <- (t1, v), Y <- X
                //   X >= Y, more points   full cycle (t2, t1): discard its peak and valley, refill (t2, t1) from the copy; v stays
                const bool act = q < nq;
                const double v = qcol[min(q, kRfQueue - 1) * kT];
                const double X = fabs(v - t1);
                const bool lt = X < Y, two = depth == 2;
                const bool closing = act && !lt;
                const bool full_c = closing && !two;
                const bool consume = act && (lt || two);
                const bool push = act && lt;
                if (push && depth >= S) { slow = true; live = false; nq = 0; }     // outgrows the copy: general path (rare)
                else {
                    const double mean = 0.5 * (t2 + t1);
                    acc.x += closing ? mean : 0.0;
                    has_item = closing && c >= rflm1;
                    item_eff = two ? 0.5 * Y : Y; item_mean = mean;
                    big = big || (closing && Y > 5);
                    c += closing ? 1 : 0;
                    if (push) smcol[max(depth - 2, 0) * kT] = t2;
                    depth += push ? 1 : (full_c ? -2 : 0);
                    const double s1 = smcol[max(depth - 1, 0) * kT], s2 = smcol[max(depth - 2, 0) * kT];
                    t2 = consume ? t1 : (full_c ? s2 : t2);
                    t1 = consume ? v : (full_c ? s1 : t1);
                    Y = consume ? X : (full_c ? (depth >= 2 ? fabs(t1 - t2) : inf) : Y);
                    q += consume ? 1 : 0;
                }
                PT_COUNT(10, 1);
                RF_APPEND(acc.y);
            }
            nq = 0;
            PT_MARK(3);
        }
        if (!__any_sync(full, more)) break;
        // reversals(): eight rows in flight, lock-step over the lanes, no branches.  Rows past k_now repeat the last
        // sample (d == 0: nothing happens); d_last * d_next < 0 is the reference's own test.
        double xb[kRfBatch];
#pragma unroll
        for (int u = 0; u < kRfBatch; u++) xb[u] = __ldcs(hcol + (size_t)(min(r0 + u, k_now) & Rm) * N);
#pragma unroll
        for (int u = 0; u < kRfBatch; u++) {
            const double d = xb[u] - x_cur;
            const bool flip = live && (dsg * d < 0);
            if (flip) { qcol[nq * kT] = x_cur; nq++; }
            dsg = (d != 0) ? d : dsg;
            x_cur = live ? xb[u] : x_cur;
        }
    }
    RF_DRAIN(acc.y);
    PT_MARK(4);
    // the top two entries go back to the stack copy
    if (live) { smcol[(depth - 1) * kT] = t1; if (depth >= 2) smcol[(depth - 2) * kT] = t2; }

    // ---- evaluation: the provisional end point x_cur on a READ-ONLY view stack[lo .. h) of the committed points
    double deg = 0;
    if (kEval && evaluate) {                                 // (uniform over the warp)
        const int len = k_now + 1;                           // samples in the reference's soc_log
        int m = c, h = depth, lo = 0, k = 0;
        double msum = acc.x, fs = 0;
        int phase = (live && len >= 3) ? 0 : 2;              // 0: closures, 1: residue, 2: done
        while (__any_sync(full, phase < 2)) {
            if (phase == 0) {
                bool closed = false;
                if (h - lo >= 2) {
                    const double x2 = smcol[(h - 1) * kT], x1 = smcol[(h - 2) * kT];
                    const double yy = fabs(x2 - x1);
                    if (!(fabs(x_cur - x2) < yy)) {
                        closed = true;
                        const double mean = 0.5 * (x1 + x2);
                        msum += mean;
                        if (m >= rflm1) { has_item = true; item_eff = h - lo == 2 ? 0.5 * yy : yy; item_mean = mean; big = big || yy > 5; }
                        m++;
                        if (h - lo == 2) lo++; else h -= 2;
                    }
                }
                if (!closed) { phase = 1; k = lo; }
            } else if (phase == 1) {
                // "count the remaining ranges as one-half cycles", bottom first; the last of them is list position m-1,
                // which the slice [rainflow_length-1 : len-1] never includes
                const double xa = smcol[k * kT], xb2 = (k + 1 < h) ? smcol[(k + 1) * kT] : x_cur;
                const double mean = 0.5 * (xa + xb2);
                msum += mean;
                if (k + 1 < h) {
                    const double rg = fabs(xa - xb2);
                    if (m >= rflm1) { has_item = true; item_eff = 0.5 * rg; item_mean = mean; big = big || rg > 5; }
                    k++;
                } else phase = 2;
                m++;
            }
            RF_APPEND(fs);
        }
        RF_DRAIN(fs);
        if (live) {
            bool consumed;
            deg = sei_fade_update(p, i, len, m, rflm1 + 1, msum, acc.y + fs, big, s_temp, consumed);
            if (consumed) acc.y = 0;         // committed cycles below position m-1 can never be in a later slice
        }
    }
#undef RF_APPEND
#undef RF_DRAIN
    PT_MARK(5);
    if (live) {
        for (int s = 0; s < S; s += 2)
            *reinterpret_cast<double2*>(stk + s) = make_double2(smcol[s * kT], smcol[(s + 1) * kT]);
        p.rf_dc[i] = (unsigned int)depth | ((unsigned int)c << 16);
        p.rf_acc[i] = acc;
    }
    PT_MARK(6);
    if (slow) deg = rf_vehicle_slow(p, e, n, k_done, k_now, evaluate, s_temp);
    PT_MARK(7);
    return deg;
}

// --------------------------------------------------------------------------------------- TMA bulk store helpers
__device__ __forceinline__ void bulk_store_s2g(void* gdst, const void* ssrc, uint32_t bytes) {
    // make the generic-proxy shared-memory writes visible to the async proxy, then one bulk copy (UBLKCP)
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;"
                 :: "l"(gdst), "r"((uint32_t)__cvta_generic_to_shared(ssrc)), "r"(bytes) : "memory");
    asm volatile("cp.async.bulk.commit_group;" ::: "memory");
}
__device__ __forceinline__ void bulk_store_s2g_nofence(void* gdst, const void* ssrc, uint32_t bytes) {
    // observations are written once and never read by the kernels: evict-first keeps them from displacing the tables in L2
    uint64_t pol;
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group.L2::cache_hint [%0], [%1], %2, %3;"
                 :: "l"(gdst), "r"((uint32_t)__cvta_generic_to_shared(ssrc)), "r"(bytes), "l"(pol) : "memory");
    asm volatile("cp.async.bulk.commit_group;" ::: "memory");
}
// One thread sends nfl floats from shared to global memory where source and destination have the SAME offset inside a
// 16-byte line (the pf kernel lays its observation tile out with the phase of its destination): up to three scalar head
// floats, one bulk store for the 16-byte aligned middle, up to three scalar tail floats.  Any D and any tile size.
__device__ __forceinline__ void thread_store_range(float* gdst, const float* ssrc, int nfl) {
    int head = (int)(((16u - (unsigned)((uintptr_t)gdst & 15u)) & 15u) >> 2);
    head = head < nfl ? head : nfl;
    const int mid = (nfl - head) & ~3;
    for (int k = 0; k < head; k++) gdst[k] = ssrc[k];
    if (mid > 0) bulk_store_s2g_nofence(gdst + head, ssrc + head, (uint32_t)mid * 4u);
    for (int k = head + mid; k < nfl; k++) gdst[k] = ssrc[k];
}
__device__ __forceinline__ void bulk_store_wait_read() {
    asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
}

// ------------------------------------------------------------------------------------------ one (env, EV) slot
// The reference's inner logic for one vehicle and one step, shared by the two step kernels: EvCharger.charge
// (ev_charger.py:98-206), the action*there term of check_violation (fleet_environment.py:491), the SOC update
// (:470) and the departure / stay / gone / arrival transition with the target flip and soc_deg (:528-623).
// float64, reference operation order, no FMA contraction (the file is compiled with -fmad=false).
//   in : es (per-env factors of time t: S, F_cr, F_dr, Rfac, pv_share, flags), a = action, soh, sr / ntl = schedule
//        SOC_on_return / time_left at t+1, there = presence at t, flip = target already raised to 0.9
//   io : soc, hl, sdeg      out: the vehicle's terms of the five per-env sums
__device__ __forceinline__ void ev_slot_step(const StepParams& p, const EnvS& es, size_t i, bool flip, double a, double soh,
                                             double sr, float ntl, int there, double& soc, float& hl, double& sdeg,
                                             double& q_rew, double& q_cash, double& q_ath, double& q_miss, double& q_nviol,
                                             double& q_en) {
    const double tgt = flip ? 0.9 : p.target;                       // FleetEnv.target_soc[car]
    const double cap = soh * p.cap0;                                // episode.battery_cap[car]
    double c_cr = 0, c_dr = 0, c_inv = 0, c_oc = 0, c_dep = 0, c_cost = 0, c_rev = 0, c_miss = 0, c_nviol = 0;
    double num = 0;                                                 // next_soc = soc + num / cap
    if (a >= 0) {                                                   // ev_charger.py:98-156
        const double dem = (tgt - soc) * cap;
        const double req = p.P * a * p.dt;
        if (req * p.eta_c > dem) {
            const double d = req - dem;
            const double pen = p.pen_oc * (d * d);
            c_oc = pen > p.clip_oc ? pen : p.clip_oc;
        }
        double en = 0;
        if (there == 1) en = fmin(dem / p.eta_c, req);              // IEEE divide: SOC must be bit-exact
        else if (fabs(a) > 0.05) c_inv = p.pen_inv * (a * a);
        num = en * p.eta_c;
        q_en = en;                                                  // charge_log, ev_charger.py:212
        double ge = en - es.pv_share;
        ge = ge > 0 ? ge : 0;
        c_cost = ge * es.S * p.mult;
        c_cr = es.F_cr * ge;
    } else if (a < 0) {                                             // ev_charger.py:159-206
        const double left = -1 * soc * cap;
        const double req = p.P * a * p.dt;
        if (req * p.eta_d < left && there != 0) {
            const double d = left - req;
            c_oc = p.pen_oc * (d * d);
        }
        double en = 0.0;
        if (there == 1) en = fmax(left, req);
        else if (fabs(a) > 0.05) c_inv = p.pen_inv * (a * a);
        num = en;
        q_en = en;
        c_rev = -1 * en * es.Rfac;
        c_dr = es.F_dr * en;
    } else {
        q_en = 0;
        atomicOr(p.err_flags, 1u);                                  // NaN action: TypeError ev_charger.py:209
    }
    q_ath = a * (double)there;                                      // fleet_environment.py:491
    // ev_charger.py:128,189 ; :470.  num == 0 (absent vehicle, zero action) adds exactly 0: skipping the division there
    // is bit-identical and keeps the warp out of the slow path of the f64 divide.
    if (num != 0) soc = soc + num / cap;

    // time has advanced to t+1: departure / still there / gone / arrival   :528-618
    if (hl != 0.f && ntl == 0.f) {
        const double tg = (p.is_ct && (es.flags & EF_LUNCH)) ? p.target_lunch : tgt;
        const double diff = tg - soc;
        if (diff > p.eps) {
            c_miss = diff; c_nviol = 1;
            c_dep = -500 / (1 + exp(-16.48461585 * (diff - 0.29229767))) + 1;   // score_config.py:26-30
        } else {
            c_dep = p.full_reward;
        }
    }
    if (ntl != 0.f && hl != 0.f) hl -= p.dt_f;
    else { hl = ntl; soc = sr; }
    if (soh <= 0.9 && !flip) {                                      // :613-614 (visible from the next step on)
        p.tflip[i] = 1;
        atomicAdd(p.n_flips, 1);
    }
    if (hl != 0.f) sdeg = soc;                                      // :621-623
    q_rew = c_cr + c_dr + c_inv + c_oc + c_dep;                     // per-vehicle reward terms (:228,548-590)
    q_cash = -1 * c_cost + c_rev;                                   // ev_charger.py:225
    q_miss = c_miss; q_nviol = c_nviol;
}

// ------------------------------------------------------------------------------------------------ step kernel
// Work-list entry pushed by the step kernel for envs that need the post kernel (daily degradation and/or reset).
constexpr int WL_TRIGGER = 1, WL_RESET = 2, WL_FLUSH = 4;
// Entries with a daily evaluation are by far the longest (consumption + residue stress + fade): they are pushed from the
// front of the list and fetched first by the post kernel, everything else from the back, so that the kernel does not end
// with one late-started evaluation.  Flush-only entries (most entries; wl_flags) go to a list of their own, which the post kernel
// works through in units of 32 vehicles per warp after the other entries; they carry the env's k_done and k_now, so the
// post kernel never reads env4 of an env whose k_done another warp of the same launch may already have advanced.
__device__ __forceinline__ void wl_push(const StepParams& p, int e, int wf, int k_done, int k_now) {
    if (wf == WL_FLUSH) p.wl_flush[atomicAdd(p.wl_count + 3, 1)] = make_int4(e, k_done, k_now, 0);
    else if (wf & WL_TRIGGER) p.wl[atomicAdd(p.wl_count, 1)] = make_int2(e, wf);
    else p.wl[p.E - 1 - atomicAdd(p.wl_count + 2, 1)] = make_int2(e, wf);
}
__device__ __forceinline__ int2 wl_fetch(const StepParams& p, int w, int n_front) {
    return p.wl[w < n_front ? w : p.E - 1 - (w - n_front)];
}
// Work-list flags of an env whose step k (history sample k+1) has just been taken.  The rainflow state is read only by
// the daily evaluations, and the reset restarts it, so samples are consumed only while an evaluation remains in the
// episode (EF_EVAL_AHEAD).  Then WL_FLUSH is pushed when with the next sample the ring would hold more than R rows
// (samples k_done .. k+2), so the pending ones are consumed now.  After the last evaluation the ring wraps over unconsumed samples and k_done falls behind; the rule is monotone within
// an episode, so no consumer ever starts from such a k_done.
__device__ __forceinline__ int wl_flags(const StepParams& p, int env_flags, int k, int k_done) {
    int wf = ((env_flags & EF_TRIGGER) ? WL_TRIGGER : 0) | ((env_flags & EF_RESET) ? WL_RESET : 0);
    if (p.rf_on && (env_flags & EF_EVAL_AHEAD) && k + 1 - k_done >= p.R - 1) wf |= WL_FLUSH;
    return wf;
}

// ---- env-level parts of a step, one thread per env, shared by the two step kernels
// Fills the env scratch of env4 = {t, t_start, ep_count, k_done} from env4 and the four 128-bit words r0..r3 of
// step_row[min(t, T - 2)], and returns its EF_* flags.  Without auto-reset an env whose episode is over is frozen until
// the caller resets it; the pf kernel, which only runs with auto-reset, passes auto_reset = true so that this test
// folds away.
__device__ __forceinline__ int stage_env_scratch(const StepParams& p, EnvS& es, int4 env4, int4 r0, int4 r1, int4 r2,
                                                 int4 r3, bool auto_reset) {
    es.t = env4.x; es.t_start = env4.y; es.ep_count = env4.z; es.k_done = env4.w;
    const int t_fin = env4.y + p.L;
    const uint32_t fn = (uint32_t)r3.w;                                  // flags_next
    int fl = 0;
    if (!auto_reset && env4.x >= t_fin) {
        fl = EF_FROZEN;
    } else {
        if (env4.x + 1 == t_fin) fl |= auto_reset ? EF_DONE | EF_RESET : EF_DONE;
        if ((fn & TF_TRIGGER) && p.calc_deg) fl |= EF_TRIGGER;
        if (fn & TF_LUNCH) fl |= EF_LUNCH;
        // the next 14:45 row at or after t + 2, from the row actually read (past T - 2 there is none: saturated)
        const int dist = (int)(fn >> TF_DIST_SHIFT);
        if (p.calc_deg && dist != (int)TF_DIST_NONE && min(env4.x, p.T - 2) + dist <= t_fin) fl |= EF_EVAL_AHEAD;
    }
    es.flags = fl;
    es.S = __hiloint2double(r0.y, r0.x); es.F_cr = __hiloint2double(r0.w, r0.z);
    es.F_dr = __hiloint2double(r1.y, r1.x); es.Rfac = __hiloint2double(r1.w, r1.z);
    es.pv_share = __hiloint2double(r2.y, r2.x); es.gml = __hiloint2double(r2.w, r2.z);
    es.pvv = __hiloint2double(r3.y, r3.x);
    return fl;
}

// Where env e's observation row of this step goes, or nullptr when the caller did not ask for that array.  SB3
// semantics: a finished env returns the first observation of its next episode in obs (written by the post kernel) and
// the last observation of the finished one in infos["terminal_observation"].
__device__ __forceinline__ float* obs_row_dst(const StepParams& p, int flags, int e) {
    float* const base = (flags & EF_RESET) ? p.terminal_obs : p.obs;
    return base ? base + (size_t)e * p.D : nullptr;
}

// End of env e's step from its per-env sums sums[q * B + bb]: cashflow, reward with the overload penalty
// (score_config.py:33-41), soc violation, done, episode return (ep_prev: the return so far), the statistics in stripe
// st, the advanced env4, the work-list push and the outputs.  A frozen env reports done with zero reward and adds no
// statistics.
__device__ __forceinline__ void finalise_env(const StepParams& p, const EnvS& es, int e, const double* sums, int B,
                                             int bb, double* st, double ep_prev, uint64_t keep) {
    double reward = 0, cashflow = 0, overload = 0, soc_viol = 0;
    int done = 0;
    if (es.flags & EF_FROZEN) {
        done = 1;
    } else {
        cashflow = sums[Q_CASH * B + bb];
        reward = sums[Q_REWARD * B + bb];
        const double margin = es.gml - sums[Q_ATH * B + bb] * p.evse + es.pvv;                 // load_calculation.py:93
        overload = fabs(margin < 0.0 ? margin : 0.0);
        if (overload > 0) {
            const double rel = overload / p.grid + 1;                                          // fleet_environment.py:496
            const double pen = (rel < 1.1) ? 0.0 : -700 / (1 + exp(-15.77350877 * (rel - 1.33298382)));
            reward += pen * p.pen_ovl;                                                         // score_config.py:33-41
            atomicAdd(st + FLEET_S_OVERLOAD_KW, overload);
        }
        soc_viol = fabs(sums[Q_MISS * B + bb]);                                                // :661
        const double n_viol = sums[Q_NVIOL * B + bb];
        done = (es.flags & EF_DONE) ? 1 : 0;                                                   // :627-628
        const double ep_ret = ep_prev + reward;                                                // :637
        atomicAdd(st + FLEET_S_STEPS, 1.0);
        atomicAdd(st + FLEET_S_REWARD, reward);
        atomicAdd(st + FLEET_S_CASHFLOW, cashflow);
        if (n_viol > 0) { atomicAdd(st + FLEET_S_SOC_VIOL, soc_viol); atomicAdd(st + FLEET_S_N_VIOL, n_viol); }
        if (done) {
            atomicAdd(st + FLEET_S_EPISODES, 1.0);
            atomicAdd(st + FLEET_S_EP_RETURN, ep_ret);
            p.env_f64[(size_t)EF_LAST_EP_RETURN * p.E + e] = ep_ret;
        }
        p.env_f64[(size_t)EF_EP_RETURN * p.E + e] = ep_ret;
        st_keep_v4(p.env4 + e, make_int4(es.t + 1, es.t_start, es.ep_count, es.k_done), keep);
        const int wf = wl_flags(p, es.flags, es.t - es.t_start, es.k_done);
        if (wf) wl_push(p, e, wf, es.k_done, es.t + 1 - es.t_start);   // the post kernel evaluates the degradation first and resets afterwards, like the reference
    }
    p.env_f64[(size_t)EF_REWARD64 * p.E + e] = reward;
    p.env_f64[(size_t)EF_CASHFLOW * p.E + e] = cashflow;
    p.env_f64[(size_t)EF_OVERLOAD * p.E + e] = overload;
    p.env_f64[(size_t)EF_SOC_VIOL * p.E + e] = soc_viol;
    if (p.reward) p.reward[e] = (float)reward;
    if (p.done) p.done[e] = (uint8_t)done;
}

// Shared-memory layout (dynamic): EnvS envs[B] | double contrib[kNQ][slots] | double sums[kNQ][B] |
//                                 float obs_tile[B][D] (16-byte aligned)
__host__ __device__ constexpr size_t align16(size_t x) { return (x + 15) & ~(size_t)15; }
__host__ __device__ inline size_t smem_envs_bytes(int B) { return align16((size_t)B * sizeof(EnvS)); }
__host__ __device__ inline size_t smem_obs_offset(int B, int N) {
    return align16(smem_envs_bytes(B) + (size_t)kNQ * B * N * 8 + (size_t)kNQ * B * 8);
}
__host__ __device__ inline size_t smem_step_bytes(int B, int N, int D) {
    return align16(smem_obs_offset(B, N) + (size_t)B * D * 4);
}

template <bool kNorm, bool kAux>
__global__ void __launch_bounds__(kThreads, kMinCtasPerSm) fleet_step_kernel(const StepParams p) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int N = p.N, B = p.B, D = p.D;
    EnvS* envs = reinterpret_cast<EnvS*>(smem_raw);
    double* contrib = reinterpret_cast<double*>(smem_raw + p.off_contrib);
    const int cstride = B * N;  // contrib[q][slot]
    double* sums = contrib + kNQ * cstride;
    float* obs_tile = reinterpret_cast<float*>(smem_raw + p.off_obs);

    const int tid = threadIdx.x;
    const int e0 = blockIdx.x * B;
    const int nb = min(B, p.E - e0);
    const int nslots = nb * N;
    const int npass = (nslots + kThreads - 1) / kThreads;   // 1 unless N > kThreads
    const int H = p.Ha + p.Hb;

    const uint64_t keep = l2_evict_last_policy();
    int my_any = 0;             // bit1: this env finished and auto-resets (its row goes to terminal_obs)

    // ---- P0: one thread per env: env scratch (stage_env_scratch)
    if (tid < nb) {
        const int4 ev = ld_keep_v4(p.env4 + e0 + tid, keep);
        const int4* r = reinterpret_cast<const int4*>(p.step_row + min(ev.x, p.T - 2));
        const int4 r0 = ld_keep_v4(r, keep), r1 = ld_keep_v4(r + 1, keep), r2 = ld_keep_v4(r + 2, keep),
                   r3 = ld_keep_v4(r + 3, keep);
        if (stage_env_scratch(p, envs[tid], ev, r0, r1, r2, r3, p.auto_reset != 0) & EF_RESET) my_any = 2;
    }

    const bool have_flips = (*p.n_flips != 0);
    int any = 0;
    for (int pass = 0; pass < npass; pass++) {
        // ---- P1a: one thread per (env, EV): issue every load before the barrier.  The slot reads its env's
        // time index itself (one broadcast 128-bit load) so that the schedule record and the history row do not
        // wait for P0.
        const int j = pass * kThreads + tid;
        const bool active = j < nslots;
        int b = 0, n = 0, t = 0, k = 0;
        size_t i = 0, hrow = 0;
        float a32 = 0.f, hl = 0.f;
        double soc = 0, soh = 1, sdeg = 0;
        EvRec rec;
        rec.sr = 0; rec.tl = 0; rec.there = rec.there_prev = 0; rec.pad = 0; rec.tt = rec.cl = rec.hn = rec.lax = 0;
        if (active) {
            b = (N == 1) ? j : (int)__umulhi((unsigned)j, p.n_magic);
            n = j - b * N;
            const int e = e0 + b;
            i = (size_t)e0 * N + j;
            const int4 ev = ld_keep_v4(p.env4 + e, keep);
            t = ev.x; k = ev.x - ev.y;
            a32 = __ldcs(p.actions + i);
            soc = __ldcs(p.soc + i);
            hl = __ldcs(p.hl + i);
            soh = __ldcs(p.soh + i);
            hrow = (size_t)e * p.RN + (unsigned)((k & p.Rm) * N + n);
            sdeg = __ldcs(p.hist + hrow);
            const int tr = (!p.auto_reset && k >= p.L) ? min(t, p.T - 1) : min(t + 1, p.T - 1);   // frozen: row t
            rec = load_rec_keep(&p.ev_rec[(size_t)tr * N + n], keep);
        }
        if (pass == 0) any = __syncthreads_or(my_any) ? 2 : 0;   // returns a predicate, not the OR-ed value
        // time-only part of the observation: host-precomputed float32 row per time index, one element per thread
        float hv = 0.f; int hdst = -1;
        if (pass == 0 && tid < nb * H) {
            const int bb = (H == 1) ? tid : (int)__umulhi((unsigned)tid, p.h_magic), q = tid - bb * H;
            const EnvS& eh = envs[bb];
            const int th = (eh.flags & EF_FROZEN) ? min(eh.t, p.T - 1) : min(eh.t + 1, p.T - 1);
            hv = ld_keep_f32(p.hdr + (size_t)th * p.hdr_stride + q, keep);
            hdst = bb * D + hdr_pos<kAux>(p.Ha, N, q);
        }

        // ---- P1b: charge / discharge, transition, per-EV observation parts (into the shared obs tile)
        if (active) {
            const EnvS& es = envs[b];
            float* orow = obs_tile + b * D;
            double c_rew = 0, c_cash = 0, c_ath = 0, c_miss = 0, c_nviol = 0;
            const bool flip = have_flips && p.tflip[i] != 0;
            if (!(es.flags & EF_FROZEN)) {
                double c_en = 0;
                ev_slot_step(p, es, i, flip, (double)a32, soh, rec.sr, rec.tl, rec.there_prev, soc, hl, sdeg,
                             c_rew, c_cash, c_ath, c_miss, c_nviol, c_en);
                if (p.charge_log) p.charge_log[i] = c_en;

                __stcs(p.soc + i, soc);
                __stcs(p.hl + i, hl);
                const size_t hnext = hrow - (size_t)((k & p.Rm) * N) + (size_t)(((k + 1) & p.Rm) * N);
                __stcs(p.hist + hnext, sdeg);                                   // log_soc, :655-656
            } else if (p.charge_log) {
                p.charge_log[i] = 0;                                            // frozen env: nothing flows
            }
            write_ev_obs<kNorm, kAux>(p, orow, n, soc, hl, rec, flip);
            contrib[Q_REWARD * cstride + j] = c_rew;  contrib[Q_CASH * cstride + j] = c_cash;
            contrib[Q_ATH * cstride + j] = c_ath;     contrib[Q_MISS * cstride + j] = c_miss;
            contrib[Q_NVIOL * cstride + j] = c_nviol;
        }
        if (hdst >= 0) obs_tile[hdst] = hv;
    }
    // remaining header elements when the tile holds more than kThreads of them (small N)
    for (int w = kThreads + tid; w < nb * H; w += kThreads) {
        const int bb = w / H, q = w - bb * H;
        const EnvS& eh = envs[bb];
        const int th = (eh.flags & EF_FROZEN) ? min(eh.t, p.T - 1) : min(eh.t + 1, p.T - 1);
        obs_tile[bb * D + hdr_pos<kAux>(p.Ha, N, q)] = __ldg(p.hdr + (size_t)th * p.hdr_stride + q);
    }
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // writers: generic-proxy stores -> async proxy
    __syncthreads();

    // ---- observation tile -> HBM: one TMA bulk store per CTA when every row goes to obs[e0 .. e0+nb)
    const bool use_bulk = p.bulk_ok && nb == B && !(any & 2) && p.obs != nullptr;
    if (use_bulk) {
        if (tid == 0) bulk_store_s2g(p.obs + (size_t)e0 * D, obs_tile, (uint32_t)(B * D * 4));
    } else {
        for (int w = tid; w < nb * D; w += kThreads) {
            const int bb = w / D;
            float* dst = obs_row_dst(p, envs[bb].flags, e0 + bb);
            if (dst) dst[w - bb * D] = obs_tile[w];
        }
    }

    // ---- P2: one thread per (quantity, env): sequential sum over the env's EVs in car order (deterministic)
    for (int w = tid; w < kNQ * nb; w += kThreads) {
        const int q = w / nb, bb = w - q * nb;
        const double* c = contrib + q * cstride + bb * N;
        double s = 0;
#pragma unroll 10
        for (int nn = 0; nn < N; nn++) s += c[nn];
        sums[q * B + bb] = s;
    }
    __syncthreads();

    // ---- P3: one thread per env: finalise_env
    if (tid < nb) {
        const int e = e0 + tid;
        finalise_env(p, envs[tid], e, sums, B, tid, p.stats + (size_t)(blockIdx.x % kStatStripes) * FLEET_S__COUNT,
                     p.env_f64[(size_t)EF_EP_RETURN * p.E + e], keep);
    }
    if (use_bulk && tid == 0) bulk_store_wait_read();   // the tile must stay valid until the bulk copy has read it
}

// ------------------------------------------------------------------------------ persistent prefetching step kernel
// Same arithmetic as fleet_step_kernel, through the same functions: ev_slot_step per vehicle, stage_env_scratch,
// obs_row_dst and finalise_env per env.  What differs is how the work is fed and laid out.  The generic kernel is bound
// by exposed memory latency: ~57 % of the scheduler cycles have no eligible warp (ncu), because every warp first waits
// two dependent round trips (env4 -> schedule record / history row) and the 64-register budget caps residency at 32
// warps per SM.  Here
//  * CTAs are persistent (grid = #SMs x resident CTAs, 2 per SM) and loop over tiles of B = kPfSlots / N consecutive envs;
//  * 8 COMPUTE warps, one thread per (env, EV) slot: each thread copies its own inputs of a tile (action, state,
//    history row, schedule record, header element) into a shared-memory stage with cp.async (LDGSTS) kPfStages tiles
//    ahead; the per-env time index those addresses depend on is loaded one tile period before the copies are issued,
//    so that no dependent address ever waits; the slot -> (env, EV) mapping and parameter loads are paid once; with an
//    even N the two vehicles of a lane pair (same env) pre-add their contributions with one shuffle;
//  * 2 EPILOGUE warps, behind the compute warps: warp 0 loads env4 and step_row and stages the env scratch three tiles
//    ahead, then runs finalise_env for the current tile, one lane per env (a tile holds at most 32); warp 1 sends the
//    finished observation tile to HBM with TMA bulk stores (cp.async.bulk, SASS UBLKCP) and does the per-env sums (one
//    lane per (quantity, env), car order), which it hands to warp 0;
//  * no CTA-wide barrier in the loop: producer/consumer hand-offs are mbarriers on kPfOut contribution + observation
//    buffers, kPfEnvs env-scratch buffers and two sums buffers.
// Selected when auto_reset is on and 8 <= N <= 256 (one pass per tile); otherwise the generic kernel runs.
constexpr int kPfSlots = 256;                  // slots ((env, EV) pairs) of a tile = compute threads
constexpr int kPfThreads = kPfSlots + 64;      // + two epilogue warps
// measured on B200 at cfg2: 2 CTAs/SM x 10 warps with ~100 registers (no spills, L1 left for the tables) beat 3 CTAs/SM
// at 64 registers by 5-6 %
constexpr int kPfMaxReg = 96;

// input stage of the pf kernel: the per-slot inputs of one tile, structure of arrays indexed by the slot's thread
// (byte offsets)
constexpr int kPfStA32 = 0, kPfStHl = 4 * kPfSlots, kPfStHv = 8 * kPfSlots, kPfStSoc = 12 * kPfSlots,
              kPfStSoh = 20 * kPfSlots, kPfStSdeg = 28 * kPfSlots, kPfStR0 = 36 * kPfSlots, kPfStR1 = 52 * kPfSlots,
              kPfStageBytes = 68 * kPfSlots;
constexpr int kPfStages = 2;  // input stages: the copies of a tile are issued two tiles ahead
constexpr int kPfOut = 3;     // output buffers (contributions + obs tile): the epilogue may lag two tiles behind
constexpr int kPfEnvs = 4;    // env-scratch buffers: staged three tiles ahead
// Tile geometry and shared-memory layout of the pf kernel for N vehicles, observation width D and a history ring of R
// rows: filled into StepParams by fleet_create, and folded to literals inside a shape-specialised instance.
struct PfLayout {
    int B;                    // envs per tile
    int pair;                 // even N: neighbouring vehicles' contributions are added in the compute warp (one shuffle),
    int cslots, cper;         // halving the buffer; contribution entries per quantity and tile / per env
    unsigned int tile_hist;   // B * R * N: history elements per tile
    int envs_b, contrib_b, obs_b;                  // bytes of one env-scratch / contribution / obs buffer
    int off_contrib, off_sums, off_obs, off_stage;
    size_t smem;              // dynamic shared memory
};
__host__ __device__ constexpr PfLayout pf_layout(int N, int D, int R) {
    PfLayout l{};
    l.B = kPfSlots / N;
    l.pair = (N & 1) ? 0 : 1;
    l.cslots = l.pair ? (l.B * N) / 2 : l.B * N;
    l.cper = l.pair ? N / 2 : N;
    l.tile_hist = (unsigned int)((size_t)l.B * R * N);
    l.envs_b = (int)align16((size_t)l.B * sizeof(EnvS));
    l.contrib_b = (int)align16((size_t)kNQ * l.cslots * 8);
    l.obs_b = (int)align16((size_t)l.B * D * 4 + 12);   // + the destination's phase inside a 16-byte line
    l.off_contrib = kPfEnvs * l.envs_b;
    l.off_sums = l.off_contrib + kPfOut * l.contrib_b;
    l.off_obs = l.off_sums + 2 * (int)align16((size_t)kNQ * l.B * 8);
    l.off_stage = (int)align16((size_t)l.off_obs + (size_t)kPfOut * l.obs_b);
    l.smem = (size_t)l.off_stage + (size_t)kPfStages * kPfStageBytes;
    return l;
}

// Compile-time shape of a pf kernel instance.  All zero: any fleet, sizes read from StepParams.  Otherwise the instance
// runs only fleets of exactly N vehicles, observation width D, header Ha + Hb and a history ring of R rows, and every
// size, index and shared-memory offset derived from them is a literal (a fifth fewer instructions).
template <int kN, int kD, int kHa, int kHb, int kR>
struct PfShape {
    static constexpr int N = kN, D = kD, Ha = kHa, Hb = kHb, R = kR;
};
using PfAnyShape = PfShape<0, 0, 0, 0, 0>;
// bench.py's metric workload (cfg2): last-mile-delivery fleet of 50 EVs, full observer (price look-ahead 8, building /
// PV look-ahead 4, auxiliary terms, not normalised), rainflow-SEI with the default 16-row history ring
using PfCfg2Shape = PfShape<50, 388, 28, 10, 16>;

// The kernel's parameter block with the geometry of a specialised shape overwritten by literals (a local copy: every
// field the kernel reads is still a constant-bank operand, the overwritten ones fold into the code).
template <class Shape>
__device__ __forceinline__ StepParams pf_params(const StepParams& pk) {
    static_assert(Shape::N == 0 || (Shape::N >= 8 && Shape::N <= kPfSlots && Shape::D == 7 * Shape::N + Shape::Ha + Shape::Hb &&
                                    Shape::R >= 4 && (Shape::R & (Shape::R - 1)) == 0),
                  "a specialised shape has auxiliary terms (D = 7 N + Ha + Hb) and a power-of-two ring");
    StepParams p = pk;
    if constexpr (Shape::N != 0) {
        constexpr int N = Shape::N, H = Shape::Ha + Shape::Hb;
        constexpr PfLayout l = pf_layout(N, Shape::D, Shape::R);
        p.N = N; p.D = Shape::D; p.Ha = Shape::Ha; p.Hb = Shape::Hb; p.hdr_stride = (H + 3) / 4 * 4;
        p.R = Shape::R; p.Rm = Shape::R - 1; p.RN = (unsigned long long)Shape::R * N;
        p.n_magic = (unsigned int)((0x100000000ull + N - 1) / N);
        p.pf_B = l.B; p.pf_pair = l.pair; p.pf_cslots = l.cslots; p.pf_cper = l.cper; p.pf_tile_hist = l.tile_hist;
        p.pf_envs_b = l.envs_b; p.pf_contrib_b = l.contrib_b; p.pf_obs_b = l.obs_b;
        p.pf_off_contrib = l.off_contrib; p.pf_off_sums = l.off_sums; p.pf_off_obs = l.off_obs; p.pf_off_stage = l.off_stage;
    }
    return p;
}

__device__ __forceinline__ uint32_t smem_u32(const void* ptr) { return (uint32_t)__cvta_generic_to_shared(ptr); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" :: "r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" :: "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
    // the suspend-time hint (ns) only bounds how long the hardware may park the thread before it re-checks; the thread
    // resumes as soon as the phase completes, so a generous hint just means fewer spin iterations in the issue slots
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity), "r"(20000u) : "memory");
    return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    // try_wait suspends the thread for a hardware-defined time before returning false (a __nanosleep back-off here
    // was measured to be 2.4x slower: the hand-offs are on the critical path)
    while (!mbar_try_wait(bar, parity)) { }
}
// pf kernel hand-offs are mbarriers (not named barriers): a waiting warp then depends only on the producer of what it
// waits for, never on its sibling compute warps, so the eight compute warps drift apart by up to a tile and their
// per-tile imbalance (charging / discharging / absent vehicles) averages out instead of adding up.
#ifdef PF_TIMING
__device__ unsigned long long g_pf_clk[16 + 128];   // [16]: per role; [16 + warp * 8 + mark]: per compute warp (PF_FLUSH_W)
#define PF_MARK(k) do { const long long _c = clock64(); _acc[(k) & 7] += (unsigned long long)(_c - _pt); _pt = _c; } while (0)
#define PF_START() long long _pt = clock64()
#define PF_SETTLE() do { int _d; asm volatile("ld.volatile.shared.s32 %0, [%1];" : "=r"(_d) : "r"((uint32_t)__cvta_generic_to_shared(smem_raw)) : "memory"); if (_d == 0x7fffffff) _acc[7]++; } while (0)
#define PF_DECL() unsigned long long _acc[8] = {0, 0, 0, 0, 0, 0, 0, 0}
// timeline of CTA 0, iterations 16..23: g_pf_trace[role 0..9 (compute warps, epilogue 0, epilogue 1)][iteration][event]
__device__ unsigned long long g_pf_trace[10 * 8 * 8];
#define PF_TRACE(role_, it_, ev_) do { if (blockIdx.x == 0 && (threadIdx.x & 31) == 0 && (it_) >= 16 && (it_) < 24) g_pf_trace[((role_) * 8 + ((it_) - 16)) * 8 + (ev_)] = (unsigned long long)clock64(); } while (0)
#define PF_FLUSH(base) do { if ((threadIdx.x & 31) == 0) { for (int _k = 0; _k < 8; _k++) if (_acc[_k]) { atomicAdd(&g_pf_clk[(base) + _k], _acc[_k]); if ((base) == 8) atomicAdd(&g_pf_clk[16 + (threadIdx.x >> 5) * 8 + _k], _acc[_k]); } } } while (0)
#else
#define PF_MARK(k) do {} while (0)
#define PF_START() do {} while (0)
#define PF_SETTLE() do {} while (0)
#define PF_DECL() do {} while (0)
#define PF_TRACE(role_, it_, ev_) do {} while (0)
#define PF_FLUSH(base) do {} while (0)
#endif
// kLog: keep EvCharger's charge_log (fleet_enable_charge_log); a template flag so that the default instance carries
// neither the extra live register nor the store.  Shape: PfAnyShape or a specialised PfShape (fleet_create checks that
// the fleet matches it).
template <bool kNorm, bool kAux, bool kLog, class Shape>
__global__ void __maxnreg__(kPfMaxReg) fleet_step_pf_kernel(const StepParams pk) {
    const StepParams p = pf_params<Shape>(pk);
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int N = p.N, B = p.pf_B, D = p.D;
    const int cstride = B * N;
    const bool pair = p.pf_pair != 0;                        // contributions of vehicle pairs are pre-added (even N)
    const int cslots = p.pf_cslots;                          // contribution entries per quantity and tile
    const int cper = p.pf_cper;                              // ... per env
    unsigned char* envs0 = smem_raw;
    unsigned char* contrib0 = smem_raw + p.pf_off_contrib;
    double* sums = reinterpret_cast<double*>(smem_raw + p.pf_off_sums);
    unsigned char* obs0 = smem_raw + p.pf_off_obs;

    const int tid = threadIdx.x;
    const int ntiles = p.pf_ntiles;
    const int H = p.Ha + p.Hb;
    const uint64_t keep = l2_evict_last_policy();
    const int tile0 = blockIdx.x, G = gridDim.x;

    // done[buf]: compute -> epilogue, tile written (all compute threads arrive); freeb[buf]: epilogue -> compute,
    // contribution + obs buffers may be reused; envb[ebuf]: epilogue -> compute, env scratch of the tile is staged
    // sums_ready / sums_free[sbuf]: hand-off of the per-env sums between the two epilogue warps
    __shared__ uint64_t bar_done[kPfOut], bar_free[kPfOut], bar_env[kPfEnvs], bar_sums_ready[2], bar_sums_free[2];
    __shared__ int s_have_flips, s_any_reset[kPfEnvs];
    if (tid == 0) {
        for (int q = 0; q < kPfOut; q++) { mbar_init(&bar_done[q], kPfSlots); mbar_init(&bar_free[q], 1); }
        for (int q = 0; q < kPfEnvs; q++) mbar_init(&bar_env[q], 1);
        for (int q = 0; q < 2; q++) { mbar_init(&bar_sums_ready[q], 1); mbar_init(&bar_sums_free[q], 1); }
        s_have_flips = (*p.n_flips != 0);
    }
    __syncthreads();

    const int sums_stride = (int)align16((size_t)kNQ * B * 8) / 8;   // doubles per sums buffer
    if (tid >= kPfSlots + 32) {
        // =================================================================== epilogue warp 1: tile -> HBM, per-env sums
        // The latency chain between a finished tile and the release of its buffers: bulk store of the observation tile,
        // the per-env sums (handed to warp 0 through sums[sbuf]), read-completion of the bulk store.
        const int lane = tid - kPfSlots - 32;
        int it = 0;
        PF_DECL();
        PF_START();
        for (int tile = tile0; tile < ntiles; tile += G, it++) {
            const int buf = it % kPfOut, sbuf = it & 1;
            const EnvS* envs = reinterpret_cast<const EnvS*>(envs0 + (it % kPfEnvs) * p.pf_envs_b);
            const double* contrib = reinterpret_cast<const double*>(contrib0 + buf * p.pf_contrib_b);
            // the tile sits in shared memory at the 16-byte phase of its destination obs + e0 * D (0 when B * D % 4 == 0)
            const float* obs_tile = reinterpret_cast<const float*>(obs0 + buf * p.pf_obs_b) + (int)(((size_t)tile * (size_t)(B * D)) & 3);
            double* sums_w = sums + sbuf * sums_stride;
            const int e0 = tile * B;
            const int nb = min(B, p.E - e0);
            PF_MARK(0);
            mbar_wait(&bar_done[buf], (uint32_t)((it / kPfOut) & 1));   // the compute warps have written tile `tile`
            PF_SETTLE();
            PF_MARK(1);
            PF_TRACE(9, it, 0);

            // ---- observation tile -> HBM
            const bool use_bulk = p.pf_bulk && nb == B && !s_any_reset[it % kPfEnvs] && p.obs != nullptr;
            if (use_bulk) {
                // the writers have run fence.proxy.async before arriving on bar_done: no second fence here
                if (lane == 0) thread_store_range(p.obs + (size_t)e0 * D, obs_tile, B * D);
            } else if (p.pf_bulk) {
                // rows of finishing envs go to terminal_obs: one bulk store per env row (row e has the same 16-byte phase
                // in obs, in terminal_obs and in the tile)
                if (lane < nb) {
                    float* dst = obs_row_dst(p, envs[lane].flags, e0 + lane);
                    if (dst) thread_store_range(dst, obs_tile + (size_t)lane * D, D);
                }
            } else {
                for (int w = lane; w < nb * D; w += 32) {
                    const int bb = w / D;
                    float* dst = obs_row_dst(p, envs[bb].flags, e0 + bb);
                    if (dst) dst[w - bb * D] = obs_tile[w];
                }
            }
            PF_MARK(6);
            // ---- per-env sums: one lane per (quantity, env); five interleaved partial sums in car order, combined in
            // a fixed order (deterministic run to run; the dependent-add chain is 5x shorter than a sequential sum)
            PF_TRACE(9, it, 1);
            if (it >= 2) mbar_wait(&bar_sums_free[sbuf], (uint32_t)(((it >> 1) - 1) & 1));
            PF_TRACE(9, it, 2);
            for (int w = lane; w < kNQ * nb; w += 32) {
                const int q = w / nb, bb = w - q * nb;
                const double* c = contrib + q * cslots + bb * cper;
                double s0 = 0, s1 = 0, s2 = 0, s3 = 0, s4 = 0;
                int nn = 0;
                for (; nn + 5 <= cper; nn += 5) { s0 += c[nn]; s1 += c[nn + 1]; s2 += c[nn + 2]; s3 += c[nn + 3]; s4 += c[nn + 4]; }
                for (; nn < cper; nn++) s0 += c[nn];
                sums_w[q * B + bb] = ((s0 + s1) + (s2 + s3)) + s4;
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(&bar_sums_ready[sbuf]);
            PF_MARK(2);
            PF_TRACE(9, it, 3);
            if (p.pf_bulk && (use_bulk ? lane == 0 : lane < nb)) bulk_store_wait_read();
            __syncwarp();
            PF_MARK(3);
            if (lane == 0) mbar_arrive(&bar_free[buf]);       // contribution + obs buffers of this tile are free again
            PF_MARK(4);
            PF_TRACE(9, it, 4);
        }
        PF_FLUSH(0);
        bulk_store_wait_read();
        return;
    }
    if (tid >= kPfSlots) {
        // =================================================================== epilogue warp 0: env scratch, finalisation
        const int lane = tid - kPfSlots;
        int4 envA = make_int4(0, 0, 0, 0), envQ = make_int4(0, 0, 0, 0), r0, r1, r2, r3;
        r0 = r1 = r2 = r3 = make_int4(0, 0, 0, 0);
        // two-deep load pipeline, no dependent load is ever waited for in the loop: env4 of a tile is fetched one
        // iteration before its step_row (whose address needs env4.t)
        auto load_env4 = [&](int tile) {                      // lane < B: env4 of env tile*B + lane -> envQ
            const int e = tile * B + lane;
            if (lane < B && tile < ntiles && e < p.E) envQ = ld_keep_v4(p.env4 + e, keep);
        };
        auto load_rows = [&](int tile) {                      // step_row[t] of the env in envA -> r0..r3
            const int e = tile * B + lane;
            if (lane < B && tile < ntiles && e < p.E) {
                const int4* r = reinterpret_cast<const int4*>(p.step_row + min(envA.x, p.T - 2));
                r0 = ld_keep_v4(r, keep); r1 = ld_keep_v4(r + 1, keep); r2 = ld_keep_v4(r + 2, keep); r3 = ld_keep_v4(r + 3, keep);
            }
        };
        auto stage_env = [&](int tile, int ebuf) -> bool {    // returns: some env of the tile finishes (and resets)
            const int e = tile * B + lane;
            int fl = 0;
            if (lane < B && tile < ntiles && e < p.E) {
                EnvS& es = reinterpret_cast<EnvS*>(envs0 + ebuf * p.pf_envs_b)[lane];
                fl = stage_env_scratch(p, es, envA, r0, r1, r2, r3, true);
            }
            const bool any = __any_sync(0xffffffffu, (fl & EF_RESET) != 0);
            if (lane == 0) s_any_reset[ebuf] = any;
            return any;
        };
        // env scratch of the first three tiles; the loads of the next two go in flight
        load_env4(tile0); envA = envQ; load_rows(tile0); stage_env(tile0, 0);
        __syncwarp(); if (lane == 0) mbar_arrive(&bar_env[0]);
        load_env4(tile0 + G); envA = envQ; load_rows(tile0 + G); stage_env(tile0 + G, 1);
        __syncwarp(); if (lane == 0) mbar_arrive(&bar_env[1]);
        load_env4(tile0 + 2 * G); envA = envQ; load_rows(tile0 + 2 * G); stage_env(tile0 + 2 * G, 2);
        __syncwarp(); if (lane == 0) mbar_arrive(&bar_env[2]);
        load_env4(tile0 + 3 * G); envA = envQ; load_rows(tile0 + 3 * G);
        load_env4(tile0 + 4 * G);

        int it = 0;
        for (int tile = tile0; tile < ntiles; tile += G, it++) {
            const int sbuf = it & 1;
            const EnvS* envs = reinterpret_cast<const EnvS*>(envs0 + (it % kPfEnvs) * p.pf_envs_b);
            const double* sums_r = sums + sbuf * sums_stride;
            const int e0 = tile * B;
            const int nb = min(B, p.E - e0);

            // env scratch three tiles ahead goes first: its buffer has been free since the previous iteration (tile-1
            // is complete on the compute side, waited for through warp 1's sums, and finalised here)
            stage_env(tile + 3 * G, (it + 3) % kPfEnvs);
            __syncwarp();
            if (lane == 0) mbar_arrive(&bar_env[(it + 3) % kPfEnvs]);
            PF_TRACE(8, it, 0);
            envA = envQ; load_rows(tile + 4 * G);             // in flight during this iteration
            load_env4(tile + 5 * G);
            double ep_prev = 0;                               // episode return so far (lane < nb), fetched ahead of its use
            if (lane < nb) ep_prev = p.env_f64[(size_t)EF_EP_RETURN * p.E + e0 + lane];
            mbar_wait(&bar_sums_ready[sbuf], (uint32_t)((it >> 1) & 1));   // warp 1 has summed tile `tile`
            PF_TRACE(8, it, 1);

            // ---- env-level finalisation: one lane per env (a tile holds at most 32 envs)
            if (lane < nb)
                finalise_env(p, envs[lane], e0 + lane, sums_r, B, lane,
                             p.stats + (size_t)(tile % kStatStripes) * FLEET_S__COUNT, ep_prev, keep);
            __syncwarp();
            if (lane == 0) mbar_arrive(&bar_sums_free[sbuf]);
            PF_TRACE(8, it, 2);
        }
        return;
    }

    // ======================================================================= compute warps
    // thread tid owns slot j = tid of every tile
    const int j = tid;
    const int b = (N == 1) ? j : (int)__umulhi((unsigned)j, p.n_magic);     // slot -> (env of tile, EV): same for every tile
    const int n = j - b * N;
    const bool slot = j < cstride;
    const int hpos = hdr_pos<kAux>(p.Ha, N, n);

    // Input pipeline: the per-slot inputs of a tile (action, soc, hours_left, soh, previous history row, both halves of
    // ev_rec[t+1], the header element) are copied by the slot's OWN thread into a shared-memory stage with cp.async
    // (LDGSTS) two tiles ahead.  The bytes in flight live in shared memory instead of registers: ~32 KB per CTA, which
    // is what the HBM latency x bandwidth product asks for (a register pipeline one tile deep was latency bound), and
    // since every thread reads back only what it copied itself no barrier is involved, just cp.async.wait_group.
    const uint32_t stage0 = smem_u32(smem_raw + p.pf_off_stage);
    const uint64_t stream = l2_evict_first_policy();          // (keep: created at the top of the kernel)
    const size_t hist_slot = (size_t)b * p.RN + n;            // this slot's offset inside its tile's history block
    auto load_env2 = [&](int tile) -> int2 {
        const int e = tile * B + b;
        int2 v = make_int2(0, 0);
        if (slot && tile < ntiles && e < p.E) {   // predicated load straight into the pipeline register (a select here
            asm volatile("ld.global.nc.v2.s32 {%0,%1}, [%2];" : "+r"(v.x), "+r"(v.y) : "l"(p.env4 + e));   // would wait on it)
        }
        return v;
    };
    auto issue_copies = [&](int tile, const int2 ev, int stage) {
        const int e = tile * B + b;
        if (slot && tile < ntiles && e < p.E) {
            const size_t i = (size_t)tile * cstride + j;
            const uint32_t st = stage0 + (uint32_t)stage * kPfStageBytes;
            const int k = ev.x - ev.y;
            const int t1 = min(ev.x + 1, p.T - 1);
            const int4* rp = reinterpret_cast<const int4*>(p.ev_rec + (size_t)t1 * N + n);
            const double* hp = p.hist + ((size_t)(unsigned)tile * p.pf_tile_hist + hist_slot + (unsigned)((k & p.Rm) * N));
            const float* hd = p.hdr + (size_t)t1 * p.hdr_stride + n;
            cp_async4_hint(st + kPfStA32 + j * 4, p.actions + i, stream);
            cp_async8_hint(st + kPfStSoc + j * 8, p.soc + i, stream);
            cp_async4_hint(st + kPfStHl + j * 4, p.hl + i, stream);
            cp_async8_hint(st + kPfStSoh + j * 8, p.soh + i, stream);
            cp_async8_hint(st + kPfStSdeg + j * 8, hp, stream);
            cp_async16_hint(st + kPfStR0 + j * 16, rp, keep);
            cp_async16_hint(st + kPfStR1 + j * 16, rp + 1, keep);
            if (n < H) cp_async4_hint(st + kPfStHv + j * 4, hd, keep);
        }
        cp_async_commit();
    };
#pragma unroll
    for (int q = 0; q < kPfStages; q++) issue_copies(tile0 + q * G, load_env2(tile0 + q * G), q);

    // rotating buffer indices and mbarrier phase bits (no division in the loop)
    int it = 0, buf = 0, stg = 0, ebuf = 0;
    uint32_t ph_env = 0, ph_free = 0;                          // parity to wait for on bar_env[ebuf] / bar_free[buf]
    PF_DECL();
    PF_START();
    for (int tile = tile0; tile < ntiles; tile += G, it++) {
        const EnvS* envs = reinterpret_cast<const EnvS*>(envs0 + ebuf * p.pf_envs_b);
        double* contrib = reinterpret_cast<double*>(contrib0 + buf * p.pf_contrib_b);
        float* obs_tile = reinterpret_cast<float*>(obs0 + buf * p.pf_obs_b) + (int)(((size_t)tile * (size_t)(B * D)) & 3);
        const int e0 = tile * B;
        const int nb = min(B, p.E - e0);
        const bool active = slot && b < nb;

        // ---- this tile's inputs: wait for the thread's own copies; they are read from the stage where they are needed
        // and the stage is refilled (for the tile after next) at the end of the tile, one tile period ahead of its use
        const int2 ev_next = load_env2(tile + kPfStages * G);
        cp_async_wait_group<kPfStages - 1>();
        const unsigned char* stp = smem_raw + p.pf_off_stage + stg * kPfStageBytes;
        PF_MARK(4);
        PF_TRACE(tid >> 5, it, 0);
        mbar_wait(&bar_env[ebuf], ph_env);                    // env scratch of this tile is staged
        PF_SETTLE();
        PF_MARK(0);
        PF_TRACE(tid >> 5, it, 1);
        if (it >= kPfOut) mbar_wait(&bar_free[buf], ph_free);  // contribution + obs buffers are free again
        PF_SETTLE();
        PF_MARK(2);
        PF_TRACE(tid >> 5, it, 2);
#ifdef PF_TIMING_LDS      /* one more shared-memory load round trip, timed on its own */
        PF_SETTLE();
        PF_MARK(7);
#endif

        double q_rew = 0, q_cash = 0, q_ath = 0, q_miss = 0, q_nviol = 0;   // this vehicle's terms of the per-env sums
        double o_soc = 0, o_sdeg = 0, o_en = 0;                             // new state, stored after the hand-off
        float o_hl = 0.f;
        size_t o_hist = 0;
        if (active) {
            const EnvS& es = envs[b];
            float* orow = obs_tile + b * D;
            const size_t i = (size_t)tile * cstride + j;
            const int t1 = min(es.t + 1, p.T - 1);
            const int k = es.t - es.t_start;
            // every input first (the stage and the observation tile may alias as far as the compiler knows: loads placed after
            // the observation stores would have to wait for them)
            const EvRec rec = decode_rec(reinterpret_cast<const int4*>(stp + kPfStR0)[j],
                                         reinterpret_cast<const int4*>(stp + kPfStR1)[j]);
            o_soc = reinterpret_cast<const double*>(stp + kPfStSoc)[j];
            o_sdeg = reinterpret_cast<const double*>(stp + kPfStSdeg)[j];
            const double soh = reinterpret_cast<const double*>(stp + kPfStSoh)[j];
            o_hl = reinterpret_cast<const float*>(stp + kPfStHl)[j];
            const double a = (double)reinterpret_cast<const float*>(stp + kPfStA32)[j];
            float hv0 = 0.f;
            if (n < H) hv0 = reinterpret_cast<const float*>(stp + kPfStHv)[j];
            const bool flip = s_have_flips && p.tflip[i] != 0;
            ev_slot_step(p, es, i, flip, a, soh, rec.sr, rec.tl, rec.there_prev, o_soc, o_hl, o_sdeg, q_rew, q_cash, q_ath,
                         q_miss, q_nviol, o_en);
            o_hist = (size_t)(unsigned)tile * p.pf_tile_hist + hist_slot + (unsigned)(((k + 1) & p.Rm) * N);
            write_ev_obs<kNorm, kAux>(p, orow, n, o_soc, o_hl, rec, flip);
            // time-only part of the observation: element n of this env's header row (+ the rest when N < H)
            if (n < H) orow[hpos] = hv0;
            for (int q = n + N; q < H; q += N)
                orow[hdr_pos<kAux>(p.Ha, N, q)] = ld_keep_f32(p.hdr + (size_t)t1 * p.hdr_stride + q, keep);
        }
        // even N: the two vehicles of a lane pair (same env) are added here, even lane + odd lane
        if (pair) {
            q_rew += __shfl_xor_sync(0xffffffffu, q_rew, 1);
            q_cash += __shfl_xor_sync(0xffffffffu, q_cash, 1);
            q_ath += __shfl_xor_sync(0xffffffffu, q_ath, 1);
            q_miss += __shfl_xor_sync(0xffffffffu, q_miss, 1);
            q_nviol += __shfl_xor_sync(0xffffffffu, q_nviol, 1);
        }
        if (active && !(pair && (j & 1))) {
            const int cj = pair ? (j >> 1) : j;
            contrib[Q_REWARD * cslots + cj] = q_rew;
            contrib[Q_CASH * cslots + cj] = q_cash;
            contrib[Q_ATH * cslots + cj] = q_ath;
            contrib[Q_MISS * cslots + cj] = q_miss;
            contrib[Q_NVIOL * cslots + cj] = q_nviol;
        }
        PF_MARK(1);
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // generic-proxy stores -> async proxy (bulk store)
        mbar_arrive(&bar_done[buf]);
        PF_MARK(5);
        PF_TRACE(tid >> 5, it, 3);
        // the new state goes to HBM after the hand-off: the fence above (MEMBAR + proxy fence) then only has shared-memory
        // stores to wait for, not these
        if (active) {
            const size_t i = (size_t)tile * cstride + j;
            __stcs(p.soc + i, o_soc);
            __stcs(p.hl + i, o_hl);
            __stcs(p.hist + o_hist, o_sdeg);
            if (kLog) __stcs(p.charge_log + i, o_en);
        }
        PF_MARK(6);
        issue_copies(tile + kPfStages * G, ev_next, stg);     // refill the stage this tile has just consumed
        PF_MARK(3);
        PF_TRACE(tid >> 5, it, 4);
        if (++stg == kPfStages) stg = 0;
        if (++ebuf == kPfEnvs) { ebuf = 0; ph_env ^= 1u; }
        if (++buf == kPfOut) { buf = 0; if (it >= kPfOut) ph_free ^= 1u; }
    }
    PF_FLUSH(8);
}

// ------------------------------------------------------------------------------------------------ post kernel
// One CTA of kPostThreads threads per work-list entry (persistent grid, entries fetched dynamically), one vehicle per
// thread.  An entry is an env that, in this step,
//   WL_TRIGGER  reached the daily evaluation (fleet_environment.py:665-673): consume the pending history samples, then
//               RainflowSeiDegradation / EmpiricalDegradation.calculate_degradation, soh -= degradation;
//   WL_FLUSH    is about to wrap its history ring: consume the pending samples (no evaluation);
//   WL_RESET    finished its episode with auto-reset on: FleetEnv.reset (:330-434) AFTER the evaluation, i.e. the order in
//               which a SubprocVecEnv worker runs them.
// Entries that are WL_FLUSH and nothing else are not work items: once the items are exhausted, every warp consumes them
// in flush units of 32 vehicles (see the end of fleet_post_kernel).
// The last CTA of a post kernel to finish clears the work lists for the next step.
__device__ __forceinline__ void post_finish_lists(const StepParams& p) {
    if (threadIdx.x == 0) {
        __threadfence();
        const unsigned int d = atomicAdd(p.wl_done, 1u);
        if (d == gridDim.x - 1) {
            p.wl_count[0] = 0; p.wl_count[1] = 0; p.wl_count[2] = 0; p.wl_count[3] = 0; p.wl_count[4] = 0;
            *p.wl_done = 0;
        }
    }
}

// kT = threads per CTA = lanes per work item: 32 (one warp per item, fleets of up to 32 vehicles) or 64 (two warps)
template <bool kNorm, bool kAux, int kT>
__global__ void __launch_bounds__(kT, kT == 32 ? 2 * kPostMinCtas : kPostMinCtas) fleet_post_kernel(const __grid_constant__ StepParams p) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    double* sm_stack = reinterpret_cast<double*>(smem_raw);                    // [rf_S][kT]
    double* sm_queue = sm_stack + (size_t)p.rf_S * kT;               // [kRfQueue][kT]
    double2* sm_pend = reinterpret_cast<double2*>(sm_queue + (size_t)kRfQueue * kT);   // [kRfPend][kT]
    __shared__ int s_w;
    __shared__ int2 s_ent;
    __shared__ int4 s_ev;
    __shared__ double s_deg;
    const int tid = threadIdx.x, N = p.N;
    const int n_front = p.wl_count[0];
    const int count = n_front + p.wl_count[2];
    const double temp_ref = 25, k_temp = 6.93E-2;
    const double s_temp = exp(k_temp * (p.temperature - temp_ref) * ((temp_ref + 273.15) / (p.temperature + 273.15)));  // :72-73

    // A work item is one CHUNK of an entry's vehicles (post_cv = ceil(N / post_chunks) <= kT of them): the chunks of an env
    // are independent (each vehicle has its own rainflow state) and may run in different CTAs at different times.  They
    // all read the env's env4 record when they start; whichever finishes LAST (per-entry counter) writes it back.
    // The first item of a CTA is static (item blockIdx.x), further ones come from a counter; thread 0 fetches the NEXT
    // item's list record and env4 while the current one is processed, so the two dependent round trips are hidden.
    const int chunks = p.post_chunks, cv = p.post_cv;
    const int items = count * chunks;
    if (tid == 0) {
        s_w = blockIdx.x; s_deg = 0;
        if (s_w < items) { s_ent = wl_fetch(p, s_w / chunks, n_front); s_ev = p.env4[s_ent.x]; }
    }
    for (;;) {
        __syncthreads();
        const int item = s_w;
        if (item >= items) break;
        const int w = item / chunks, chunk = item - w * chunks;
        const int2 ent = s_ent;
        const int e = ent.x, wf = ent.y;
        const int4 ev = s_ev;                           // {t (already advanced), t_start, ep_count, k_done}
        const int k_now = ev.x - ev.y;                  // newest history sample (samples 0..k_now exist)
        const int n = chunk * cv + tid;                 // this thread's vehicle
        const bool mine = tid < cv && n < N;
        int w_next = 0;
        int2 ent_next = make_int2(0, 0);
        int4 ev_next = make_int4(0, 0, 0, 0);
        if (tid == 0) {
            w_next = atomicAdd(p.wl_count + 1, 1) + (int)gridDim.x;
            if (w_next < items) { ent_next = wl_fetch(p, w_next / chunks, n_front); ev_next = p.env4[ent_next.x]; }
        }
        PT_START((wf & WL_TRIGGER) != 0);
        PT_COUNT(11, 1);
        if (p.rf_on && (wf & (WL_TRIGGER | WL_FLUSH))) {
            PT_COUNT(12, 1);
            const double deg = rf_vehicle<kT, true>(p, e, n, mine, ev.w, k_now, (wf & WL_TRIGGER) != 0, s_temp, sm_stack + tid,
                                              sm_queue + tid, sm_pend + tid);             // (all lanes of a warp go in together)
            if (deg != 0) atomicAdd(&s_deg, deg);
        } else if ((wf & WL_TRIGGER) && mine) {         // EmpiricalDegradation: the last two samples only
            const double* hbase = p.hist + (size_t)e * p.RN;
            const size_t ii = (size_t)e * N + n;
            double deg = 0;
            if (k_now >= 1) deg = empirical_eval(p.dt, p.evse, hbase[(size_t)((k_now - 1) & p.Rm) * N + n], hbase[(size_t)(k_now & p.Rm) * N + n]);
            p.n_cycles[ii] = 0;
            p.last_deg[ii] = deg;
            p.soh[ii] = p.soh[ii] - deg;
            if (deg != 0) atomicAdd(&s_deg, deg);
        }
        __syncthreads();
        PT_MARK(8);
        if (tid == 0 && s_deg != 0)
            atomicAdd(p.stats + (size_t)(w % kStatStripes) * FLEET_S__COUNT + FLEET_S_DEGRADATION, s_deg);
        // FleetEnv.reset of this chunk's vehicles, as the SubprocVecEnv worker calls it right after a done step
        int t0 = 0;
        if (wf & WL_RESET) {
            PT_COUNT(13, 1);
            t0 = episode_start(p, p.next_start, e, ev.z);
            if (mine) reset_slot<kNorm, kAux>(p, e, n, t0, p.obs ? p.obs + (size_t)e * p.D : nullptr, !p.carry);
            PT_MARK(14);
        }
        if (tid == 0) {
            bool last = true;
            if (chunks > 1) {
                __threadfence();
                last = atomicAdd(p.wl_chunks + w, 1) == chunks - 1;
                if (last) p.wl_chunks[w] = 0;
            }
            if (last) {
                if (wf & WL_RESET) {
                    begin_episode(p, e, t0, ev.z);
                } else if (p.rf_on) {
                    p.env4[e] = make_int4(ev.x, ev.y, ev.z, k_now);    // samples up to k_now are consumed
                }
            }
        }
        __syncthreads();                                 // everybody has read s_w / s_ent / s_ev / s_deg
        PT_MARK(9);
        if (tid == 0) { s_w = w_next; s_ent = ent_next; s_ev = ev_next; s_deg = 0; }
    }

    // Flush units: the flush-only entries as one flattened index space of (entry, vehicle) pairs, cut into units of 32
    // consecutive vehicles.  Each warp fetches units on its own (no CTA barrier), lane l takes vehicle 32 u + l, so a unit
    // may span two or more envs; a flush needs no evaluation, no reset and no shared sum.  Whoever holds vehicle N-1 of an
    // env stores its new k_done.
    const int n_flush = p.wl_count[3];
    if (n_flush > 0) {
        const unsigned full = 0xffffffffu;
        const int lane = tid & 31;
        const int vehicles = n_flush * N;                // < 2^31: E * N is checked at create time
        const int units = (vehicles + 31) >> 5;
        for (;;) {
            int u = 0;
            if (lane == 0) u = atomicAdd(p.wl_count + 4, 1);
            u = __shfl_sync(full, u, 0);
            if (u >= units) break;
#ifdef POST_TIMING
            const long long pt_u = clock64();
#endif
            const int v = (u << 5) + lane;
            const bool active = v < vehicles;
            int4 fe = make_int4(0, 0, 0, 0);             // an inactive lane reads env 0, row 0, and consumes nothing
            int n = 0;
            if (active) {
                const int f = v / N;
                n = v - f * N;
                fe = p.wl_flush[f];
            }
            if (active && n == N - 1) p.env4[fe.x].w = fe.z;     // samples up to k_now are consumed (read by the next step)
            rf_vehicle<kT, false>(p, fe.x, n, active, fe.y, fe.z, false, s_temp, sm_stack + tid, sm_queue + tid, sm_pend + tid);
#ifdef POST_TIMING
            if (lane == 0) { atomicAdd(&g_post_clk[15], 1ull); atomicAdd(&g_post_clk[0], (unsigned long long)(clock64() - pt_u)); }
#endif
        }
    }
    __syncthreads();                                     // no warp of this CTA fetches a unit once the lists are cleared
    post_finish_lists(p);
}

template <bool kNorm, bool kAux>
__global__ void __launch_bounds__(kThreads) fleet_reset_kernel(const StepParams p) {
    const int N = p.N, B = p.B;
    const int e0 = blockIdx.x * B;
    const int nb = min(B, p.E - e0);
    const int nslots = nb * N;
    for (int j = threadIdx.x; j < nslots; j += kThreads) {
        const int b = j / N, n = j - b * N;
        const int e = e0 + b;
        if (p.mask && !p.mask[e]) continue;
        const int t0 = episode_start(p, p.start_idx, e, p.env4[e].z);
        reset_slot<kNorm, kAux>(p, e, n, t0, p.obs ? p.obs + (size_t)e * p.D : nullptr, !p.carry);
    }
    __syncthreads();  // all slots have read env4 before it is rewritten
    if (threadIdx.x < nb) {
        const int e = e0 + threadIdx.x;
        if (!(p.mask && !p.mask[e])) {
            const int ep_count = p.env4[e].z;
            begin_episode(p, e, episode_start(p, p.start_idx, e, ep_count), ep_count);
        }
    }
}

// ------------------------------------------------------------------------------------------ small utility kernels
__global__ void init_state_kernel(StepParams p) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const size_t EN = (size_t)p.E * p.N;
    if (i < EN) {
        p.soc[i] = 0; p.hl[i] = 0; p.soh[i] = p.init_soh;
        p.rf_len[i] = 1; p.fd_cyc[i] = 0; p.life[i] = 1 - p.init_soh; p.n_cycles[i] = 0; p.last_deg[i] = 0;
        p.tflip[i] = 0;
        if (p.rf_on) { p.rf_dc[i] = 1u; p.rf_acc[i] = make_double2(0.0, 0.0); p.rf_ext[i] = -1; }
    }
    if (i < (size_t)p.E) p.env4[i] = make_int4(0, 0, 0, 0);
}

// field gathers that are not plain arrays
// Rule-based charging policies of the reference's benchmarking scripts, one thread per (env, EV); the actions are what
// those scripts hand to VecEnv.step, as float32 (the action space's dtype):
//   uncontrolled  benchmarking/uncontrolled_charging.py:51-54   a = 1
//   distributed   benchmarking/distributed_charging.py:50-54    a = clip(hours_needed / (hours_left + 0.001), 0, 1) from the
//                 SCHEDULE observation at the current time (FleetEnv.get_dist_factor, fleet_environment.py:782-799)
//   night         benchmarking/night_charging.py:81-98          a = 1 inside a charging window that opens at
//                 (charging_hour, charging_minute) and stays open for more than int(max_time_needed) hours, 0 outside; the
//                 caretaker use case follows the distributed rule between 11:00 and 14:59.  The window flag and its
//                 opening time are per-env state (st_in -> st_out), carried across episodes like the script's locals.
__global__ void policy_kernel(StepParams p, int policy, int ch_hour, int ch_minute, int max_h, const uint16_t* __restrict__ tod,
                              const int2* __restrict__ st_in, int2* __restrict__ st_out, float* __restrict__ actions) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (size_t)p.E * p.N) return;
    const int e = (int)(i / p.N), n = (int)(i - (size_t)e * p.N);
    const int t = min(p.env4[e].x, p.T - 1);
    float a = 1.f;
    if (policy != FLEET_POLICY_UNCONTROLLED) {
        const EvRec rec = load_rec(&p.ev_rec[(size_t)t * p.N + n]);
        const bool flip = (*p.n_flips != 0) && p.tflip[i] != 0;
        const double tgt = flip ? 0.9 : p.target;
        const double cl = tgt * (double)rec.there - rec.sr;                       // observer_bl_pv.py:86-88
        const double hn = cl * p.lc_batt_cap / p.hn_den;                          // :89
        double d = hn / ((double)rec.tl + 0.001);                                 // fleet_environment.py:799
        d = d < 0 ? 0 : (d > 1 ? 1 : d);
        if (policy == FLEET_POLICY_DISTRIBUTED) {
            a = (float)d;
        } else {
            const int hour = tod[t] / 60, minute = tod[t] % 60;
            int2 st = st_in[e];                                                   // {charging, index of the window start}
            if (p.is_ct && hour >= 11 && hour <= 14) {
                a = (float)d;                                                     // night_charging.py:84-87 (state untouched)
            } else {
                if ((ch_hour <= hour && ch_minute <= minute) || st.x) {           // :89
                    if (!st.x) st.y = t;
                    st.x = 1;
                    a = 1.f;
                } else {
                    a = 0.f;
                }
                if (st.x && (double)(t - st.y) * p.dt > (double)max_h) st.x = 0;  // :97-98
            }
            if (n == 0) st_out[e] = st;
        }
    }
    actions[i] = a;
}

__global__ void gather_field_kernel(StepParams p, int field, void* dst) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const size_t EN = (size_t)p.E * p.N;
    switch (field) {
        case FLEET_F_SOC_DEG:
            if (i < EN) {
                const int e = (int)(i / p.N), n = (int)(i - (size_t)e * p.N);
                const int4 ev = p.env4[e];
                const int k = ev.x - ev.y;
                ((double*)dst)[i] = p.hist[((size_t)e * p.R + (k & p.Rm)) * p.N + n];
            }
            break;
        case FLEET_F_TARGET_SOC:
            if (i < EN) ((double*)dst)[i] = (*p.n_flips != 0 && p.tflip[i]) ? 0.9 : p.target;
            break;
        case FLEET_F_TIME_IDX: if (i < (size_t)p.E) ((int*)dst)[i] = p.env4[i].x; break;
        case FLEET_F_FINISH_IDX: if (i < (size_t)p.E) ((int*)dst)[i] = p.env4[i].y + p.L; break;
        case FLEET_F_EP_COUNT: if (i < (size_t)p.E) ((int*)dst)[i] = p.env4[i].z; break;
        default: break;
    }
}

__global__ void scatter_target_kernel(StepParams p, const double* src) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < (size_t)p.E * p.N) {
        const uint8_t f = (src[i] == 0.9 && p.target != 0.9) ? 1 : 0;
        p.tflip[i] = f;
        if (f) atomicAdd(p.n_flips, 1);
    }
}

__global__ void reduce_stats_kernel(const double* stats, double* dst, double price_mult) {
    __shared__ double tot[FLEET_S__COUNT];
    const int q = threadIdx.x;
    if (q < FLEET_S__COUNT) {
        double s = 0;
        for (int k = 0; k < kStatStripes; k++) s += stats[(size_t)k * FLEET_S__COUNT + q];
        tot[q] = s;
    }
    __syncthreads();
    if (q < FLEET_S__COUNT)   // penalty = reward - cashflow*price_multiplier is linear, so its sum is derived (:659)
        dst[q] = (q == FLEET_S_PENALTY) ? tot[FLEET_S_REWARD] - tot[FLEET_S_CASHFLOW] * price_mult : tot[q];
}

// ------------------------------------------------------------------------------------------------ device-side log
// DataLogger.log_data (utils/data_logger/data_logger.py:21-68) for a handful of selected envs: one row per reset
// (fleet_environment.py:420-432) and per step that does not end the episode (:679-690), kept in a ring in HBM.  Row layout
// (float64): {ep_count, time index, reward, cashflow, penalties, grid overloading, SOC violation, kind (1 reset row,
// 2 step row at a daily evaluation, 0 other step row)}, Action[N], Degradation[N], Charging energy[N], SOH[N], Observation[D].
constexpr int kLogHead = 8;
struct LogParams {
    const int* ids;            // [n] logged envs
    long long* counts;         // [n] rows written so far (ring position = count % rows)
    double* rows;              // [n][rows][row_doubles]
    int n, cap, row_doubles;
};

__global__ void fleet_log_kernel(const StepParams p, const LogParams lg, int after_reset) {
    const int l = blockIdx.x;
    const int e = lg.ids[l];
    const int N = p.N, D = p.D;
    const int4 ev = p.env4[e];
    const int k = ev.x - ev.y;
    int kind;
    if (after_reset) {
        if (p.mask && !p.mask[e]) return;
        kind = 1;
    } else if (k == 0 && p.auto_reset) kind = 1;                  // finished and auto-reset inside this fleet_step: the finishing
    else if (k >= p.L) return;                                    // step is not logged (:679), the reset row is
    else kind = ((p.step_row[min(ev.x, p.T - 1)].flags & TF_TRIGGER) && p.calc_deg) ? 2 : 0;
    double* row = lg.rows + ((size_t)l * lg.cap + (size_t)(lg.counts[l] % lg.cap)) * lg.row_doubles;
    const size_t i0 = (size_t)e * N;
    if (threadIdx.x == 0) {
        const bool st = kind != 1;
        const double reward = st ? p.env_f64[(size_t)EF_REWARD64 * p.E + e] : 0.0;
        const double cash = st ? p.env_f64[(size_t)EF_CASHFLOW * p.E + e] : 0.0;
        row[0] = (double)ev.z; row[1] = (double)ev.x; row[2] = reward; row[3] = cash;
        row[4] = st ? reward - cash * p.price_mult : 0.0;                                      // :659
        row[5] = st ? p.env_f64[(size_t)EF_OVERLOAD * p.E + e] : 0.0;                          // :660
        row[6] = st ? p.env_f64[(size_t)EF_SOC_VIOL * p.E + e] : 0.0;                          // :661
        row[7] = (double)kind;
        // "Charging energy": EvCharger appends charging_energy + discharging_energy, and those two locals survive
        // from car to car (ev_charger.py:81-82,212): a car's entry carries the last opposite-sign car's energy
        double last_c = 0, last_d = 0;
        double* ce = row + kLogHead + 2 * N;
        for (int n = 0; n < N; n++) {
            double v = 0;
            if (st && p.charge_log && p.actions) {
                const double en = p.charge_log[i0 + n];
                if (p.actions[i0 + n] >= 0.f) last_c = en; else last_d = en;
                v = last_c + last_d;
            }
            ce[n] = v;
        }
    }
    for (int n = threadIdx.x; n < N; n += blockDim.x) {
        row[kLogHead + n] = (kind != 1 && p.actions) ? (double)p.actions[i0 + n] : 0.0;
        row[kLogHead + N + n] = (kind == 2) ? p.last_deg[i0 + n] : 0.0;                        // :665-676
        row[kLogHead + 3 * N + n] = p.soh[i0 + n];
    }
    for (int q = threadIdx.x; q < D; q += blockDim.x) row[kLogHead + 4 * N + q] = p.obs ? (double)p.obs[(size_t)e * D + q] : 0.0;
    __syncthreads();
    if (threadIdx.x == 0) lg.counts[l] += 1;
}

}  // namespace

// =============================================================================================== host side / C ABI

constexpr int kTimingRing = 1024;   // fleet_set_timing keeps the event triplets of the last kTimingRing steps

struct FleetHandle {
    FleetConsts c;
    int device = 0;
    int E = 0, N = 0, T = 0, D = 0;
    StepParams p;
    std::vector<void*> allocs;
    int64_t bytes = 0;
    int64_t launches = 0;
    std::string err;
    size_t smem_step = 0, smem_post = 0, smem_pf = 0;
    int grid_pf = 0, use_pf = 0;
    int pf_cfg2 = 0;                    // the fleet has the shape of the specialised pf instance (PfCfg2Shape)
    int grid = 0, grid_post = 0, need_post = 0, num_sms = 0, post_threads = kPostThreads;
    int max_smem_optin = 0;
    double* charge_log_buf = nullptr;   // fleet_enable_charge_log
    int host_zerocopy = 1;              // fleet_step_host: use page-locked host buffers in place (FLEETSTEP_HOST_ZEROCOPY)
    // rule-based policies (fleet_policy_actions): minute of day per table row; night-charging state, double buffered
    uint16_t* tod = nullptr;
    int2* pol_state[2] = {nullptr, nullptr};
    int pol_flip = 0;
    // optional per-kernel timing (fleet_set_timing): event triplets {before step, between, after post} in a ring
    int timing = 0;
    std::vector<cudaEvent_t> tev;
    int64_t tcount = 0;
    // device-side DataLogger ring (fleet_enable_log)
    int* log_ids = nullptr; long long* log_counts = nullptr; double* log_rows = nullptr;
    int log_n = 0, log_cap = 0, log_row_doubles = 0;
    // host-call staging (fleet_step_host)
    float* h_actions_dev = nullptr; float* h_obs_dev = nullptr; float* h_reward_dev = nullptr; uint8_t* h_done_dev = nullptr;
};

namespace {

int fail(FleetHandle* h, int code, const std::string& msg) {
    if (h) h->err = msg;
    return code;
}

#define CUDA_TRY(h, expr)                                                                              \
    do {                                                                                               \
        cudaError_t _e = (expr);                                                                       \
        if (_e != cudaSuccess)                                                                         \
            return fail(h, FLEET_E_CUDA, std::string(#expr) + ": " + cudaGetErrorString(_e));          \
    } while (0)

template <typename T>
int dev_alloc(FleetHandle* h, T** out, size_t count, bool zero = true) {
    void* ptr = nullptr;
    const size_t bytes = count * sizeof(T);
    cudaError_t e = cudaMalloc(&ptr, bytes ? bytes : 16);
    if (e != cudaSuccess) {
        char buf[256];
        snprintf(buf, sizeof buf, "cudaMalloc of %zu bytes failed: %s (handle already holds %lld bytes)", bytes,
                 cudaGetErrorString(e), (long long)h->bytes);
        return fail(h, FLEET_E_NOMEM, buf);
    }
    if (zero) cudaMemset(ptr, 0, bytes ? bytes : 16);
    h->allocs.push_back(ptr);
    h->bytes += (int64_t)bytes;
    *out = (T*)ptr;
    return FLEET_OK;
}

int obs_dim_of(const FleetConsts& c, int* Ha, int* Hb) {
    int a = 0, b = 0;
    if (c.include_price) a += 2 * (c.price_lookahead + 1);
    if (c.include_price && c.include_building) a += c.bl_pv_lookahead + 1;
    if (c.include_price && c.include_pv) a += c.bl_pv_lookahead + 1;
    if (c.aux) {
        b += 1 + 6;
        if (c.include_price && c.include_building) b += 3;
    }
    *Ha = a; *Hb = b;
    return 2 * c.num_evs + a + (c.aux ? 5 * c.num_evs : 0) + b;   // detect_dim_and_bounds, fleet_environment.py:854-949
}

// look-ahead element k at time index t (observer_bl_pv.py:50-80): 0 -> row t, k>=1 -> first row of the k-th next hour
inline int look_idx(const FleetConsts& c, const FleetTables& tb, int t, int k) {
    const int sph = c.steps_per_hour;
    const int pos = (int)tb.minute[t] * sph / 60;
    int i = (k == 0) ? t : t - pos + k * sph;
    if (i > c.table_len - 1) i = c.table_len - 1;
    return i;
}

using StepKernel = void (*)(const StepParams);

StepKernel pick_step(const FleetHandle* h) {
    if (h->c.normalize) return h->c.aux ? fleet_step_kernel<true, true> : fleet_step_kernel<true, false>;
    return h->c.aux ? fleet_step_kernel<false, true> : fleet_step_kernel<false, false>;
}
// The fleet has exactly the compile-time shape S and the flags of its instance (kNorm = false, kAux = true).
template <class S>
bool pf_shape_is(const FleetHandle* h) {
    const StepParams& p = h->p;
    return !h->c.normalize && h->c.aux && p.N == S::N && p.D == S::D && p.Ha == S::Ha && p.Hb == S::Hb && p.R == S::R;
}
StepKernel pick_pf(const FleetHandle* h, bool log) {
    using A = PfAnyShape;
    if (h->pf_cfg2 && !log) return fleet_step_pf_kernel<false, true, false, PfCfg2Shape>;
    if (log) {
        if (h->c.normalize) return h->c.aux ? fleet_step_pf_kernel<true, true, true, A> : fleet_step_pf_kernel<true, false, true, A>;
        return h->c.aux ? fleet_step_pf_kernel<false, true, true, A> : fleet_step_pf_kernel<false, false, true, A>;
    }
    if (h->c.normalize) return h->c.aux ? fleet_step_pf_kernel<true, true, false, A> : fleet_step_pf_kernel<true, false, false, A>;
    return h->c.aux ? fleet_step_pf_kernel<false, true, false, A> : fleet_step_pf_kernel<false, false, false, A>;
}
template <int kT>
StepKernel pick_post_t(const FleetHandle* h) {
    if (h->c.normalize) return h->c.aux ? fleet_post_kernel<true, true, kT> : fleet_post_kernel<true, false, kT>;
    return h->c.aux ? fleet_post_kernel<false, true, kT> : fleet_post_kernel<false, false, kT>;
}
StepKernel pick_post(const FleetHandle* h) { return h->post_threads == 32 ? pick_post_t<32>(h) : pick_post_t<64>(h); }
StepKernel pick_reset(const FleetHandle* h) {
    if (h->c.normalize) return h->c.aux ? fleet_reset_kernel<true, true> : fleet_reset_kernel<true, false>;
    return h->c.aux ? fleet_reset_kernel<false, true> : fleet_reset_kernel<false, false>;
}

}  // namespace

static void fleet_log_launch(FleetHandle* h, const StepParams& p, int after_reset, cudaStream_t stream) {
    LogParams lg;
    lg.ids = h->log_ids; lg.counts = h->log_counts; lg.rows = h->log_rows;
    lg.n = h->log_n; lg.cap = h->log_cap; lg.row_doubles = h->log_row_doubles;
    fleet_log_kernel<<<h->log_n, 128, 0, stream>>>(p, lg, after_reset);
    h->launches++;
}

// every device array that makes up the env state, in the order fleet_export_state writes them
static std::vector<std::pair<void*, size_t>> state_arrays(FleetHandle* h) {
    const StepParams& p = h->p;
    const size_t E = (size_t)h->E, EN = E * (size_t)h->N;
    std::vector<std::pair<void*, size_t>> v;
    v.push_back({p.env4, E * sizeof(int4)});
    v.push_back({p.soc, EN * 8}); v.push_back({p.hl, EN * 4}); v.push_back({p.soh, EN * 8});
    v.push_back({p.hist, EN * (size_t)p.R * 8});
    v.push_back({p.tflip, EN}); v.push_back({p.n_flips, 4});
    v.push_back({p.env_f64, (size_t)EF__COUNT * E * 8});
    v.push_back({p.rf_len, EN * 4}); v.push_back({p.fd_cyc, EN * 8}); v.push_back({p.life, EN * 8});
    v.push_back({p.n_cycles, EN * 4}); v.push_back({p.last_deg, EN * 8});
    if (p.rf_on) {
        v.push_back({p.rf_stack, EN * (size_t)p.rf_S * 8}); v.push_back({p.rf_dc, EN * 4}); v.push_back({p.rf_acc, EN * 16});
        v.push_back({p.rf_ext, EN * 4});
        v.push_back({p.ext_owner, (size_t)(p.rf_P > 0 ? p.rf_P : 1) * 4});
        v.push_back({p.ext_val, (size_t)(p.rf_P > 0 ? p.rf_P : 1) * (size_t)(p.rf_X > 0 ? p.rf_X : 1) * 8});
    }
    v.push_back({p.stats, sizeof(double) * kStatStripes * FLEET_S__COUNT});
    return v;
}
struct StateHeader { uint64_t magic; int32_t E, N, R, S, X, P, L, T; };
constexpr uint64_t kStateMagic = 0x464c54535432ull;   // "FLTST2"

extern "C" {

int fleet_abi_version(void) { return FLEETSTEP_ABI_VERSION; }

int fleet_enable_log(FleetHandle* h, const int32_t* env_ids_host, int32_t n_envs, int32_t rows_per_env) {
    if (!h) return FLEET_E_INVALID;
    CUDA_TRY(h, cudaSetDevice(h->device));
    if (h->log_n) return fail(h, FLEET_E_INVALID, "the log is already enabled on this handle");
    if (!env_ids_host || n_envs < 1 || rows_per_env < 1) return fail(h, FLEET_E_INVALID, "fleet_enable_log: need env ids, n_envs >= 1 and rows_per_env >= 1");
    for (int k = 0; k < n_envs; k++)
        if (env_ids_host[k] < 0 || env_ids_host[k] >= h->E) return fail(h, FLEET_E_INVALID, "fleet_enable_log: env id out of range");
    int rc;
    if ((rc = fleet_enable_charge_log(h, 1))) return rc;     // "Charging energy" needs EvCharger's charge_log
    const int rd = kLogHead + 4 * h->N + h->D;
    if ((rc = dev_alloc(h, &h->log_ids, (size_t)n_envs))) return rc;
    if ((rc = dev_alloc(h, &h->log_counts, (size_t)n_envs))) return rc;
    if ((rc = dev_alloc(h, &h->log_rows, (size_t)n_envs * (size_t)rows_per_env * (size_t)rd))) return rc;
    CUDA_TRY(h, cudaMemcpy(h->log_ids, env_ids_host, sizeof(int) * (size_t)n_envs, cudaMemcpyHostToDevice));
    h->log_n = n_envs; h->log_cap = rows_per_env; h->log_row_doubles = rd;
    return FLEET_OK;
}

int fleet_log_layout(const FleetHandle* h, int32_t* n_envs, int32_t* rows_per_env, int32_t* row_doubles) {
    if (!h) return FLEET_E_INVALID;
    if (n_envs) *n_envs = h->log_n;
    if (rows_per_env) *rows_per_env = h->log_cap;
    if (row_doubles) *row_doubles = h->log_row_doubles;
    return FLEET_OK;
}

int fleet_read_log(FleetHandle* h, double* rows_host, int64_t* counts_host, void* stream) {
    if (!h) return FLEET_E_INVALID;
    if (!h->log_n) return fail(h, FLEET_E_STATE, "fleet_read_log: the log is not enabled (fleet_enable_log)");
    CUDA_TRY(h, cudaSetDevice(h->device));
    const size_t nb = (size_t)h->log_n * (size_t)h->log_cap * (size_t)h->log_row_doubles * 8;
    if (rows_host) CUDA_TRY(h, cudaMemcpyAsync(rows_host, h->log_rows, nb, cudaMemcpyDeviceToHost, (cudaStream_t)stream));
    if (counts_host) CUDA_TRY(h, cudaMemcpyAsync(counts_host, h->log_counts, sizeof(long long) * (size_t)h->log_n, cudaMemcpyDeviceToHost, (cudaStream_t)stream));
    CUDA_TRY(h, cudaStreamSynchronize((cudaStream_t)stream));
    return FLEET_OK;
}

int64_t fleet_state_bytes(FleetHandle* h) {
    if (!h) return 0;
    size_t n = sizeof(StateHeader);
    for (auto& a : state_arrays(h)) n += a.second;
    return (int64_t)n;
}

// The blob holds the state as the kernels left it: an env exported after the last daily evaluation of its episode may
// hold a history ring that has wrapped over samples the rainflow state never consumed (k_done < k_now - R + 1).  Nothing
// reads them before the env's next reset, so an import continues it exactly.
int fleet_export_state(FleetHandle* h, void* dst_host, void* stream) {
    if (!h || !dst_host) return FLEET_E_INVALID;
    CUDA_TRY(h, cudaSetDevice(h->device));
    const StepParams& p = h->p;
    StateHeader hd = {kStateMagic, h->E, h->N, p.R, p.rf_S, p.rf_X, p.rf_P, p.L, p.T};
    unsigned char* dst = (unsigned char*)dst_host;
    memcpy(dst, &hd, sizeof hd);
    size_t off = sizeof hd;
    for (auto& a : state_arrays(h)) {
        CUDA_TRY(h, cudaMemcpyAsync(dst + off, a.first, a.second, cudaMemcpyDeviceToHost, (cudaStream_t)stream));
        off += a.second;
    }
    CUDA_TRY(h, cudaStreamSynchronize((cudaStream_t)stream));
    return FLEET_OK;
}

int fleet_import_state(FleetHandle* h, const void* src_host, void* stream) {
    if (!h || !src_host) return FLEET_E_INVALID;
    CUDA_TRY(h, cudaSetDevice(h->device));
    const StepParams& p = h->p;
    StateHeader hd;
    memcpy(&hd, src_host, sizeof hd);
    if (hd.magic != kStateMagic || hd.E != h->E || hd.N != h->N || hd.R != p.R || hd.S != p.rf_S || hd.X != p.rf_X ||
        hd.P != p.rf_P || hd.L != p.L || hd.T != p.T)
        return fail(h, FLEET_E_INVALID, "fleet_import_state: the blob was exported from a handle with a different geometry");
    const unsigned char* src = (const unsigned char*)src_host;
    size_t off = sizeof hd;
    for (auto& a : state_arrays(h)) {
        CUDA_TRY(h, cudaMemcpyAsync(a.first, src + off, a.second, cudaMemcpyHostToDevice, (cudaStream_t)stream));
        off += a.second;
    }
    CUDA_TRY(h, cudaStreamSynchronize((cudaStream_t)stream));
    return FLEET_OK;
}


const char* fleet_last_error(const FleetHandle* h) { return h ? h->err.c_str() : "null handle"; }

int fleet_obs_dim(const FleetHandle* h) { return h ? h->D : FLEET_E_INVALID; }
int fleet_num_evs(const FleetHandle* h) { return h ? h->N : FLEET_E_INVALID; }
int fleet_num_envs(const FleetHandle* h) { return h ? h->E : FLEET_E_INVALID; }
int64_t fleet_launch_count(const FleetHandle* h) { return h ? h->launches : 0; }

int fleet_enable_charge_log(FleetHandle* h, int32_t enable) {
    if (!h) return FLEET_E_INVALID;
    CUDA_TRY(h, cudaSetDevice(h->device));
    if (enable && !h->charge_log_buf) {
        int rc;
        if ((rc = dev_alloc(h, &h->charge_log_buf, (size_t)h->E * h->N))) return rc;
    }
    h->p.charge_log = enable ? h->charge_log_buf : nullptr;
    return FLEET_OK;
}

const char* fleet_step_kernel_name(const FleetHandle* h) {
    if (!h) return "";
    // the pf name keeps its historical template suffix: bench.py reports it as `kernel` and the recorded profiles carry it
    return h->use_pf ? "fleet_step_pf_kernel<kV=1>" : "fleet_step_kernel";
}

int fleet_launch_geometry(const FleetHandle* h, int32_t* step_grid, int32_t* step_tiles, int32_t* envs_per_tile,
                          int32_t* post_grid) {
    if (!h) return FLEET_E_INVALID;
    const int B = h->use_pf ? h->p.pf_B : h->p.B;
    if (step_grid) *step_grid = h->use_pf ? h->grid_pf : h->grid;
    if (step_tiles) *step_tiles = h->use_pf ? h->p.pf_ntiles : h->grid;
    if (envs_per_tile) *envs_per_tile = B;
    if (post_grid) *post_grid = h->need_post ? h->grid_post : 0;
    return FLEET_OK;
}

int fleet_set_timing(FleetHandle* h, int32_t enable) {
    if (!h) return FLEET_E_INVALID;
    CUDA_TRY(h, cudaSetDevice(h->device));
    if (enable && h->tev.empty()) {
        h->tev.resize((size_t)kTimingRing * 3);
        for (auto& ev : h->tev) CUDA_TRY(h, cudaEventCreate(&ev));
    }
    h->timing = enable ? 1 : 0;
    h->tcount = 0;
    return FLEET_OK;
}

int fleet_get_timing(FleetHandle* h, double* step_ms, double* post_ms, int64_t* steps) {
    if (!h) return FLEET_E_INVALID;
    CUDA_TRY(h, cudaSetDevice(h->device));
    const int64_t n = h->tcount < kTimingRing ? h->tcount : kTimingRing;
    double a = 0, b = 0;
    for (int64_t k = 0; k < n; k++) {
        cudaEvent_t* tev = &h->tev[(size_t)k * 3];
        float t0 = 0, t1 = 0;
        CUDA_TRY(h, cudaEventSynchronize(tev[2]));
        CUDA_TRY(h, cudaEventElapsedTime(&t0, tev[0], tev[1]));
        CUDA_TRY(h, cudaEventElapsedTime(&t1, tev[1], tev[2]));
        a += t0; b += t1;
    }
    if (step_ms) *step_ms = a;
    if (post_ms) *post_ms = b;
    if (steps) *steps = n;
    return FLEET_OK;
}
#ifdef POST_TIMING
int32_t fleet_debug_post_clk(unsigned long long* out, int32_t reset) {
    cudaDeviceSynchronize();
    cudaMemcpyFromSymbol(out, g_post_clk, sizeof(unsigned long long) * 16);
    if (reset) { unsigned long long z[16] = {0}; cudaMemcpyToSymbol(g_post_clk, z, sizeof(z)); }
    return 0;
}
#endif
#ifdef PF_TIMING
int32_t fleet_debug_pf_clk(unsigned long long* out, int32_t reset) {
    cudaDeviceSynchronize();
    cudaMemcpyFromSymbol(out, g_pf_clk, sizeof(unsigned long long) * (16 + 128));     /* out: 144 values */
    if (reset) { unsigned long long z[16 + 128] = {0}; cudaMemcpyToSymbol(g_pf_clk, z, sizeof(z)); }
    return 0;
}
int32_t fleet_debug_pf_trace(unsigned long long* out) {   /* out: 640 values, g_pf_trace of the last launch */
    cudaDeviceSynchronize();
    cudaMemcpyFromSymbol(out, g_pf_trace, sizeof(unsigned long long) * 640);
    return 0;
}
#endif
int64_t fleet_device_bytes(const FleetHandle* h) { return h ? h->bytes : 0; }

int fleet_debug_stress(const double* eff_dev, const double* mean_dev, double* out_dev, int32_t n, void* stream) {
    if (!eff_dev || !mean_dev || !out_dev || n < 0) return FLEET_E_INVALID;
    if (n) debug_stress_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(eff_dev, mean_dev, out_dev, n);
    return cudaGetLastError() == cudaSuccess ? FLEET_OK : FLEET_E_CUDA;
}

int fleet_destroy(FleetHandle* h) {
    if (!h) return FLEET_E_INVALID;
    cudaSetDevice(h->device);
    for (cudaEvent_t ev : h->tev) cudaEventDestroy(ev);
    for (void* ptr : h->allocs) cudaFree(ptr);
    delete h;
    return FLEET_OK;
}

int fleet_create(const FleetConsts* consts, const FleetTables* tb, int32_t num_envs, int32_t device, int64_t env_id_offset,
                 FleetHandle** out) {
    if (!out) return FLEET_E_INVALID;
    *out = nullptr;
    FleetHandle* h = new FleetHandle();
    *out = h;  // returned even on failure so that fleet_last_error works; caller destroys it
    if (!consts || !tb) return fail(h, FLEET_E_INVALID, "consts/tables is NULL");
    const FleetConsts& c = *consts;
    if (c.abi_version != FLEETSTEP_ABI_VERSION) return fail(h, FLEET_E_INVALID, "FleetConsts.abi_version mismatch");
    if (num_envs < 1 || c.num_evs < 1 || c.table_len < 3) return fail(h, FLEET_E_INVALID, "num_envs, num_evs must be >= 1 and table_len >= 3");
    if (!c.include_price)
        return fail(h, FLEET_E_INVALID, "include_price=False is unsupported: the reference raises KeyError('price_reward_curve') at ev_charger.py:155");
    if (c.normalize && c.include_pv && !c.include_building)
        return fail(h, FLEET_E_INVALID, "normalize_in_env with PV only is unsupported: the reference raises at oracle_normalization.py:120-121");
    if (!tb->there || !tb->time_left || !tb->soc_on_return || !tb->delu || !tb->tariff || !tb->price_reward_curve ||
        !tb->tariff_reward_curve || !tb->cal_sincos || !tb->hour || !tb->minute)
        return fail(h, FLEET_E_INVALID, "a mandatory table pointer is NULL");
    if (c.include_building && !tb->load) return fail(h, FLEET_E_INVALID, "include_building set but load table is NULL");
    if (c.include_pv && !tb->pv) return fail(h, FLEET_E_INVALID, "include_pv set but pv table is NULL");
    if (c.steps_per_hour < 1 || c.episode_steps < 1) return fail(h, FLEET_E_INVALID, "steps_per_hour and episode_steps must be >= 1");
    if ((double)(float)c.dt != c.dt) return fail(h, FLEET_E_INVALID, "dt is not exactly representable in float32 (hours_left is kept in float32)");
    if (c.episode_steps + 1 > 65535) return fail(h, FLEET_E_INVALID, "episodes longer than 65534 steps are not supported (16-bit cycle counters)");

    h->c = c; h->device = device; h->E = num_envs; h->N = c.num_evs; h->T = c.table_len;
    const int E = h->E, N = h->N, T = h->T;
    int Ha = 0, Hb = 0;
    h->D = obs_dim_of(c, &Ha, &Hb);

    cudaError_t ce = cudaSetDevice(device);
    if (ce != cudaSuccess) return fail(h, FLEET_E_CUDA, std::string("cudaSetDevice: ") + cudaGetErrorString(ce) + " (no CPU fallback exists)");
    cudaDeviceProp prop;
    CUDA_TRY(h, cudaGetDeviceProperties(&prop, device));
    h->max_smem_optin = (int)prop.sharedMemPerBlockOptin;
    // (a persisting-L2 set-aside for the tables was measured: it shrinks the write-combining capacity for the streaming
    //  state and made the step 45 % slower, so only per-access evict_last / evict-first hints are used)

    // ---- build the HBM tables on the host (float64, reference operation order), then upload
    std::vector<EvRec> rec((size_t)T * N);
    for (int n = 0; n < N; n++) {
        for (int t = 0; t < T; t++) {
            const double tl = tb->time_left[(size_t)n * T + t];
            const float tlf = (float)tl;
            const double steps = tl / c.dt;
            if ((double)tlf != tl || steps != floor(steps) || steps > 4194304.0) {
                char buf[200];
                snprintf(buf, sizeof buf, "time_left[%d][%d]=%.17g is not an exact float32 multiple of dt=%.17g", n, t, tl, c.dt);
                return fail(h, FLEET_E_INVALID, buf);
            }
            EvRec& r = rec[(size_t)t * N + n];
            r.sr = tb->soc_on_return[(size_t)n * T + t];
            r.tl = tlf;
            r.there = tb->there[(size_t)n * T + t];
            r.there_prev = t > 0 ? tb->there[(size_t)n * T + t - 1] : 0;
            r.pad = 0;
            // auxiliary observation terms for the configured target SOC (observer_bl_pv.py:85-91), normalised per
            // oracle_normalization.py:146-150 when requested; float64 in the reference's order, cast once.
            {
                const double th = (double)r.there;
                double tt = (1.0 * c.target_soc) * th;
                double cl = tt - r.sr;
                double hn = cl * c.lc_batt_cap / (c.evse_max_power * c.charging_eff);
                double lax = (tl / (hn + 0.001) - 1) * th;
                lax = lax < 0 ? 0 : (lax > 5 ? 5 : lax);
                if (c.normalize) {
                    const double max_soc = c.target_soc;
                    const double max_hn = (c.target_soc * c.init_battery_cap) / (c.evse_max_power * c.charging_eff);
                    tt = tt / max_soc; cl = cl / max_soc; hn = hn / max_hn; lax = lax / 5;
                }
                r.tt = (float)tt; r.cl = (float)cl; r.hn = (float)hn; r.lax = (float)lax;
            }
        }
    }
    std::vector<StepRow> rows((size_t)T);
    const double spot_offset = c.fixed_markup / 1000;                                    // ev_charger.py:35
    // next_trig[t]: the first 14:45 row at or after t (T: none)
    std::vector<int> next_trig((size_t)T + 2, T);
    for (int t = T - 1; t >= 0; t--) next_trig[t] = (tb->hour[t] == 14 && tb->minute[t] == 45) ? t : next_trig[t + 1];
    for (int t = 0; t < T; t++) {
        StepRow& r = rows[t];
        double connected = 0;
        for (int n = 0; n < N; n++) connected += (double)tb->there[(size_t)n * T + t];   // ev_charger.py:138
        connected = connected > 1 ? connected : 1;                                       // :140
        const double pv_energy = tb->pv ? tb->pv[t] * c.dt : 0.0;                        // :133-136
        r.S = tb->delu[t] / 1000.0 + spot_offset;                                        // :145,149
        r.F_cr = -1 * c.price_multiplier * tb->price_reward_curve[t] / 1000;             // :154-156
        r.F_dr = -1 * c.price_multiplier * tb->tariff_reward_curve[t] / 1000;            // :204-206
        r.Rfac = c.discharging_eff * tb->tariff[t] / 1000 * (1 - c.feed_in_deduction);   // :196-199 (regrouped; cashflow tolerance)
        r.pv_share = pv_energy / connected;                                              // :142
        r.gml = c.grid_connection - ((c.include_building && tb->load) ? tb->load[t] : 0.0);  // load_calculation.py:93
        r.pvv = (c.include_pv && tb->pv) ? tb->pv[t] : 0.0;
        auto tf = [&](int tt) -> uint32_t {
            uint32_t f = 0;
            if (tb->hour[tt] == 14 && tb->minute[tt] == 45) f |= TF_TRIGGER;
            if (tb->hour[tt] > 11 && tb->hour[tt] < 15) f |= TF_LUNCH;
            return f;
        };
        r.flags = tf(t);
        const int nt = next_trig[t + 2 < T ? t + 2 : T];
        const uint32_t dist = nt < T ? std::min((uint32_t)(nt - t), TF_DIST_NONE) : TF_DIST_NONE;
        r.flags_next = tf(t + 1 < T ? t + 1 : T - 1) | dist << TF_DIST_SHIFT;
    }
    const int hdr_stride = ((Ha + Hb + 3) / 4) * 4 > 0 ? ((Ha + Hb + 3) / 4) * 4 : 4;
    std::vector<float> hdr((size_t)T * hdr_stride, 0.f);
    const bool norm = c.normalize != 0;
    for (int t = 0; t < T; t++) {
        float* o = hdr.data() + (size_t)t * hdr_stride;
        int q = 0;
        for (int k = 0; k <= c.price_lookahead; k++) {                                   // observer_bl_pv.py:63
            double v = (tb->delu[look_idx(c, *tb, t, k)] + c.fixed_markup) * c.variable_multiplier;
            if (norm) v = (v - c.min_price) / (c.max_price - c.min_price);               // oracle_normalization.py:70
            o[q++] = (float)v;
        }
        for (int k = 0; k <= c.price_lookahead; k++) {                                   // observer_bl_pv.py:64
            double v = tb->tariff[look_idx(c, *tb, t, k)] * (1 - c.feed_in_deduction);
            if (norm) v = (v - c.min_tariff) / (c.max_tariff - c.min_tariff);            // :72
            o[q++] = (float)v;
        }
        if (c.include_building)
            for (int k = 0; k <= c.bl_pv_lookahead; k++) {
                double v = tb->load[look_idx(c, *tb, t, k)];
                if (norm) v = v / c.max_building;
                o[q++] = (float)v;
            }
        if (c.include_pv)
            for (int k = 0; k <= c.bl_pv_lookahead; k++) {
                double v = tb->pv[look_idx(c, *tb, t, k)];
                if (norm) v = v / c.max_pv;
                o[q++] = (float)v;
            }
        if (c.aux) {
            double evse = c.evse_max_power;
            o[q++] = (float)(norm ? evse / c.evse_max_power : evse);                     // observer_bl_pv.py:93
            if (c.include_building) {
                double grid = c.grid_connection;                                         // :95
                double avail = grid - tb->load[t];                                       // :96
                if (c.include_pv) avail = avail + tb->pv[t];
                double poss = avail / ((double)N * evse);                                // :98
                if (poss > 1) poss = 1;
                if (norm) { grid = grid / c.grid_connection; avail = avail / c.grid_connection; poss = poss / 1; }
                o[q++] = (float)grid; o[q++] = (float)avail; o[q++] = (float)poss;
            }
            for (int k = 0; k < 6; k++) o[q++] = (float)tb->cal_sincos[(size_t)t * 6 + k];   // :100-107
        }
    }

    // ---- device allocations
    StepParams& p = h->p;
    memset(&p, 0, sizeof p);
    EvRec* d_rec; StepRow* d_rows; float* d_hdr;
    int rc;
    if ((rc = dev_alloc(h, &d_rec, rec.size(), false))) return rc;
    if ((rc = dev_alloc(h, &d_rows, rows.size(), false))) return rc;
    if ((rc = dev_alloc(h, &d_hdr, hdr.size(), false))) return rc;
    CUDA_TRY(h, cudaMemcpy(d_rec, rec.data(), rec.size() * sizeof(EvRec), cudaMemcpyHostToDevice));
    CUDA_TRY(h, cudaMemcpy(d_rows, rows.data(), rows.size() * sizeof(StepRow), cudaMemcpyHostToDevice));
    CUDA_TRY(h, cudaMemcpy(d_hdr, hdr.data(), hdr.size() * sizeof(float), cudaMemcpyHostToDevice));

    // History ring and incremental rainflow geometry.  Samples are only needed until the post kernel has consumed them
    // (at the daily trigger, or when the ring is about to wrap while an evaluation remains in the episode), so R rows
    // suffice for any episode length.
    bool any_trigger = false;
    for (int t = 0; t < T; t++) any_trigger = any_trigger || (rows[t].flags & TF_TRIGGER);
    const bool rf_on = c.calc_degradation && c.deg_mode == FLEET_DEG_SEI && any_trigger;   // (no 14:45 row, e.g. 1-h grids: never evaluated)
    auto env_int = [](const char* name, int dflt) { const char* v = getenv(name); return (v && *v) ? atoi(v) : dflt; };
    int R = 2;
    if (rf_on) {
        int want = c.rf_ring_rows > 0 ? c.rf_ring_rows : env_int("FLEETSTEP_RF_RING", 16);
        if (want < 4) want = 4;
        while (R < want) R <<= 1;                                                          // power of two: row = k & (R-1)
    }
    int rfS = 0, rfX = 0, rfP = 0;
    const size_t EN = (size_t)E * N;
    if (rf_on) {
        rfS = c.rf_stack_depth > 0 ? c.rf_stack_depth : env_int("FLEETSTEP_RF_STACK", 12);
        if (rfS < 2) rfS = 2;
        if (rfS > c.episode_steps + 1) rfS = c.episode_steps + 1;                          // a stack can never be deeper than the log
        if (rfS < 2) rfS = 2;
        rfS += rfS & 1;                                                                    // even: 16-byte vector access
        if (rfS > 256) return fail(h, FLEET_E_INVALID, "rf_stack_depth > 256 is not supported (shared-memory stack copy)");
        rfX = env_int("FLEETSTEP_RF_EXT", 52);
        if (rfS + rfX > c.episode_steps + 1) rfX = c.episode_steps + 1 - rfS;
        if (rfX < 0) rfX = 0;
        rfP = rfX > 0 ? env_int("FLEETSTEP_RF_EXT_SLOTS", (int)(EN / 128 < 64 ? 64 : (EN / 128 > (1u << 20) ? (1u << 20) : EN / 128))) : 0;
        if (EN >= 0x7fffffffull) return fail(h, FLEET_E_INVALID, "num_envs * num_evs must be below 2^31");
    }
    if ((rc = dev_alloc(h, &p.env4, (size_t)E))) return rc;
    if ((rc = dev_alloc(h, &p.soc, EN))) return rc;
    if ((rc = dev_alloc(h, &p.hl, EN))) return rc;
    if ((rc = dev_alloc(h, &p.soh, EN))) return rc;
    if ((rc = dev_alloc(h, &p.hist, EN * (size_t)R))) return rc;
    if ((rc = dev_alloc(h, &p.tflip, EN))) return rc;
    if ((rc = dev_alloc(h, &p.n_flips, (size_t)4))) return rc;
    if ((rc = dev_alloc(h, &p.env_f64, (size_t)EF__COUNT * E))) return rc;
    if ((rc = dev_alloc(h, &p.rf_len, EN))) return rc;
    if ((rc = dev_alloc(h, &p.fd_cyc, EN))) return rc;
    if ((rc = dev_alloc(h, &p.life, EN))) return rc;
    if ((rc = dev_alloc(h, &p.n_cycles, EN))) return rc;
    if ((rc = dev_alloc(h, &p.last_deg, EN))) return rc;
    if ((rc = dev_alloc(h, &p.stats, (size_t)kStatStripes * FLEET_S__COUNT))) return rc;
    if ((rc = dev_alloc(h, &p.err_flags, (size_t)4))) return rc;
    if ((rc = dev_alloc(h, &p.wl, (size_t)E))) return rc;
    if ((rc = dev_alloc(h, &p.wl_flush, (size_t)E))) return rc;
    if (rf_on) {
        if ((rc = dev_alloc(h, &p.rf_stack, EN * (size_t)rfS))) return rc;
        if ((rc = dev_alloc(h, &p.rf_dc, EN))) return rc;
        if ((rc = dev_alloc(h, &p.rf_acc, EN))) return rc;
        if ((rc = dev_alloc(h, &p.rf_ext, EN))) return rc;
        if ((rc = dev_alloc(h, &p.ext_owner, (size_t)(rfP > 0 ? rfP : 1)))) return rc;
        if ((rc = dev_alloc(h, &p.ext_val, (size_t)(rfP > 0 ? rfP : 1) * (size_t)(rfX > 0 ? rfX : 1), false))) return rc;
        CUDA_TRY(h, cudaMemset(p.ext_owner, 0xff, sizeof(int) * (size_t)(rfP > 0 ? rfP : 1)));
    }
    if ((rc = dev_alloc(h, &p.wl_count, (size_t)8))) return rc;
    if ((rc = dev_alloc(h, &p.wl_done, (size_t)4))) return rc;

    p.rf_on = rf_on ? 1 : 0; p.rf_S = rfS; p.rf_X = rfX; p.rf_P = rfP;
    p.E = E; p.N = N; p.T = T; p.R = R; p.Rm = R - 1; p.L = c.episode_steps; p.D = h->D; p.Ha = Ha; p.Hb = Hb; p.hdr_stride = hdr_stride;
    p.B = N >= kThreads ? 1 : kThreads / N;
    p.RN = (unsigned long long)R * (unsigned long long)N;
    p.is_ct = c.is_caretaker; p.calc_deg = c.calc_degradation; p.deg_mode = c.deg_mode; p.carry = c.carry_degradation_state;
    p.auto_reset = c.auto_reset; p.start_lo = c.start_lo; p.start_hi = c.start_hi; p.seed = c.seed;
    p.env_id_offset = env_id_offset;
    p.dt = c.dt; p.dt_f = (float)c.dt;
    p.P = c.obc_max_power < c.evse_max_power ? c.obc_max_power : c.evse_max_power;       // ev_charger.py:95
    p.eta_c = c.charging_eff; p.eta_d = c.discharging_eff; p.mult = c.variable_multiplier; p.cap0 = c.init_battery_cap;
    p.target = 1.0 * c.target_soc; p.target_lunch = c.target_soc_lunch; p.eps = c.soc_eps; p.def_soc = c.def_soc;
    p.min_lax = c.min_laxity; p.pen_inv = c.penalty_invalid_action; p.pen_oc = c.penalty_overcharging;
    p.clip_oc = c.clip_overcharging; p.pen_ovl = c.penalty_overloading; p.full_reward = c.fully_charged_reward;
    p.evse = c.evse_max_power; p.grid = c.grid_connection; p.init_soh = c.init_soh; p.lc_batt_cap = c.lc_batt_cap;
    p.hn_den = c.evse_max_power * c.charging_eff;                                        // observer_bl_pv.py:89
    p.price_mult = c.price_multiplier; p.temperature = c.temperature;
    p.max_tl = c.max_time_left; p.max_soc = c.target_soc;                                // oracle_normalization.py:34,49
    p.max_hn = (c.target_soc * c.init_battery_cap) / (c.evse_max_power * c.charging_eff);   // :50-51
    p.ev_rec = d_rec; p.step_row = d_rows; p.hdr = d_hdr;
    {
        std::vector<uint16_t> tod((size_t)T);
        for (int tt = 0; tt < T; tt++) tod[tt] = (uint16_t)(tb->hour[tt] * 60 + tb->minute[tt]);
        if ((rc = dev_alloc(h, &h->tod, (size_t)T, false))) return rc;
        CUDA_TRY(h, cudaMemcpy(h->tod, tod.data(), tod.size() * sizeof(uint16_t), cudaMemcpyHostToDevice));
    }

    p.n_magic = (unsigned int)((0x100000000ull + (unsigned long long)N - 1) / (unsigned long long)N);
    {
        const unsigned long long Hh = (unsigned long long)(Ha + Hb > 0 ? Ha + Hb : 1);
        p.h_magic = (unsigned int)((0x100000000ull + Hh - 1) / Hh);
    }
    p.off_contrib = (int)smem_envs_bytes(p.B);
    p.off_obs = (int)smem_obs_offset(p.B, N);
    p.bulk_ok = ((p.B * h->D) % 4 == 0) ? 1 : 0;

    // shared memory of the step kernel: env scratch + contributions + sums + obs tile
    size_t sm = smem_step_bytes(p.B, N, h->D);
    if ((int64_t)sm > (int64_t)h->max_smem_optin) {
        char buf[256];
        snprintf(buf, sizeof buf, "step kernel needs %zu bytes of shared memory (N=%d, D=%d) but the device allows %d", sm, N,
                 h->D, h->max_smem_optin);
        return fail(h, FLEET_E_INVALID, buf);
    }
    // post kernel: one CTA of kPostThreads threads per work-list env; shared memory = the vehicles' stack copies + the
    // per-batch reversal lists
    h->num_sms = prop.multiProcessorCount;
    h->need_post = (c.calc_degradation || c.auto_reset) ? 1 : 0;
    // one warp per work item for fleets of up to 32 vehicles (cfg3: 35 instead of 49 us), two warps otherwise (a 50-vehicle
    // env as two one-warp items of 25 lanes measured 55 against 52 us)
    h->post_threads = N <= 32 ? 32 : 64;
    p.post_chunks = (N + h->post_threads - 1) / h->post_threads;
    p.post_cv = (N + p.post_chunks - 1) / p.post_chunks;
    if (p.post_chunks > 1 && (rc = dev_alloc(h, &p.wl_chunks, (size_t)E))) return rc;
    h->smem_post = align16((size_t)(rfS + kRfQueue + 2 * kRfPend) * h->post_threads * 8);
    if ((int64_t)h->smem_post > (int64_t)h->max_smem_optin) return fail(h, FLEET_E_INVALID, "rf_stack_depth does not fit the post kernel's shared memory");
    {
        int per_sm = 1;
        CUDA_TRY(h, cudaFuncSetAttribute(pick_post(h), cudaFuncAttributeMaxDynamicSharedMemorySize, (int)h->smem_post));
        CUDA_TRY(h, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, pick_post(h), h->post_threads, h->smem_post));
        if (per_sm < 1) per_sm = 1;
        const int64_t g = (int64_t)h->num_sms * per_sm;
        h->grid_post = (int)(g < E ? g : E);
        // FLEETSTEP_POST_GRID=G (diagnostic, G >= 1) caps the grid so that every CTA fetches many work items per launch
        const int cap = env_int("FLEETSTEP_POST_GRID", 0);
        if (cap > 0 && cap < h->grid_post) h->grid_post = cap;
    }
    h->smem_step = sm;
    {
        const char* zc = getenv("FLEETSTEP_HOST_ZEROCOPY");
        h->host_zerocopy = (zc && atoi(zc) == 0) ? 0 : 1;
    }
    // persistent prefetching kernel (default where applicable)
    {
        const char* force = getenv("FLEETSTEP_KERNEL");   // "generic" / "pf"; default: pf when applicable
        const bool want = !force || strcmp(force, "pf") == 0;
        const int pfB = kPfSlots / N;
        if (want && c.auto_reset && N >= 8 && pfB >= 1 && pfB <= 32) {   // the epilogue warps use one lane per env of a tile
            const PfLayout l = pf_layout(N, h->D, R);
            const size_t smpf = l.smem;
            h->pf_cfg2 = pf_shape_is<PfCfg2Shape>(h) ? 1 : 0;
            int per_sm = 0;
            if ((int64_t)smpf <= (int64_t)h->max_smem_optin &&
                cudaFuncSetAttribute(pick_pf(h, false), cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smpf) == cudaSuccess &&
                cudaFuncSetAttribute(pick_pf(h, true), cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smpf) == cudaSuccess &&
                cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, pick_pf(h, true), kPfThreads, smpf) == cudaSuccess && per_sm >= 1) {
                h->smem_pf = smpf;
                const int ntiles = (E + pfB - 1) / pfB;
                p.pf_B = l.B;
                p.pf_bulk = 1;                                  // (cleared per call when obs / terminal_obs are not 16-byte aligned)
                p.pf_ntiles = ntiles;
                p.pf_tile_hist = l.tile_hist;
                p.pf_pair = l.pair;
                p.pf_cslots = l.cslots;
                p.pf_cper = l.cper;
                p.pf_envs_b = l.envs_b;
                p.pf_contrib_b = l.contrib_b;
                p.pf_obs_b = l.obs_b;
                p.pf_off_contrib = l.off_contrib;
                p.pf_off_sums = l.off_sums;
                p.pf_off_obs = l.off_obs;
                p.pf_off_stage = l.off_stage;
                const int g = prop.multiProcessorCount * per_sm;
                h->grid_pf = g < ntiles ? g : ntiles;
                // FLEETSTEP_PF_GRID=G (diagnostic, G >= 1) caps the persistent grid so that every CTA runs many tiles: the
                // steady state of the buffer rotation at test sizes
                const int cap = env_int("FLEETSTEP_PF_GRID", 0);
                if (cap > 0 && cap < h->grid_pf) h->grid_pf = cap;
                h->use_pf = 1;
            }
            cudaGetLastError();
        }
        if (force && strcmp(force, "pf") == 0 && !h->use_pf)
            return fail(h, FLEET_E_INVALID, "FLEETSTEP_KERNEL=pf requested but the configuration does not qualify (needs auto_reset, 8 <= N <= 256)");
    }
    h->grid = (E + p.B - 1) / p.B;
    CUDA_TRY(h, cudaFuncSetAttribute(pick_step(h), cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm));

    init_state_kernel<<<(unsigned)((EN > (size_t)E ? EN : (size_t)E) + 255) / 256, 256>>>(p);
    h->launches++;
    CUDA_TRY(h, cudaGetLastError());
    CUDA_TRY(h, cudaDeviceSynchronize());
    return FLEET_OK;
}

int fleet_reset(FleetHandle* h, const int32_t* start_idx_dev, const uint8_t* mask_dev, float* obs_dev, void* stream) {
    if (!h) return FLEET_E_INVALID;
    CUDA_TRY(h, cudaSetDevice(h->device));
    StepParams p = h->p;
    p.start_idx = start_idx_dev; p.mask = mask_dev; p.obs = obs_dev;
    pick_reset(h)<<<h->grid, kThreads, 0, (cudaStream_t)stream>>>(p);
    h->launches++;
    if (h->log_n) fleet_log_launch(h, p, 1, (cudaStream_t)stream);
    CUDA_TRY(h, cudaGetLastError());
    return FLEET_OK;
}

int fleet_step(FleetHandle* h, const float* actions_dev, float* obs_dev, float* reward_dev, uint8_t* done_dev,
               float* terminal_obs_dev, void* stream) {
    if (!h) return FLEET_E_INVALID;
    if (!actions_dev) return fail(h, FLEET_E_INVALID, "actions_dev is NULL");
    CUDA_TRY(h, cudaSetDevice(h->device));
    StepParams p = h->p;
    p.actions = actions_dev; p.obs = obs_dev; p.reward = reward_dev; p.done = done_dev; p.terminal_obs = terminal_obs_dev;
    if ((((uintptr_t)obs_dev) | ((uintptr_t)terminal_obs_dev)) & 15) { p.bulk_ok = 0; p.pf_bulk = 0; }   // bulk stores need 16-byte aligned rows
    cudaEvent_t* tev = nullptr;
    if (h->timing && !h->tev.empty()) tev = &h->tev[(size_t)(h->tcount % kTimingRing) * 3];
    if (tev) cudaEventRecord(tev[0], (cudaStream_t)stream);
    if (h->use_pf) pick_pf(h, p.charge_log != nullptr)<<<h->grid_pf, kPfThreads, h->smem_pf, (cudaStream_t)stream>>>(p);
    else pick_step(h)<<<h->grid, kThreads, h->smem_step, (cudaStream_t)stream>>>(p);
    h->launches++;
    if (tev) cudaEventRecord(tev[1], (cudaStream_t)stream);
    if (h->need_post) {   // daily degradation, then auto-reset, for the envs the step kernel put on the work list
        pick_post(h)<<<h->grid_post, h->post_threads, h->smem_post, (cudaStream_t)stream>>>(p);
        h->launches++;
    }
    if (tev) { cudaEventRecord(tev[2], (cudaStream_t)stream); h->tcount++; }
    if (h->log_n) { fleet_log_launch(h, p, 0, (cudaStream_t)stream); }
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail(h, FLEET_E_CUDA, std::string("fleet_step launch: ") + cudaGetErrorString(e));
    return FLEET_OK;
}

int fleet_step_host(FleetHandle* h, const float* actions_host, float* obs_host, float* reward_host, uint8_t* done_host,
                    float* terminal_obs_dev, void* stream) {
    if (!h) return FLEET_E_INVALID;
    if (!actions_host) return fail(h, FLEET_E_INVALID, "actions_host is NULL");
    CUDA_TRY(h, cudaSetDevice(h->device));
    cudaStream_t s = (cudaStream_t)stream;
    const size_t EN = (size_t)h->E * h->N, ED = (size_t)h->E * h->D;
    int rc;
    if (!h->h_actions_dev) {
        if ((rc = dev_alloc(h, &h->h_actions_dev, EN, false))) return rc;
        if ((rc = dev_alloc(h, &h->h_obs_dev, ED, false))) return rc;
        if ((rc = dev_alloc(h, &h->h_reward_dev, (size_t)h->E, false))) return rc;
        if ((rc = dev_alloc(h, &h->h_done_dev, (size_t)h->E, false))) return rc;
    }
    // Page-locked (pinned / registered) host buffers are device-accessible: the kernels then read the actions and write
    // the observations straight through PCIe (both directions at once, overlapped with the step itself) instead of
    // staging them with separate copies.  Pageable buffers take the staging path.  FLEETSTEP_HOST_ZEROCOPY=0 disables.
    auto mapped = [&](const void* host) -> void* {
        if (!host || !h->host_zerocopy) return nullptr;
        cudaPointerAttributes at;
        if (cudaPointerGetAttributes(&at, host) != cudaSuccess) { cudaGetLastError(); return nullptr; }
        return (at.type == cudaMemoryTypeHost) ? at.devicePointer : nullptr;
    };
    const float* a_dev = reinterpret_cast<const float*>(mapped(actions_host));
    float* o_dev = reinterpret_cast<float*>(mapped(obs_host));
    if (!a_dev) {
        CUDA_TRY(h, cudaMemcpyAsync(h->h_actions_dev, actions_host, EN * 4, cudaMemcpyHostToDevice, s));
        a_dev = h->h_actions_dev;
    }
    const bool obs_direct = (o_dev != nullptr);
    if (!obs_direct) o_dev = obs_host ? h->h_obs_dev : nullptr;
    if ((rc = fleet_step(h, a_dev, o_dev, h->h_reward_dev, h->h_done_dev, terminal_obs_dev, stream))) return rc;
    if (obs_host && !obs_direct) CUDA_TRY(h, cudaMemcpyAsync(obs_host, h->h_obs_dev, ED * 4, cudaMemcpyDeviceToHost, s));
    if (reward_host) CUDA_TRY(h, cudaMemcpyAsync(reward_host, h->h_reward_dev, (size_t)h->E * 4, cudaMemcpyDeviceToHost, s));
    if (done_host) CUDA_TRY(h, cudaMemcpyAsync(done_host, h->h_done_dev, (size_t)h->E, cudaMemcpyDeviceToHost, s));
    CUDA_TRY(h, cudaStreamSynchronize(s));
    return FLEET_OK;
}

int fleet_policy_actions(FleetHandle* h, int32_t policy, int32_t charging_hour, int32_t charging_minute,
                         int32_t max_hours, float* actions_dev, void* stream) {
    if (!h) return FLEET_E_INVALID;
    if (!actions_dev) return fail(h, FLEET_E_INVALID, "actions_dev is NULL");
    if (policy < FLEET_POLICY_UNCONTROLLED || policy > FLEET_POLICY_NIGHT) return fail(h, FLEET_E_INVALID, "unknown policy");
    CUDA_TRY(h, cudaSetDevice(h->device));
    int rc;
    if (policy == FLEET_POLICY_NIGHT && !h->pol_state[0]) {
        if ((rc = dev_alloc(h, &h->pol_state[0], (size_t)h->E))) return rc;
        if ((rc = dev_alloc(h, &h->pol_state[1], (size_t)h->E))) return rc;
    }
    const size_t cnt = (size_t)h->E * h->N;
    policy_kernel<<<(unsigned)((cnt + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
        h->p, policy, charging_hour, charging_minute, max_hours, h->tod, h->pol_state[h->pol_flip], h->pol_state[h->pol_flip ^ 1],
        actions_dev);
    if (policy == FLEET_POLICY_NIGHT) h->pol_flip ^= 1;
    h->launches++;
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail(h, FLEET_E_CUDA, std::string("fleet_policy_actions: ") + cudaGetErrorString(e));
    return FLEET_OK;
}

int fleet_policy_reset(FleetHandle* h, void* stream) {
    if (!h) return FLEET_E_INVALID;
    CUDA_TRY(h, cudaSetDevice(h->device));
    for (int k = 0; k < 2; k++)
        if (h->pol_state[k]) CUDA_TRY(h, cudaMemsetAsync(h->pol_state[k], 0, (size_t)h->E * sizeof(int2), (cudaStream_t)stream));
    return FLEET_OK;
}

int fleet_set_next_start(FleetHandle* h, const int32_t* next_start_idx_dev) {
    if (!h) return FLEET_E_INVALID;
    h->p.next_start = next_start_idx_dev;
    return FLEET_OK;
}

int fleet_field_info(const FleetHandle* h, int32_t field, int32_t* elem_bytes, int64_t* count) {
    if (!h || field < 0 || field >= FLEET_F__COUNT) return FLEET_E_INVALID;
    const int64_t EN = (int64_t)h->E * h->N, E = h->E;
    int eb = 8; int64_t cnt = EN;
    switch (field) {
        case FLEET_F_SOC: case FLEET_F_SOC_DEG: case FLEET_F_SOH: case FLEET_F_TARGET_SOC: case FLEET_F_FD_CYC:
        case FLEET_F_LIFE: case FLEET_F_LAST_DEG: case FLEET_F_CHARGE_LOG: eb = 8; cnt = EN; break;
        case FLEET_F_HOURS_LEFT: eb = 4; cnt = EN; break;
        case FLEET_F_RF_LEN: case FLEET_F_N_CYCLES: eb = 4; cnt = EN; break;
        case FLEET_F_TIME_IDX: case FLEET_F_FINISH_IDX: case FLEET_F_EP_COUNT: eb = 4; cnt = E; break;
        default: eb = 8; cnt = E; break;
    }
    if (elem_bytes) *elem_bytes = eb;
    if (count) *count = cnt;
    return FLEET_OK;
}

static const void* plain_field_ptr(const FleetHandle* h, int32_t field) {
    const StepParams& p = h->p;
    switch (field) {
        case FLEET_F_SOC: return p.soc;
        case FLEET_F_HOURS_LEFT: return p.hl;
        case FLEET_F_SOH: return p.soh;
        case FLEET_F_REWARD64: return p.env_f64 + (size_t)EF_REWARD64 * h->E;
        case FLEET_F_CASHFLOW: return p.env_f64 + (size_t)EF_CASHFLOW * h->E;
        case FLEET_F_RF_LEN: return p.rf_len;
        case FLEET_F_FD_CYC: return p.fd_cyc;
        case FLEET_F_LIFE: return p.life;
        case FLEET_F_EP_RETURN: return p.env_f64 + (size_t)EF_EP_RETURN * h->E;
        case FLEET_F_LAST_EP_RETURN: return p.env_f64 + (size_t)EF_LAST_EP_RETURN * h->E;
        case FLEET_F_N_CYCLES: return p.n_cycles;
        case FLEET_F_LAST_DEG: return p.last_deg;
        case FLEET_F_CHARGE_LOG: return p.charge_log;
        case FLEET_F_OVERLOAD: return p.env_f64 + (size_t)EF_OVERLOAD * h->E;
        case FLEET_F_SOC_VIOL: return p.env_f64 + (size_t)EF_SOC_VIOL * h->E;
        default: return nullptr;
    }
}

int fleet_get_state(FleetHandle* h, int32_t field, void* dst_dev, void* stream) {
    if (!h || !dst_dev) return FLEET_E_INVALID;
    int32_t eb; int64_t cnt;
    if (fleet_field_info(h, field, &eb, &cnt)) return fail(h, FLEET_E_INVALID, "unknown field");
    CUDA_TRY(h, cudaSetDevice(h->device));
    if (field == FLEET_F_CHARGE_LOG && !h->p.charge_log)
        return fail(h, FLEET_E_STATE, "FLEET_F_CHARGE_LOG is only kept after fleet_enable_charge_log(h, 1)");
    const void* src = plain_field_ptr(h, field);
    if (src) {
        CUDA_TRY(h, cudaMemcpyAsync(dst_dev, src, (size_t)cnt * eb, cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
    } else {
        gather_field_kernel<<<(unsigned)((cnt + 255) / 256), 256, 0, (cudaStream_t)stream>>>(h->p, field, dst_dev);
        h->launches++;
        CUDA_TRY(h, cudaGetLastError());
    }
    return FLEET_OK;
}

int fleet_set_state(FleetHandle* h, int32_t field, const void* src_dev, void* stream) {
    if (!h || !src_dev) return FLEET_E_INVALID;
    int32_t eb; int64_t cnt;
    if (fleet_field_info(h, field, &eb, &cnt)) return fail(h, FLEET_E_INVALID, "unknown field");
    CUDA_TRY(h, cudaSetDevice(h->device));
    if (field == FLEET_F_TARGET_SOC) {
        CUDA_TRY(h, cudaMemsetAsync(h->p.n_flips, 0, 4, (cudaStream_t)stream));
        scatter_target_kernel<<<(unsigned)((cnt + 255) / 256), 256, 0, (cudaStream_t)stream>>>(h->p, (const double*)src_dev);
        h->launches++;
        CUDA_TRY(h, cudaGetLastError());
        return FLEET_OK;
    }
    void* dst = const_cast<void*>(plain_field_ptr(h, field));
    if (!dst) return fail(h, FLEET_E_INVALID, "field is not writable");
    CUDA_TRY(h, cudaMemcpyAsync(dst, src_dev, (size_t)cnt * eb, cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
    return FLEET_OK;
}

int fleet_get_stats(FleetHandle* h, double* dst_dev, void* stream) {
    if (!h || !dst_dev) return FLEET_E_INVALID;
    CUDA_TRY(h, cudaSetDevice(h->device));
    reduce_stats_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(h->p.stats, dst_dev, h->p.price_mult);
    h->launches++;
    CUDA_TRY(h, cudaGetLastError());
    return FLEET_OK;
}

int fleet_reset_stats(FleetHandle* h, void* stream) {
    if (!h) return FLEET_E_INVALID;
    CUDA_TRY(h, cudaSetDevice(h->device));
    CUDA_TRY(h, cudaMemsetAsync(h->p.stats, 0, sizeof(double) * kStatStripes * FLEET_S__COUNT, (cudaStream_t)stream));
    return FLEET_OK;
}

int fleet_check_errors(FleetHandle* h, uint32_t* flags_host, void* stream) {
    if (!h) return FLEET_E_INVALID;
    CUDA_TRY(h, cudaSetDevice(h->device));
    uint32_t f = 0;
    CUDA_TRY(h, cudaMemcpyAsync(&f, h->p.err_flags, 4, cudaMemcpyDeviceToHost, (cudaStream_t)stream));
    CUDA_TRY(h, cudaStreamSynchronize((cudaStream_t)stream));
    CUDA_TRY(h, cudaMemsetAsync(h->p.err_flags, 0, 4, (cudaStream_t)stream));
    if (flags_host) *flags_host = f;
    if (f) {
        std::string m = "device error flags:";
        if (f & 1u) m += " NaN action (reference: TypeError ev_charger.py:209)";
        if (f & 2u) m += " negative battery life (rainflow_sei_degradation.py:179-180)";
        if (f & 4u) m += " DoD > 5 (rainflow_sei_degradation.py:164-167)";
        if (f & 8u) m += " rainflow stack capacity exceeded (raise FleetConsts.rf_stack_depth)";
        return fail(h, FLEET_E_STATE, m);
    }
    return FLEET_OK;
}

}  // extern "C"
