/*
 * fleetstep.h — C ABI of libfleetstep: the B200-native FleetRL environment step.
 *
 * This is the drop-in boundary for ONE path of EnzoCording/FleetRL: FleetEnv.reset()/step()
 * (reference: fleetrl/fleet_env/fleet_environment.py:330-702 and the fleetrl/utils modules it calls),
 * batched over (env, EV) on one GPU.  Plain pointers and sizes only; no torch types.  Every entry point
 * cites the reference interface it replaces.  The Python host side (fleetrl_b200/) binds these with
 * ctypes; INTEGRATION.md shows the stub a reference maintainer would add.
 *
 * Conventions
 *   - every function returns 0 on success or a negative FLEET_E_* code; nothing throws across the ABI;
 *     fleet_last_error(h) returns a human-readable message for the last failure on that handle.
 *   - pointers suffixed _dev are device pointers on the handle's GPU; _host are host pointers.
 *   - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream).  Calls only enqueue work;
 *     they never synchronise unless stated.  Calls on one handle are not re-entrant.
 *   - the caller owns all I/O buffers; the library owns the handle, its HBM tables and the env state.
 */
#ifndef FLEETSTEP_H_
#define FLEETSTEP_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define FLEETSTEP_ABI_VERSION 2

enum {
    FLEET_OK = 0,
    FLEET_E_INVALID = -1,   /* bad argument / unsupported configuration (reference: AssertionError / TypeError) */
    FLEET_E_CUDA = -2,      /* CUDA runtime error (sticky; message in fleet_last_error)                            */
    FLEET_E_NOMEM = -3,     /* device allocation failed (message states the bytes that were needed)               */
    FLEET_E_STATE = -4      /* device-side error flag raised by a kernel (NaN action, negative battery life, ...) */
};

/* Degradation model selector (reference: fleet_environment.py:285-288). */
enum { FLEET_DEG_SEI = 0,        /* RainflowSeiDegradation, rainflow_sei_degradation.py:91-212            */
       FLEET_DEG_EMPIRICAL = 1   /* EmpiricalDegradation, empirical_degradation.py:29-99, wired as the     */
                                 /* reference intends (SURVEY B-1: env.sei_deg = env.emp_deg), daily call  */ };

/*
 * All scalar configuration of the path, i.e. the reference's EvConfig / ScoreConfig / TimeConfig /
 * LoadCalculation objects after FleetEnv.__init__ has applied its overrides
 * (fleet_env/config/; load_calculation.py:15-60; fleet_environment.py:129-211).
 */
typedef struct FleetConsts {
    int32_t abi_version;          /* must be FLEETSTEP_ABI_VERSION                                             */
    int32_t num_evs;              /* N = db.ID.max()+1                         fleet_environment.py:260         */
    int32_t table_len;            /* T = rows per vehicle in the schedule                                      */
    int32_t steps_per_hour;       /* int(1/dt)                                 fleet_environment.py:456         */
    int32_t episode_steps;        /* episode_length[h] * steps_per_hour        fleet_environment.py:355         */
    int32_t price_lookahead;      /* TimeConfig.price_lookahead (8)            time_config.py:12                */
    int32_t bl_pv_lookahead;      /* TimeConfig.bl_pv_lookahead (4)            time_config.py:13                */
    int32_t include_price;        /* must be 1 (reference KeyErrors otherwise, SURVEY B-10)                     */
    int32_t include_building;
    int32_t include_pv;
    int32_t aux;                  /* auxiliary observation block               observer_bl_pv.py:85-107         */
    int32_t normalize;            /* 1 = OracleNormalization, 0 = UnitNormalization                             */
    int32_t is_caretaker;         /* use_case == "ct": lunch-break target      fleet_environment.py:536-540     */
    int32_t calc_degradation;     /* calculate_degradation flag                fleet_environment.py:665         */
    int32_t deg_mode;             /* FLEET_DEG_*                                                                */
    int32_t carry_degradation_state; /* 1 = keep rainflow_length/fd_cyc/l across episodes like the reference    */
                                  /* object does (SURVEY B-3); 0 = re-initialise them at every reset            */
    int32_t auto_reset;           /* 1 = SB3 VecEnv semantics: a done env is reset inside fleet_step            */
    int32_t start_lo, start_hi;   /* inclusive start-index range used by the device RNG on auto-reset           */
                                  /* (time_picker/random_time_picker.py:25-31, eval_time_picker.py:33-39)       */
    /* Incremental rainflow (no reference counterpart; the reference keeps the whole soc_log, log_data_deg.py:14-15):  */
    int32_t rf_ring_rows;         /* rows of the per-env soc_deg history ring (rounded up to a power of two >= 4);    */
                                  /* 0 = default (16).  Pending rows are consumed at the daily evaluation, or when     */
                                  /* the ring is about to wrap                                                        */
    int32_t rf_stack_depth;       /* rainflow stack entries kept inline per vehicle, 0 = default (12); deeper stacks   */
                                  /* borrow an extension slot; beyond that error flag bit 3 is raised (never silent)  */
    int32_t reserved0;
    uint64_t seed;                /* keys the counter-based start-index RNG: (seed, env id, episode number)     */

    double dt;                    /* hours per step = minutes/60               time_config.py:24                */
    /* EvConfig (ev_config.py:6-18) */
    double init_battery_cap, obc_max_power, charging_eff, discharging_eff, def_soc, temperature;
    double target_soc, target_soc_lunch, min_laxity, fixed_markup, variable_multiplier, feed_in_deduction;
    /* LoadCalculation (load_calculation.py:15-60) */
    double evse_max_power, grid_connection, lc_batt_cap;
    /* ScoreConfig (score_config.py:11-24); price_multiplier already rescaled by fleet_environment.py:194 */
    double price_multiplier, fully_charged_reward, penalty_invalid_action, penalty_overcharging;
    double penalty_overloading, clip_overcharging;
    double init_soh;              /* fleet_environment.py:231                                                   */
    double soc_eps;               /* 0.005                                     fleet_environment.py:230         */
    /* OracleNormalization scales (oracle_normalization.py:34-54); ignored unless normalize == 1 */
    double max_time_left, min_price, max_price, min_tariff, max_tariff, max_building, max_pv;
} FleetConsts;

/*
 * The reference's pandas `db` (data_processing.py:21-118, shape_price_reward :373-416) flattened to dense
 * host arrays, vehicle-major like the stacked frame.  fleet_create() copies and re-lays them out in HBM
 * (DESIGN.md "HBM layout"); the caller may free them afterwards.  Series the configuration excludes are NULL.
 */
typedef struct FleetTables {
    const uint8_t* there;               /* [N][T]  db.There                         data_processing.py:130     */
    const double*  time_left;           /* [N][T]  db.time_left, hours              data_processing.py:206-215 */
    const double*  soc_on_return;       /* [N][T]  db.SOC_on_return                 data_processing.py:221-223 */
    const double*  delu;                /* [T]     spot price EUR/MWh               data_processing.py:261-295 */
    const double*  tariff;              /* [T]     feed-in tariff EUR/MWh           data_processing.py:297-318 */
    const double*  load;                /* [T]     building load kW or NULL         data_processing.py:320-344 */
    const double*  pv;                  /* [T]     PV kW or NULL                    data_processing.py:347-370 */
    const double*  price_reward_curve;  /* [T]                                      data_processing.py:387-400 */
    const double*  tariff_reward_curve; /* [T]                                      data_processing.py:402-414 */
    const double*  cal_sincos;          /* [T][6]  sin/cos of month/12, weekday/7, hour/24  observer_bl_pv.py:100-107 */
    const uint8_t* hour;                /* [T]     date.hour                                                   */
    const uint8_t* minute;              /* [T]     date.minute                                                 */
} FleetTables;

/* Per-vehicle / per-env state fields readable with fleet_get_state / writable with fleet_set_state. */
enum {
    FLEET_F_SOC = 0,         /* double [E][N]  Episode.soc                   episode.py:22                     */
    FLEET_F_HOURS_LEFT = 1,  /* float  [E][N]  Episode.hours_left            episode.py:29                     */
    FLEET_F_SOC_DEG = 2,     /* double [E][N]  Episode.soc_deg               episode.py:23                     */
    FLEET_F_SOH = 3,         /* double [E][N]  Episode.soh                   episode.py:28                     */
    FLEET_F_TARGET_SOC = 4,  /* double [E][N]  FleetEnv.target_soc           fleet_environment.py:263,613      *
                              *                 Only two values exist: the configured target, or 0.9 once the vehicle's
                              *                 SOH has fallen to <= 0.9.  fleet_set_state stores one flag per vehicle,
                              *                 set where the value is 0.9 (and the target is not), and recounts the
                              *                 flags; any other value reads back as the configured target.
                              *                 FleetStepHandle.set rejects such values.                               */
    FLEET_F_TIME_IDX = 5,    /* int32  [E]     index of Episode.time in the table                              */
    FLEET_F_FINISH_IDX = 6,  /* int32  [E]     index of Episode.finish_time                                    */
    FLEET_F_REWARD64 = 7,    /* double [E]     reward of the last step before the f32 cast                     */
    FLEET_F_CASHFLOW = 8,    /* double [E]     Episode.current_charging_expense of the last step               */
    FLEET_F_RF_LEN = 9,      /* int32  [E][N]  RainflowSeiDegradation.rainflow_length  rainflow_sei_degradation.py:57 */
    FLEET_F_FD_CYC = 10,     /* double [E][N]  RainflowSeiDegradation.fd_cyc           :60                     */
    FLEET_F_LIFE = 11,       /* double [E][N]  RainflowSeiDegradation.l                :34                     */
    FLEET_F_EP_RETURN = 12,  /* double [E]     Episode.cumulative_reward     fleet_environment.py:637          */
    FLEET_F_EP_COUNT = 13,   /* int32  [E]     episodes started on this env (keys the start RNG)               */
    FLEET_F_LAST_EP_RETURN = 14, /* double [E] return of the most recently finished episode (SB3 Monitor "r")  */
    FLEET_F_N_CYCLES = 15,   /* int32  [E][N]  len(rainflow_result) seen at the last daily evaluation          */
    FLEET_F_LAST_DEG = 16,   /* double [E][N]  degradation returned by the last daily evaluation               */
    FLEET_F_OVERLOAD = 17,   /* double [E]     grid overload kW of the last step  load_calculation.py:93       */
    FLEET_F_SOC_VIOL = 18,   /* double [E]     cum_soc_missing of the last step   fleet_environment.py:544,661 */
    FLEET_F_CHARGE_LOG = 19, /* double [E][N]  each vehicle's OWN energy of the last step (kWh into (+) / out of (-) its battery);
                              *                 only kept after fleet_enable_charge_log(h, 1).  The reference's charge_log entry
                              *                 (ev_charger.py:212) is charging_energy + discharging_energy, two locals that
                              *                 survive from car to car (:81-82), so a car's entry also carries the last
                              *                 opposite-sign car's energy: the log ring (fleet_enable_log) reproduces exactly
                              *                 that column, this field keeps the physical per-vehicle quantity            */
    FLEET_F__COUNT = 20
};

/* Episode statistics (sums over all envs of the handle since the last fleet_reset_stats); the columns of the
 * reference's DataLogger row (data_logger.py:55-68) reduced over envs and steps. */
enum {
    FLEET_S_EPISODES = 0,   /* finished episodes                               */
    FLEET_S_EP_RETURN = 1,  /* sum of finished-episode returns                 */
    FLEET_S_STEPS = 2,      /* env-steps executed                              */
    FLEET_S_REWARD = 3,     /* sum of rewards                                  */
    FLEET_S_CASHFLOW = 4,   /* sum of cashflow                                 */
    FLEET_S_PENALTY = 5,    /* sum of reward - cashflow*price_multiplier       fleet_environment.py:659 */
    FLEET_S_OVERLOAD_KW = 6,/* sum of grid overload kW                         fleet_environment.py:660 */
    FLEET_S_SOC_VIOL = 7,   /* sum of missing SOC at departure                 fleet_environment.py:661 */
    FLEET_S_N_VIOL = 8,     /* number of departures below target               */
    FLEET_S_DEGRADATION = 9,/* sum of SOH loss                                 */
    FLEET_S__COUNT = 10
};

typedef struct FleetHandle FleetHandle;

/* Version of the ABI this library was built with. */
int fleet_abi_version(void);

/*
 * Replaces FleetEnv.__init__ (fleet_environment.py:76-328) for E identical environments on GPU `device`.
 * `env_id_offset` is the global id of local env 0 (multi-GPU sharding: rank r passes r*E); it only keys the
 * start-index RNG so that trajectories do not depend on the number of GPUs.
 */
int fleet_create(const FleetConsts* consts, const FleetTables* tables_host, int32_t num_envs, int32_t device,
                 int64_t env_id_offset, FleetHandle** out);

/* Replaces FleetEnv.close (fleet_environment.py:704). Frees all device memory. */
int fleet_destroy(FleetHandle* h);

/* observation_space.shape[0] / action_space.shape[0] / num_envs  (fleet_environment.py:316-325, 854-949). */
int fleet_obs_dim(const FleetHandle* h);
int fleet_num_evs(const FleetHandle* h);
int fleet_num_envs(const FleetHandle* h);

/*
 * Replaces FleetEnv.reset (fleet_environment.py:330-434) for every env whose mask byte is non-zero
 * (mask_dev == NULL: all).  start_idx_dev[e] is the table index of the episode start, i.e. what
 * TimePicker.choose_time returns (utils/time_picker/); start_idx_dev == NULL draws it from the device RNG in
 * [start_lo, start_hi].  Writes the first observation of each reset env to obs_dev[e][0..D) (float32; other
 * rows untouched).  obs_dev may be NULL.
 */
int fleet_reset(FleetHandle* h, const int32_t* start_idx_dev, const uint8_t* mask_dev, float* obs_dev, void* stream);

/*
 * Replaces FleetEnv.step (fleet_environment.py:436-702) for all E envs.
 *   actions_dev  float32 [E][N] in [-1,1]                         (step's `actions`)
 *   obs_dev      float32 [E][D]  next observation                 (norm_next_obs, :652,702)
 *   reward_dev   float32 [E]                                      (reward, :702; float64 copy in FLEET_F_REWARD64)
 *   done_dev     uint8   [E]                                      (episode.done, :627-628)
 *   terminal_obs_dev float32 [E][D] or NULL: with auto_reset, rows of envs that finished receive the last
 *                observation of the finished episode (SB3 infos[i]["terminal_observation"]) while obs_dev
 *                receives the first observation of the next one.
 * No allocation, no host synchronisation.
 */
int fleet_step(FleetHandle* h, const float* actions_dev, float* obs_dev, float* reward_dev, uint8_t* done_dev,
               float* terminal_obs_dev, void* stream);

/* Same step with HOST buffers (pinned or pageable): copies actions up, steps, copies obs/reward/done back and
 * synchronises the stream.  This is the call an SB3-style NumPy caller makes; bench.py times it as "e2e".
 * Page-locked buffers are used in place: the kernels read the actions and write the observations through PCIe
 * themselves (both directions at once, overlapped with the step), pageable ones go through staging copies.
 * terminal_obs_dev (optional, DEVICE float32 [E][D]) receives the terminal rows of finished envs as in fleet_step;
 * the caller fetches only the rows it needs (finished envs are rare). */
int fleet_step_host(FleetHandle* h, const float* actions_host, float* obs_host, float* reward_host,
                    uint8_t* done_host, float* terminal_obs_dev, void* stream);

/* Start indices consumed by the next auto-resets instead of the RNG (parity runs inject them the way the
 * reference harness replaces env.time_picker, SURVEY App. C-4).  NULL restores the RNG. The array must stay
 * valid; entry e is used each time env e auto-resets. */
int fleet_set_next_start(FleetHandle* h, const int32_t* next_start_idx_dev);

/* Copy one state field (FLEET_F_*) device-to-device into / out of caller memory; backs env_method() helpers
 * (fleet_environment.py:741-799), tests and state_dict()/load_state_dict().  FLEET_F_SOC_DEG, FLEET_F_TIME_IDX,
 * FLEET_F_FINISH_IDX and FLEET_F_EP_COUNT are read-only; FLEET_F_TARGET_SOC stores, per vehicle, whether the value
 * is 0.9 (see the field). */
int fleet_get_state(FleetHandle* h, int32_t field, void* dst_dev, void* stream);
int fleet_set_state(FleetHandle* h, int32_t field, const void* src_dev, void* stream);
/* Element size in bytes and element count ([E][N] or [E]) of a field. */
int fleet_field_info(const FleetHandle* h, int32_t field, int32_t* elem_bytes, int64_t* count);

/* Episode statistics: dst_dev receives FLEET_S__COUNT doubles (this GPU's partial sums — the vector the host
 * all-reduces over NCCL).  fleet_reset_stats zeroes them. */
int fleet_get_stats(FleetHandle* h, double* dst_dev, void* stream);
int fleet_reset_stats(FleetHandle* h, void* stream);

/* Device error flags raised by kernels since the last call (bit 0: NaN action — the reference raises TypeError
 * at ev_charger.py:209; bit 1: negative battery life, rainflow_sei_degradation.py:179-180; bit 2: DoD > 5,
 * :164-167; bit 3: a vehicle's rainflow stack outgrew rf_stack_depth plus its extension slot — recreate the handle
 * with a larger rf_stack_depth).  Synchronises the stream.  Returns FLEET_E_STATE if any bit is set. */
int fleet_check_errors(FleetHandle* h, uint32_t* flags_host, void* stream);

/* Number of kernel launches issued through this handle so far (bench.py reports it as gpu_launches). */
int64_t fleet_launch_count(const FleetHandle* h);

/* Optional per-kernel timing for measurement (bench.py's roofline line): when enabled, fleet_step brackets the step
 * kernel and the post kernel with CUDA events on the caller's stream; fleet_get_timing synchronises them and returns
 * the summed durations (ms) over the last <= 1024 steps since fleet_set_timing.  No reference counterpart. */
/* Rule-based baseline policies of the reference's benchmarking scripts, evaluated on the device for every env at its
 * current time: actions_dev float32 [E][N] is what those scripts pass to VecEnv.step (as float32).
 *   FLEET_POLICY_UNCONTROLLED  a = 1                                       benchmarking/uncontrolled_charging.py:51-54
 *   FLEET_POLICY_DISTRIBUTED   a = clip(get_dist_factor(), 0, 1)           benchmarking/distributed_charging.py:50-54,
 *                                                                          fleet_environment.py:782-799
 *   FLEET_POLICY_NIGHT         charging window opening at (charging_hour, charging_minute), open for more than max_hours
 *                              hours; caretaker fleets follow the distributed rule from 11:00 to 14:59
 *                              benchmarking/night_charging.py:81-98 (charging_hour/minute/max_hours as computed at :53-71)
 * The night policy keeps {window open, opening index} per env inside the handle; fleet_policy_reset clears it. */
enum { FLEET_POLICY_UNCONTROLLED = 0, FLEET_POLICY_DISTRIBUTED = 1, FLEET_POLICY_NIGHT = 2 };
int fleet_policy_actions(FleetHandle* h, int32_t policy, int32_t charging_hour, int32_t charging_minute, int32_t max_hours,
                         float* actions_dev, void* stream);
int fleet_policy_reset(FleetHandle* h, void* stream);

/* Keep EvCharger.charge's per-vehicle charge_log (ev_charger.py:80,212; the "Charging energy" column of
 * DataLogger.log_data) of every step in device memory, readable as FLEET_F_CHARGE_LOG.  Off by default: it costs
 * 8 bytes of HBM writes per EV-step. */
int fleet_enable_charge_log(FleetHandle* h, int32_t enable);

/* Device-side DataLogger (utils/data_logger/data_logger.py:21-68, fed at fleet_environment.py:420-432 and :679-690) for a
 * few selected envs of an evaluation run: after fleet_enable_log every fleet_reset / fleet_step appends the reference's log
 * row of those envs to a ring of rows_per_env rows per env in HBM (a finishing step is not logged, the reset that follows
 * is).  A row is row_doubles float64 values: {ep_count, time index, Reward, Cashflow, Penalties, Grid overloading,
 * SOC violation, kind (1 = reset row, 2 = step with the daily degradation, 0 = other step)}, Action[N], Degradation[N],
 * Charging energy[N] (with EvCharger's carry-over of the last opposite-sign car, ev_charger.py:81-82,212), SOH[N],
 * Observation[D].  fleet_read_log copies the rings ([n_envs][rows_per_env][row_doubles]) and the per-env row counts
 * (ring position = count % rows_per_env) to the host and synchronises. */
int fleet_enable_log(FleetHandle* h, const int32_t* env_ids_host, int32_t n_envs, int32_t rows_per_env);
int fleet_log_layout(const FleetHandle* h, int32_t* n_envs, int32_t* rows_per_env, int32_t* row_doubles);
int fleet_read_log(FleetHandle* h, double* rows_host, int64_t* counts_host, void* stream);

/* Checkpoint / resume: the complete env state of the handle (time indices, SOC, SOH, history ring, rainflow stacks,
 * degradation members, statistics) as one opaque blob of fleet_state_bytes bytes in host memory.  fleet_import_state only
 * accepts a blob exported from a handle created with the same configuration and num_envs.  Both synchronise.
 * Backs FleetVecEnv.state_dict() / load_state_dict().  The night policy's window state (fleet_policy_actions) belongs
 * to the caller's evaluation loop, not to the envs: it is not in the blob (fleet_policy_reset clears it). */
int64_t fleet_state_bytes(FleetHandle* h);
int fleet_export_state(FleetHandle* h, void* dst_host, void* stream);
int fleet_import_state(FleetHandle* h, const void* src_host, void* stream);

/* Diagnostic: the SEI cycle-stress function the post kernel uses (rainflow_sei_degradation.py:68-79 at reference
 * temperature: 1 / (kd1 * dod**kd2 + kd3) * exp(k_sigma * (mean - sigma_ref))) over device arrays of n effective DoDs and
 * mean SOCs; backs the accuracy test of its series evaluation. */
int fleet_debug_stress(const double* eff_dev, const double* mean_dev, double* out_dev, int32_t n, void* stream);

const char* fleet_step_kernel_name(const FleetHandle* h);   /* which step kernel fleet_create selected */

/* Launch geometry fleet_create chose: CTAs of the step kernel, tiles it covers (envs_per_tile envs each; the persistent
 * pf kernel loops over them with a stride of step_grid, the generic kernel runs one CTA per tile) and CTAs of the post
 * kernel (0 when no post kernel runs).  Two diagnostic environment variables, read by fleet_create, cap the grids
 * below what the occupancy query gives, so that each CTA iterates over many tiles / work items at test sizes:
 * FLEETSTEP_PF_GRID (pf step kernel) and FLEETSTEP_POST_GRID (post kernel); unset or <= 0 means no cap. */
int fleet_launch_geometry(const FleetHandle* h, int32_t* step_grid, int32_t* step_tiles, int32_t* envs_per_tile,
                          int32_t* post_grid);
int fleet_set_timing(FleetHandle* h, int32_t enable);
int fleet_get_timing(FleetHandle* h, double* step_kernel_ms, double* post_kernel_ms, int64_t* steps);

/* Bytes of device memory owned by the handle. */
int64_t fleet_device_bytes(const FleetHandle* h);

const char* fleet_last_error(const FleetHandle* h);

/*
 * FleetNorm — SB3 2.3.2's VecNormalize (stable_baselines3/common/vec_env/vec_normalize.py) with its two RunningMeanStd
 * (common/running_mean_std.py) on the device, for any [E][D] float32 observation batch.  Independent of FleetHandle:
 * like SB3, the statistics live apart from the env and are saved separately.  Same arithmetic and defaults: float64
 * statistics, count 1e-4 / mean 0 / var 1 at creation, obs -> float32(clip((x - mean) / sqrt(var + eps), +-clip_obs)),
 * reward -> clip(reward / sqrt(ret_var + eps), +-clip_reward) as float32.  A training step is two calls:
 *   fleet_norm_moments  batch moments into a caller-owned float64 vector of fleet_norm_moments_len entries;
 *   (multi-GPU: all-reduce that vector with SUM: every rank holds the same statistics, so the sums add)
 *   fleet_norm_apply    merges them into the statistics and writes the normalised outputs.
 * One kernel launch each, no host synchronisation.  The batch moments are computed in float64 where SB3 reduces
 * in the observation dtype (float32): the statistics differ from SB3's at float32 rounding level.
 */
typedef struct FleetNorm FleetNorm;

/* Replaces VecNormalize.__init__ (vec_normalize.py) for num_envs envs with obs_dim observations on GPU `device`.
 * FLEET_E_INVALID for sizes < 1, clip_obs or clip_reward <= 0, gamma outside [0, 1], epsilon < 0.  *out is set
 * even on failure (fleet_norm_last_error); the caller destroys it. */
int fleet_norm_create(int32_t num_envs, int32_t obs_dim, int32_t device, double clip_obs, double clip_reward, double gamma,
                      double epsilon, FleetNorm** out);
int fleet_norm_destroy(FleetNorm* n);

/* The attributes VecNormalize.training / norm_obs / norm_reward (vec_normalize.py).  Initially all 1. */
int fleet_norm_set_flags(FleetNorm* n, int32_t training, int32_t norm_obs, int32_t norm_reward);

/* Length 2*obs_dim+4 of the moments vector: {obs n, sum(x-K)[D], sum((x-K)^2)[D], ret n, sum(r-Kr), sum((r-Kr)^2)}
 * with K, Kr the current running means and r = returns*gamma + reward the new returns. */
int fleet_norm_moments_len(const FleetNorm* n);

/* The data half of RunningMeanStd.update (running_mean_std.py) for obs_rms (VecNormalize.step_wait's
 * obs_rms.update(obs), vec_normalize.py; reset's _update_obs) and, when reward_dev is given, for ret_rms
 * (_update_reward, :236-239).  obs_dev float32 [E][D], reward_dev float32 [E] or NULL.  The obs part is computed only when
 * training and norm_obs, the returns part only when training; a part not computed has n = 0.  No side effects: writes
 * moments_dev only.  Deterministic: independent of the grid and of the SM count. */
int fleet_norm_moments(FleetNorm* n, const float* obs_dev, const float* reward_dev, double* moments_dev, void* stream);

/* The rest of VecNormalize.step_wait (vec_normalize.py) / reset and normalize_obs /
 * normalize_reward  on `rows` rows:
 *   moments_dev (ignored unless training): merged into the statistics with update_from_moments (running_mean_std.py);
 *               with rewards, also returns = returns*gamma + reward.  NULL: normalise with the current statistics only.
 *   obs_dev -> obs_out_dev        float32 [rows][D], normalised when norm_obs, else copied; obs_dev stays intact
 *   reward_dev -> reward_out_dev  float32 [rows], normalised when norm_reward, else copied
 *   done_dev uint8 [E]: returns[done] = 0, and terminal_obs_dev rows of finished envs are normalised into
 *               terminal_obs_out_dev (other rows untouched), with the statistics after this call's update.
 * Any pointer pair may be NULL.  A statistics update or done_dev requires rows == E.  Views need not be 16-byte aligned. */
int fleet_norm_apply(FleetNorm* n, const double* moments_dev, int64_t rows, const float* obs_dev, float* obs_out_dev,
                     const float* reward_dev, float* reward_out_dev, const uint8_t* done_dev, const float* terminal_obs_dev,
                     float* terminal_obs_out_dev, void* stream);

/* self.returns = np.zeros(self.num_envs) of VecNormalize.reset (vec_normalize.py). */
int fleet_norm_reset_returns(FleetNorm* n, void* stream);

/* obs_rms.mean/var/count [D]/[D]/1, ret_rms.mean/var/count 1/1/1 and returns [E] as float64 HOST arrays (the attributes
 * VecNormalize.save pickles, vec_normalize.py).  A NULL pointer skips that part.  Both synchronise. */
int fleet_norm_get_state(FleetNorm* n, double* obs_mean, double* obs_var, double* obs_count, double* ret_mean,
                         double* ret_var, double* ret_count, double* returns, void* stream);
int fleet_norm_set_state(FleetNorm* n, const double* obs_mean, const double* obs_var, const double* obs_count,
                         const double* ret_mean, const double* ret_var, const double* ret_count, const double* returns,
                         void* stream);

const char* fleet_norm_last_error(const FleetNorm* n);

/*
 * FleetRollout — SB3 2.3.2's RolloutBuffer (stable_baselines3/common/buffers.py), the transition storage of PPO, on the
 * device.  Stateless: the caller owns the storage, [T][E]... float32 arrays described by a FleetRolloutBuf
 * (T = buffer_size, E = num_envs), laid out like RolloutBuffer's attributes before swap_and_flatten.  One kernel launch per
 * call, no host synchronisation, no atomics (deterministic).  Offsets are 64-bit.  FLEET_E_INVALID for sizes < 1 or a
 * NULL storage pointer; fleet_rollout_last_error() returns the message of the calling thread's last failure.
 */
typedef struct FleetRolloutBuf {
    int32_t buffer_size, num_envs, obs_dim, action_dim;
    float* observations;      /* [T][E][obs_dim]     RolloutBuffer.observations                        */
    float* actions;           /* [T][E][action_dim]  .actions (unclipped, as the policy sampled them)  */
    float* rewards;           /* [T][E]              .rewards                                          */
    float* episode_starts;    /* [T][E]              .episode_starts, 0.0f / 1.0f                      */
    float* values;            /* [T][E]              .values                                           */
    float* log_probs;         /* [T][E]              .log_probs                                        */
    float* advantages;        /* [T][E]              .advantages                                       */
    float* returns;           /* [T][E]              .returns                                          */
} FleetRolloutBuf;

/* RolloutBuffer.add (buffers.py) into slot `slot` (its self.pos): obs float32 [E][obs_dim], action [E][action_dim],
 * reward / value / log_prob float32 [E], episode_start uint8 [E] (the env's done dtype) stored as 0.0f / 1.0f.  Any source
 * may be NULL, which leaves that field of the slot untouched (an on-device collector writes the reward after the env step
 * that overwrites the observation).  FLEET_E_INVALID for a slot outside [0, buffer_size).  Views need not be aligned. */
int fleet_rollout_add(const FleetRolloutBuf* b, int32_t slot, const float* obs, const float* action, const float* reward,
                      const uint8_t* episode_start, const float* value, const float* log_prob, void* stream);

/* RolloutBuffer.compute_returns_and_advantage (buffers.py) over the whole buffer: last_values float32 [E], dones uint8 [E]
 * (both required).  SB3's float32 arithmetic in SB3's order, bit for bit, with g = float32(gamma) and
 * gl = float32(gamma * gae_lambda):
 *   delta = (rewards[t] + (g * next_values) * nnt) - values[t];   last_gae_lam = delta + (gl * nnt) * last_gae_lam
 *   advantages[t] = last_gae_lam;   returns[t] = last_gae_lam + values[t]
 * nnt = 1 - dones at t = T-1, else 1 - episode_starts[t+1].  FLEET_E_INVALID for gamma or gae_lambda outside [0, 1]. */
int fleet_rollout_gae(const FleetRolloutBuf* b, double gamma, double gae_lambda, const float* last_values,
                      const uint8_t* dones, void* stream);

/* RolloutBuffer._get_samples (buffers.py) for `count` flat sample indices (int64, device).  SB3 numbers the samples after
 * swap_and_flatten, env-major: flat k is env k / T, step k % T; this reads row (k % T) * E + k / T of the [T][E] storage,
 * so the one-off flattened copy SB3 makes in get() is not needed.  Writes obs_out [count][obs_dim],
 * actions_out [count][action_dim] and values / log_probs / advantages / returns _out [count] (all required).  An index
 * outside [0, T*E) writes nothing to its output row.  FLEET_E_INVALID for count < 0. */
int fleet_rollout_gather(const FleetRolloutBuf* b, const int64_t* flat_idx_dev, int64_t count, float* obs_out,
                         float* actions_out, float* values_out, float* log_probs_out, float* advantages_out,
                         float* returns_out, void* stream);

/* Message of the calling thread's last failing fleet_rollout_* call. */
const char* fleet_rollout_last_error(void);

/*
 * FleetPpo — the per-minibatch loss of SB3 2.3.2's PPO.train (stable_baselines3/ppo/ppo.py) for a diagonal Gaussian
 * policy (common/distributions.py, DiagGaussianDistribution), forward and backward.  Stateless: the caller owns every
 * array, including a workspace of fleet_ppo_workspace_bytes(B, N) bytes, 256-byte aligned and zero-filled before its
 * first use (each call leaves it reusable).  No call synchronises the host, no kernel uses floating-point atomics, and
 * every output is bit-identical from call to call: reductions run in float64 over fixed chunks of rows, combined in a
 * fixed order by the last CTA of each launch.  Offsets are 64-bit.  FLEET_E_INVALID for bad sizes, NULL pointers,
 * clip_range <= 0 or a workspace that is too small; fleet_ppo_last_error() returns the calling thread's message.
 * All arrays are float32 on the device.
 */
typedef struct FleetPpoBatch {
    int64_t batch_size;          /* B                                                                          */
    int32_t action_dim;          /* N                                                                          */
    int32_t reserved;
    const float* mean;           /* [B][N]  mean_actions of the policy                                          */
    const float* log_std;        /* [N]     the policy's state-independent log_std                              */
    const float* actions;        /* [B][N]  RolloutBufferSamples.actions                                        */
    const float* values;         /* [B]     the value head's output                                            */
    const float* old_log_prob;   /* [B]     .old_log_prob                                                       */
    const float* old_values;     /* [B]     .old_values (read only when clip_range_vf >= 0)                     */
    const float* advantages;     /* [B]     .advantages                                                         */
    const float* returns;        /* [B]     .returns                                                            */
} FleetPpoBatch;

typedef struct FleetPpoParams {
    double clip_range;           /* > 0                                                                         */
    double clip_range_vf;        /* < 0: None                                                                   */
    double ent_coef, vf_coef;
    int32_t normalize_advantage; /* applied only when B > 1, as SB3 does                                        */
    int32_t reserved;
} FleetPpoParams;

/* Bytes of workspace fleet_ppo_loss and fleet_ppo_loss_backward need for B rows of N actions (0 for sizes < 1). */
int64_t fleet_ppo_workspace_bytes(int64_t batch_size, int32_t action_dim);

/* DiagGaussianDistribution.log_prob (distributions.py) over Normal(mean, ones_like(mean) * exp(log_std)) (torch's
 * Normal.log_prob): lp[i] = sum_n ( -(a - mu)^2 / (2 sigma^2) - log(sigma) - log(sqrt(2 pi)) ) with sigma = exp(log_std),
 * each term in float32 in torch's order, the sum over n in float64 in a fixed order, rounded once.  Reads mean, log_std
 * and actions of the batch; writes log_prob_out [B].  fleet_ppo_loss computes the same bits for the same inputs. */
int fleet_ppo_log_prob(const FleetPpoBatch* b, float* log_prob_out, void* stream);

/* The loss of one minibatch of PPO.train (ppo.py), in two launches:
 *   A = advantages, normalised when normalize_advantage and B > 1: (A - m) / (s + 1e-8) with the mean m and the
 *       unbiased std s reduced in float64 and rounded to float32;
 *   ratio = exp(log_prob - old_log_prob);  policy_loss = -mean(min(A * ratio, A * clamp(ratio, 1 - eps, 1 + eps)));
 *   values_pred = values, or old_values + clamp(values - old_values, -c, c) when clip_range_vf = c >= 0;
 *   value_loss = mean((returns - values_pred)^2);  entropy_loss = -mean(entropy) = -sum_n (0.5 + 0.5 log 2pi + log sigma_n);
 *   loss = policy_loss + ent_coef * entropy_loss + vf_coef * value_loss  -> *loss_out (float32, device).
 * Adds this minibatch's policy_loss, value_loss, entropy_loss, clip_fraction (mean of |ratio - 1| > eps) and approx_kl
 * (mean((ratio - 1) - log_ratio)) to stats_acc[0..4] (float64, device).  Writes sample_coef [2][B]: d loss / d log_prob
 * and d loss / d values of every row, which fleet_ppo_loss_backward reads. */
int fleet_ppo_loss(const FleetPpoBatch* b, const FleetPpoParams* p, float* loss_out, double* stats_acc,
                   float* sample_coef, void* workspace, int64_t workspace_bytes, void* stream);

/* The gradient of fleet_ppo_loss as torch autograd gives it on SB3's composition (clamp passes the gradient on its
 * closed interval, minimum splits a tie in half, the normalised advantage carries none), in one launch.  grad_loss is
 * read from device memory; with g_i = grad_loss * d loss / d log_prob_i:
 *   grad_mean [B][N] = g_i (a - mu) / sigma^2;   grad_values [B] = grad_loss * d loss / d values_i;
 *   grad_log_std [N] = sum_i g_i ((a - mu)^2 / sigma^2 - 1) - grad_loss * ent_coef  (float64 column sums).
 * b and p must be those of the fleet_ppo_loss call that wrote sample_coef. */
int fleet_ppo_loss_backward(const FleetPpoBatch* b, const FleetPpoParams* p, const float* grad_loss,
                            const float* sample_coef, float* grad_mean, float* grad_log_std, float* grad_values,
                            void* workspace, int64_t workspace_bytes, void* stream);

/* Message of the calling thread's last failing fleet_ppo_* call. */
const char* fleet_ppo_last_error(void);

#ifdef __cplusplus
}
#endif
#endif /* FLEETSTEP_H_ */
