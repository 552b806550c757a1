/*
 * glgym.h -- C-ABI of libglgym.so: the B200-native batched GreenLight env-step path.
 *
 * Drop-in boundary for two reference interfaces (see INTEGRATION.md for the binding stubs):
 *   (1) the pybind11 class `GreenLight(nx,nu,nd,np,dt).evalF(x,u,d,p) -> x_next`
 *       gl_gym/environments/models/greenlight_model.cpp:31,96-120,130-136    -> glg_evalf_batch()
 *   (2) the env-step path `TomatoEnv.reset()/step()/step_raw_control()` as consumed through SB3's VecEnv
 *       gl_gym/environments/tomato_env.py:115-173,231-270, gl_gym/RL/utils.py:44-69 -> glg_reset()/glg_step*()
 *
 * Conventions: every function returns 0 on success or a negative glg_status; no C++ types or exceptions cross the
 * boundary; `stream` is a cudaStream_t passed as void* (NULL = default stream); functions taking a stream only
 * enqueue work (no hidden synchronisation) unless documented otherwise; pointers named *_dev are device pointers
 * on the handle's device, *_host are host pointers.  Inputs are owned by the caller; state and outputs are owned
 * by the handle for its lifetime.  A handle is bound to one device and is not thread-safe (like the reference
 * object it replaces, greenlight_model.cpp:22-24).  There is no CPU fallback: without a CUDA device
 * glg_create() fails with GLG_ERR_CUDA.
 */
#ifndef GLGYM_H
#define GLGYM_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GLG_NX 28
#define GLG_NU 6
#define GLG_ND 10
#define GLG_NP 208
#define GLG_NINFO 11
#define GLG_NSTATS 16
#define GLG_NNOISE 34

typedef enum glg_status {
    GLG_OK = 0,
    GLG_ERR_ARG = -1,   /* invalid argument */
    GLG_ERR_CUDA = -2,  /* CUDA runtime error; see glg_last_error() */
    GLG_ERR_STATE = -3, /* call order (e.g. step before params/weather were set) */
    GLG_ERR_ALLOC = -4
} glg_status;

typedef struct glg_handle glg_handle;

/* Mirrors the constructor arguments of TomatoEnv / GreenLightEnv (base_env.py:41-88, tomato_env.py:27-66,
 * configs/envs/TomatoEnv.yml) plus the batch/GPU knobs. */
typedef struct glg_config {
    int32_t num_envs;        /* B: envs owned by this handle (this GPU's shard) */
    int32_t device;          /* CUDA device ordinal */
    double dt;               /* control interval [s] (900) */
    int32_t n_sub;           /* RK4 substeps per control interval (default 600, SURVEY B.6) */
    int32_t N;               /* int(season_length*86400/dt): index of the last step (base_env.py:88) */
    int32_t Np;              /* int(pred_horizon*86400/dt): forecast rows in the observation (base_env.py:80) */
    int32_t precision;       /* 0 = fp64 parity mode ; 1 = fp32 RHS / fp64 state (throughput mode) */
    int32_t auto_reset;      /* 1: SB3 VecEnv semantics (terminal obs saved, env re-initialised in the same launch) */
    double u_min[GLG_NU];    /* base_env.py:72 */
    double u_max[GLG_NU];    /* base_env.py:73 */
    double delta_u_max;      /* float32(0.1) widened to double (base_env.py:74) */
    double con_low[3];       /* co2_min [ppm], temp_min, rh_min  (tomato_env.py:51-55) */
    double con_high[3];      /* co2_max, temp_max, rh_max        (tomato_env.py:57-61) */
    double elec_price, heating_price, co2_price, fruit_price, dmfm; /* rewards.py:46-94 */
    double fixed_costs;      /* rewards.py:69-70,154 (reported in info only) */
    double uncertainty_scale;/* tomato_env.py:34,118 ; 0 = nominal parameters */
    uint64_t seed;           /* Philox key */
    int64_t env_id_offset;   /* global index of local env 0 (multi-GPU sharding; RNG streams follow the global id) */
    int32_t role_warps;      /* kernel variant: 0 = auto, 1 = one thread per env (kernel A), 2 / 3 = warp-specialised kernel C (4 owner +
                              * 12 flux-unit warps per 32 envs) compiled for one CTA per SM (latency: small batches) / two (throughput) */
    int32_t role_lanes;      /* 0 = auto (32), or 1..32: kernel C's envs-per-CTA (tuning / tests) */
    int32_t integrator;      /* 0 = fixed-step RK4, n_sub equal substeps (the parity contract);
                                1 = graded RK4: the first 12 nominal substeps of every control interval are split in 16, 8,
                                    4 x4, 2 x6 (the controls just changed: fast transients) and any nominal substep is split
                                    further while the top-compartment / cover stiffness estimate asks for it (DESIGN.md
                                    "Integrator contract"); meant for n_sub = 260: 300 RK4 steps per interval. */
    int32_t reserved2;
    /* Observation stack (tomato_env.py:77-96, configs/envs/TomatoEnv.yml:26-33): ordered list of module ids, terminated by 0;
     * an empty list (obs_modules[0] == 0) is the default stack {2,3,4,5,6,7}.  ids (observations.py:35-182):
     *   1 StateObservations (27; `np.random.rand` in the reference -> Philox uniforms here), 2 IndoorClimateObservations (4),
     *   3 BasicCropObservations (3), 4 ControlObservations (6), 5 WeatherObservations (5), 6 TimeObservations (5),
     *   7 WeatherForecastObservations (5 Np).  A module may appear at most once; the row must have at least 3 entries (the
     *   reward reads obs[0:3], rewards.py:191-198). */
    int32_t obs_modules[8];
} glg_config;

/* Fills *cfg with the defaults of configs/envs/TomatoEnv.yml (dt 900, N 5760, Np 48, n_sub 600, ...). */
void glg_default_config(glg_config *cfg);

int glg_create(const glg_config *cfg, glg_handle **out);
void glg_destroy(glg_handle *h);
/* Last error text of the handle (or of the failed glg_create when h is NULL). Never NULL. */
const char *glg_last_error(const glg_handle *h);

/* New key for the handle's Philox streams (base_env.py:166-170 set_seed); takes effect with the next launch. */
int glg_set_seed(glg_handle *h, uint64_t seed);
/* Nominal parameter table, 208 doubles (float32-rounded values as produced by init_default_params,
 * parameters.py:4-261).  Derives the parameter-only constants on the host and selects the kernel variant. */
int glg_set_params(glg_handle *h, const double *p_host);
/* Weather bank: n_tables tables of `rows` rows x 10 columns (utils.py:75-84), row-major doubles, plus the start
 * day of each table (day_of_year after reset, tomato_env.py:246).  rows >= N + Np + 1. */
int glg_set_weather(glg_handle *h, const double *tables_host, int32_t n_tables, int32_t rows, const double *start_day_host);
/* Tables a reset may pick (uniformly, Philox); default = all tables.  Mirrors rng.choice(train_days), tomato_env.py:236-244 */
int glg_set_reset_tables(glg_handle *h, const int32_t *table_ids_host, int32_t n);

/* reset(): tomato_env.py:231-270.  mask_dev: uint8[B] (1 = reset) or NULL for all.  table_ids_dev: int32[B]
 * explicit table per env or NULL to draw from the reset list.  Writes obs. */
int glg_reset(glg_handle *h, const uint8_t *mask_dev, const int32_t *table_ids_dev, void *stream);

/* step(): tomato_env.py:115-146, fused in one kernel: action->control, parametric noise, weather row fetch,
 * n_sub RK4 substeps, time update, observation, reward, info, termination, auto-reset.
 *   actions_dev : float32 [B][6] in [-1,1]
 *   noise_dev   : NULL (device Philox when uncertainty_scale > 0) or double [B][34] external multipliers n_i
 *                 (p_i <- f32(p_i + n_i p_i)), for bit-parity with a host RNG (noise.py:16-19) */
int glg_step(glg_handle *h, const float *actions_dev, const double *noise_dev, void *stream);
/* step_raw_control(): tomato_env.py:148-173.  controls_dev: double [B][6], used as-is (no clip / rate limit). */
int glg_step_raw_control(glg_handle *h, const double *controls_dev, const double *noise_dev, void *stream);

/* Rule-based controller in the loop (SURVEY 8f-1): RuleBasedController.predict, environments/baseline.py:68-227, evaluated
 * on the device from each env's state, the weather row of its current timestep and its clock, then stepped like
 * step_raw_control -- replaces the host loop of experiments/evaluate_baseline.py:21-23.
 *   settings29 : host double[29] in the order of configs/agents/rule_based.yml (lamps_on, lamps_off, lamps_day_start,
 *                lamps_day_stop, lamps_off_sun, lamp_rad_sum_limit, temp_setpoint_day, temp_setpoint_night,
 *                heat_correction, heat_deadzone, co2_day, vent_heat_Pband, rh_max, mech_dehumid_Pband, vent_rh_Pband,
 *                t_vent_off, vent_cold_Pband, thScrSpDay, thScrSpNight, thScrPband, thScrDeadZone, thScrRh, thScrRhPband,
 *                lampExtraHeat, blScrExtraRh, rhMax, tHeatBand, co2Band, useBlScr); NULL = the shipped YAML values. */
int glg_set_rule_controller(glg_handle *h, const double *settings29);
int glg_step_rule_based(glg_handle *h, const double *noise_dev, void *stream);
/* Known-answer entry for the controller alone: x_dev double [n][28], d_dev double [n][10], hod_dev / doy_dev double [n]
 * -> u_dev double [n][6]. */
int glg_rule_control_batch(const double *settings29, const double *x_dev, const double *d_dev, const double *hod_dev,
                           const double *doy_dev, double *u_dev, int32_t n, int32_t device, void *stream);
/* RuleBasedController.predict for every env of the handle, on its CURRENT state, the weather row of its current timestep and
 * its clock -- the controls glg_step_rule_based computes in its prologue.  settings_dev: NULL (the handle's settings,
 * glg_set_rule_controller) or double [B][29] in rule_based.yml order, one row per env.  controls_dev: double [B][6].
 * glg_step_raw_control(h, controls_dev, noise_dev, stream) then steps exactly as glg_step_rule_based would.  One launch.
 * GLG_ERR_ARG on a NULL handle or NULL controls_dev, GLG_ERR_STATE before the first glg_reset. */
int glg_rule_controls(glg_handle *h, const double *settings_dev, double *controls_dev, void *stream);

/* End-to-end convenience for host callers (the SB3 VecEnv numpy path; replaces SubprocVecEnv.step_async / step_wait over
 * TomatoEnv.step, RL/utils.py:44-58): copies actions host->device, runs glg_step on the handle's own stream, delivers
 * obs/reward/done in host memory and synchronises.  Any output may be NULL.  obs_host float32 [B][obs_dim], reward_host
 * double [B], done_host uint8 [B].
 * How the observation rows reach obs_host is set by glg_set_host_obs_mode:
 *   0 (default) overlapped: the WeatherForecastObservations block (observations.py:163-182; 5 Np of the row's floats) is a
 *     function of (weather table, timestep) that is known before the kernel runs, so the host writes it into obs_host from its
 *     own float32 copy of the bank WHILE the kernel runs, only the other columns cross PCIe (0.45 MB instead of 4.35 MB per
 *     step at B = 4096), and after the synchronise every row is checked against the (table, timestep) the step left behind
 *     (rows that reset in place are filled again).  Same bytes in obs_host as mode 1.
 *   1 full: one device->host copy of the [B][obs_dim] array.
 * Stacks without a forecast block always use the full copy. */
int glg_step_host(glg_handle *h, const float *actions_host, float *obs_host, double *reward_host, uint8_t *done_host);
int glg_set_host_obs_mode(glg_handle *h, int32_t mode);
/* glg_step_host / glg_step_host_split work on the handle's own stream.  A caller that has enqueued work touching the handle on
 * another stream (glg_reset / glg_step with a stream argument, writes to the device views) orders the next host step behind it
 * with this call: an event recorded on `stream` that the handle's stream waits for -- no host synchronisation. */
int glg_host_path_after(glg_handle *h, void *stream);

/* Same step with the observation returned in SPLIT form (opt-in, for host loops that do not want 240 of 263 floats per env
 * that are a pure function of (weather table, timestep)): head_host float32 [B][obs_dim - 5 Np] receives every column of the
 * row except the WeatherForecastObservations block (observations.py:163-182), packed; timestep_host / table_host int32 [B]
 * receive each env's timestep and weather table AFTER the step, from which the caller reads the forecast block out of its
 * own copy of the weather bank: rows max(timestep, 1) .. + Np - 1, columns 0..4.  D2H per step at B = 4096: 0.43 MB instead of
 * 4.35 MB.  Any output may be NULL. */
int glg_step_host_split(glg_handle *h, const float *actions_host, float *head_host, int32_t *timestep_host, int32_t *table_host,
                        double *reward_host, uint8_t *done_host);

/* Output / state accessors: device pointers owned by the handle, valid until glg_destroy. */
int32_t glg_obs_dim(const glg_handle *h);          /* 23 + 5*Np */
float *glg_obs_dev(glg_handle *h);                 /* float32 [B][obs_dim]  (observations.py:59-182) */
float *glg_terminal_obs_dev(glg_handle *h);        /* float32 [B][obs_dim], rows valid where done=1 */
double *glg_reward_dev(glg_handle *h);             /* double [B]  (rewards.py:218-231) */
uint8_t *glg_done_dev(glg_handle *h);              /* uint8 [B]   terminated (tomato_env.py:131-132) */
double *glg_info_dev(glg_handle *h);               /* double [11][B]: EPI, revenue, variable_costs, fixed_costs, co2_cost,
                                                      heat_cost, elec_cost, temp_violation, co2_violation, rh_violation,
                                                      lamp_violation (tomato_env.py:208-222) */
double *glg_state_dev(glg_handle *h);              /* double [28][B] structure-of-arrays */
double *glg_controls_dev(glg_handle *h);           /* double [6][B] */
int32_t *glg_timestep_dev(glg_handle *h);          /* int32 [B] */
int32_t *glg_table_dev(glg_handle *h);             /* int32 [B] weather table of each env */
double *glg_time_dev(glg_handle *h);               /* double [2][B]: day_of_year, hour_of_day */
/* Finished-episode statistics (sums since the last clear): [0] episodes, [1] sum return, [2] sum length,
 * [3..13] sums of the 11 info entries, [14] non-finite terminations, [15] RK4 micro-steps executed, summed over envs
 * (counted by kernel B's guarded loop, i.e. with parametric uncertainty or the graded integrator; 0 otherwise). */
double *glg_stats_dev(glg_handle *h);
int glg_clear_stats(glg_handle *h, void *stream);

/* Test / teacher-forcing helpers (host arrays, synchronous).  x_host double [B][28], u_host double [B][6].
 * glg_set_state with a timestep also moves each env's clock to that timestep (day_of_year = start_day(table) + k dt/86400,
 * hour_of_day = (k dt/3600) mod 24, tomato_env.py:126-128,246-247); timesteps outside [0, N] are rejected. */
int glg_set_state(glg_handle *h, const double *x_host, const double *u_host, const int32_t *timestep_host);
int glg_get_state(glg_handle *h, double *x_host, double *u_host, int32_t *timestep_host);
/* Full per-env state for checkpoint / restore: everything a step reads besides the parameter table and the weather bank.
 * Any pointer may be NULL (skipped).  Host arrays: x [B][28], u [B][6], timestep [B], table [B] (0 <= id < n_tables),
 * time [B][2] (day_of_year, hour_of_day), step_ctr [B] (Philox stream position), ep_return [B], ep_len [B],
 * ep_info [B][11] (episode accumulators of the VecMonitor-style statistics). */
typedef struct glg_env_state {
    double *x, *u;
    int32_t *timestep, *table;
    double *time;
    uint32_t *step_ctr;
    double *ep_return;
    int32_t *ep_len;
    double *ep_info;
} glg_env_state;
int glg_get_state_ex(glg_handle *h, const glg_env_state *out_host);
int glg_set_state_ex(glg_handle *h, const glg_env_state *in_host);

/* ---- device rollout: VecNormalize statistics + normalisation, on-policy rollout buffer, GAE (SURVEY 8f-3) -------------------
 * What the reference's training loop puts between env.step and the PPO update -- SubprocVecEnv -> VecMonitor -> VecNormalize
 * (gl_gym/RL/utils.py:60-67; norm_obs / norm_reward / clip_obs / clip_reward / gamma from RL/experiment_manager.py:142-147) and
 * SB3's RolloutBuffer with generalised advantage estimation (configs/agents/ppo.yml: n_steps, gamma, gae_lambda) -- as kernels
 * on the handle's own outputs (csrc/glg_rollout.cuh), so a rollout never leaves the device.  Its own object: several rollout
 * buffers may share one env handle; destroy each before glg_destroy of the handle.  Errors are reported through glg_last_error of
 * the handle.  Episode return / length bookkeeping (VecMonitor) is part of the step kernel (glg_stats_dev).
 * Buffers (device, owned by the rollout): obs float32 [T+1][B][obs_dim] (normalised, clipped; slot t = what the policy sees
 * at step t, slot T = the observation after the last step), rewards float32 [T][B] (normalised), episode_starts float32
 * [T+1][B], advantages / returns float32 [T][B], statistics double [obs_dim + 1][3] = running (mean, var, count) per observation
 * column, last row = statistics of the discounted return. */
typedef struct glg_rollout_config {
    int32_t n_steps;     /* T */
    int32_t training;    /* 1: update the running statistics (VecNormalize.training) */
    int32_t norm_obs, norm_reward;
    double gamma, gae_lambda;
    double clip_obs, clip_reward, epsilon; /* 10, 10, 1e-8 in the reference's setup */
} glg_rollout_config;
typedef struct glg_rollout glg_rollout;
int glg_rollout_create(glg_handle *h, const glg_rollout_config *cfg, glg_rollout **out);
void glg_rollout_destroy(glg_rollout *r);
/* After glg_reset (t = -1): statistics fed with the first observations, normalised into slot 0, returns zeroed, every env
 * starts an episode.  After the glg_step* of rollout step t (0 <= t < T): observation statistics updated with the new raw
 * observations, which are normalised into slot t + 1; ret <- ret gamma + reward feeds the return statistics; the normalised
 * reward goes to slot t; episode_starts[t + 1] = done; ret[done] = 0.  Three launches on `stream`. */
int glg_rollout_store(glg_rollout *r, int32_t t, void *stream);
/* Start the next rollout without a reset: slot T (observation, episode_starts) becomes slot 0. */
int glg_rollout_carry(glg_rollout *r, void *stream);
/* RolloutBuffer.compute_returns_and_advantage: values_dev float32 [T+1][B] (row T = value of the slot-T observation). */
int glg_rollout_gae(glg_rollout *r, const float *values_dev, void *stream);
float *glg_rollout_obs_dev(glg_rollout *r);
float *glg_rollout_rewards_dev(glg_rollout *r);
float *glg_rollout_starts_dev(glg_rollout *r);
float *glg_rollout_advantages_dev(glg_rollout *r);
float *glg_rollout_returns_dev(glg_rollout *r);
double *glg_rollout_stats_dev(glg_rollout *r);

/* ---- device replay buffer for off-policy agents (SAC) ------------------------------------------------------------------------
 * SB3 2.6.0's ReplayBuffer (optimize_memory_usage False, handle_timeout_termination True) filled the way
 * OffPolicyAlgorithm._store_transition fills it behind VecNormalize (RL/utils.py:60-67), as kernels on the handle's outputs
 * (csrc/glg_replay.cuh).  Its own object: several buffers may share one env handle; destroy each before glg_destroy of the handle.
 * Capacity max(buffer_size / B, 1) slots per env, a ring indexed by pos with a `full` flag.  Each slot holds, per env, the raw
 * observation the transition started from, the raw next observation (the terminal observation of an env that finished under
 * auto_reset), the action, the raw reward (float32) and done.  Observations are stored without their WeatherForecastObservations
 * block plus the bank row that block is read from (221 B per transition at the default stack instead of 2140 B); the sample
 * kernel rebuilds the block from the weather bank bit for bit.  So glg_set_weather invalidates every replay buffer of the handle:
 * their store and sample then fail with GLG_ERR_STATE.  Errors are reported through glg_last_error of the handle. */
typedef struct glg_replay_config {
    int64_t buffer_size;  /* transitions over all envs (SB3 buffer_size) */
    int32_t training;     /* 1: update the running statistics (VecNormalize.training) */
    int32_t norm_obs, norm_reward, reserved;
    double gamma, clip_obs, clip_reward, epsilon; /* VecNormalize's; 0.99 / 10 / 10 / 1e-8 by default */
    uint64_t seed;        /* Philox key of the sample indices */
} glg_replay_config;
typedef struct glg_replay glg_replay;
int glg_replay_create(glg_handle *h, const glg_replay_config *cfg, glg_replay **out);
void glg_replay_destroy(glg_replay *r);
/* After glg_reset: the observation statistics are fed with the new observations, which are normalised into glg_replay_obs_dev,
 * the discounted returns are zeroed and every env's next transition starts from its current observation (VecNormalize.reset).
 * Stored transitions are kept.  Four launches on `stream`. */
int glg_replay_reset(glg_replay *r, void *stream);
/* After any glg_step* of the handle: VecNormalize.step_wait on the new observations and rewards (statistics, normalised current
 * observation, returns) and the transition into slot pos.  actions_dev float32 [B][6]: the action to store (SB3 stores the
 * policy's scaled action).  Four launches on `stream`. */
int glg_replay_store(glg_replay *r, const float *actions_dev, void *stream);
/* ReplayBuffer.sample(n) with VecNormalize: n transitions drawn with replacement, slot = Philox-uniform in [0, glg_replay_size),
 * env uniform in [0, B) (glg_replay_draw in csrc/glg_philox.h: draw block 65, counter (65, sample-call number, i, 0), key = seed).
 * obs_dev / next_obs_dev float32 [n][obs_dim] normalised with the current statistics and clipped, actions_dev float32 [n][6],
 * rewards_dev float32 [n] normalised by the return statistics and clipped, dones_dev float32 [n]; index_dev int32 [n][2]
 * receives the drawn (slot, env) pairs, or NULL.  GLG_ERR_STATE on an empty buffer.  One launch on `stream`. */
int glg_replay_sample(glg_replay *r, int32_t n, float *obs_dev, float *next_obs_dev, float *actions_dev, float *rewards_dev,
                      float *dones_dev, int32_t *index_dev, void *stream);
int64_t glg_replay_size(const glg_replay *r);   /* valid slots per env: pos, or the capacity once the ring is full */
int64_t glg_replay_bytes(const glg_replay *r);  /* device bytes the buffer holds */
float *glg_replay_obs_dev(glg_replay *r);       /* float32 [B][obs_dim]: normalised current observation */
double *glg_replay_stats_dev(glg_replay *r);    /* double [obs_dim + 1][3]: running (mean, var, count); last row = returns */

/* ---- receding-horizon planner: model-predictive control by the cross-entropy method (CEM) ------------------------------------
 * Scores candidate action sequences from the envs' CURRENT states with the step kernels (csrc/glg_plan.cuh) on the same reward as
 * the env.  A planner belongs to one env handle of B envs; it owns a second, internal handle of B K planning envs (planning env
 * c = b K + k starts from env b) created with the env's configuration except auto_reset 0, uncertainty_scale 0 (nominal model),
 * env_id_offset 0 and automatic kernel selection.  The env handle is only read.  Per env it keeps a sampling distribution over
 * sequences, mean and std float32 [H][B][6] in the action space (initially 0 and init_std), plus a seed and a call counter.
 * glg_plan_run, each of n_iterations CEM iterations:
 *   1. fan-out: x, u, timestep, table, clock and step_ctr of env b are copied into its K planning envs (device to device);
 *      their episode accumulators and done are zeroed.
 *   2. sample: candidate k = 0 is the mean; k >= 1: a = (float) clamp(mean + std z, -1, 1) in fp64, z standard normal by
 *      Box-Muller from Philox4x32-10 with counter (66, call, (it H + t) 3 + p, c) and key seed (glg_plan_normal2 in
 *      csrc/glg_philox.h; call = earlier glg_plan_run calls, p = component pair), laid out [H][B K][6].
 *   3. roll out: H glg_step of the planning envs; R_c = sum_t gamma^t reward_t over the steps up to and including the one that
 *      ends the episode (done); nothing after it counts.
 *   4. update: the n_elites largest returns of each env (ties to the lower k; non-finite returns rank last) give the new mean and
 *      population standard deviation per (t, component), summed in fp64 in ascending k, stored float32.  Deterministic.
 * The action returned for env b is the final mean[0][b].  Parameters (glg_set_params) are taken from the env at every call;
 * glg_set_weather on the env invalidates the planner (GLG_ERR_STATE).  Destroy the planner before its env handle.  Errors are
 * reported through glg_last_error of the env handle. */
typedef struct glg_plan_config {
    int32_t horizon;       /* H >= 1 steps */
    int32_t n_candidates;  /* K sequences per env, 1 .. 4096; num_envs * K <= 4194304 */
    int32_t n_elites;      /* E, 1 .. K */
    int32_t n_iterations;  /* I >= 1 CEM iterations per glg_plan_run */
    double gamma;          /* discount in (0, 1] */
    double init_std;       /* > 0: std after create and glg_plan_shift */
    uint64_t seed;         /* Philox key of the samples */
} glg_plan_config;
typedef struct glg_plan glg_plan;
int glg_plan_create(glg_handle *h, const glg_plan_config *cfg, glg_plan **out);
void glg_plan_destroy(glg_plan *p);
/* One decision: n_iterations CEM iterations from the env's current states; actions_dev float32 [B][6] <- mean[0].  GLG_ERR_STATE
 * before the env's first glg_reset.  Enqueued on `stream` (n_iterations (3 + 2 H) launches). */
int glg_plan_run(glg_plan *p, float *actions_dev, void *stream);
/* Fan-out and roll-out alone, for caller-supplied sequences: seq_dev float32 [H][B K][6], returns_dev double [B K] (may be
 * glg_plan_returns_dev). */
int glg_plan_evaluate(glg_plan *p, const float *seq_dev, double *returns_dev, void *stream);
/* Receding horizon: mean[t] <- mean[t + 1], mean[H - 1] <- 0 (hold the current controls), std <- init_std. */
int glg_plan_shift(glg_plan *p, void *stream);
/* glg_plan_run from caller-given states x_dev double [28][B] (SoA, the layout of glg_state_dev; e.g. glg_est_mean_dev) instead of
 * the env's x: output feedback.  u, timestep, table, clock and step_ctr still come from the env.  glg_plan_run(p, a, s) is
 * glg_plan_run_from(p, glg_state_dev(env), a, s). */
int glg_plan_run_from(glg_plan *p, const double *x_dev, float *actions_dev, void *stream);
float *glg_plan_mean_dev(glg_plan *p);        /* float32 [H][B][6]; writeable (re-initialise the distribution) */
float *glg_plan_std_dev(glg_plan *p);         /* float32 [H][B][6]; writeable */
float *glg_plan_candidates_dev(glg_plan *p);  /* float32 [H][B K][6]: the last iteration's samples */
double *glg_plan_returns_dev(glg_plan *p);    /* double [B K]: the last roll-out's returns */

/* ---- state estimation: an unscented Kalman filter (UKF) over the envs' observations -------------------------------------------
 * An estimator belongs to one env handle of B envs and keeps, per env, a state estimate x^ (double [28][B], the layout of
 * glg_state_dev) and its covariance P (double [B][28][28]).  It owns a second, internal handle of B S shadow envs (S = 57; sigma
 * point c = b S + i belongs to env b) created with the env's configuration except auto_reset 0, uncertainty_scale 0 (nominal
 * model), env_id_offset 0, automatic kernel selection and the IndoorClimateObservations stack alone.  The env handle is only read.
 * Filter contract (n = 28, S = 2n + 1 = 57):
 *   Weights: scaled unscented transform with alpha > 0, beta >= 0, kappa and n + lambda > 0: lambda = alpha^2 (n + kappa) - n,
 *     gamma = sqrt(n + lambda); Wm0 = lambda / (n + lambda), Wc0 = Wm0 + 1 - alpha^2 + beta; Wi = 1 / (2 (n + lambda)) for i >= 1.
 *     Defaults: alpha = 1, beta = 2, kappa = 0.
 *   Cholesky rule: P = L L^T column by column, summing over k in ascending order.  For column j, d = P[j][j] - sum_k L[j][k]^2; if
 *     d <= 1e-12 P[j][j] (which includes P[j][j] = 0), column j of L is zero; otherwise L[j][j] = sqrt(d) and
 *     L[i][j] = (P[i][j] - sum_k L[i][k] L[j][k]) / L[j][j].  (x27, the day counter, is deterministic: with p0_std[27] =
 *     q_std[27] = 0 its variance is exactly 0.)
 *   Sigma points: chi_0 = x^, chi_i = x^ + gamma L[:, i-1], chi_{n+i} = x^ - gamma L[:, i-1].
 *   Predict: chi'_i is one control interval of the env's nominal model (the env's precision, integrator and n_sub) from chi_i, with
 *     the controls the env just applied and the weather row the env's step just read.  xbar = sum Wm_i chi'_i,
 *     P- = sum Wc_i (chi'_i - xbar)(chi'_i - xbar)^T + diag(q_std^2); sums over i in ascending order.
 *   Measurement: h(x) = the 7 state-dependent observation entries in glg_obs_head order (co2_air ppm = dens2ppm(x2, 1e-6 x0), x2,
 *     rh(x2, x15), x9, x21, x25, x26: co2_air, temp_air, rh_air, pipe_temp, 24CanTemp, cFruit, tSum); meas_mask selects the measured
 *     subset M (bit r = entry r; 0 = all 7).  Additive-noise UKF on the propagated points, no redraw after adding Q:
 *     Y_i = h_M(chi'_i), ybar = sum Wm_i Y_i, S = sum Wc_i (Y_i - ybar)(Y_i - ybar)^T + diag(r_std_M^2),
 *     C = sum Wc_i (chi'_i - xbar)(Y_i - ybar)^T, K = C S^-1 (through the Cholesky of S), x^ = xbar + K (y - ybar),
 *     P = sym(P- - K S K^T), sym(A) = (A + A^T) / 2.  Without a measurement (y_dev NULL): x^ = xbar, P = P-.
 *   Episodes, read from the env handle after its step: the interval is the one at the env's pre-step timestep (timestep - 1; weather
 *     row min(k, rows - Np - 1) as in the step kernels) with the env's u and table.  An env that finished under auto_reset
 *     restarts: x^ <- the env's new state, P <- diag(p0_std^2).  The reset state is init_state(d0), a known function of the
 *     weather table, so the restart uses no privileged information.
 *   Status (uint8 bit flags per env, rewritten by every glg_est_update):
 *     1  a sigma point's step was non-finite (its shadow env is done while the pre-step timestep is < N): x^ and P unchanged;
 *     2  S is not positive definite: the prediction is kept, the update skipped;
 *     4  re-initialised by an auto-reset;
 *     8  the env's step_ctr is not the recorded value + 1 (the env was stepped or reset other than once since the last
 *        glg_est_update / glg_est_reset; the new value is recorded): x^ and P unchanged.
 * glg_set_weather on the env invalidates the estimator (GLG_ERR_STATE).  Errors are reported through glg_last_error of the env
 * handle.  The estimator may be destroyed before or after its env handle. */
typedef struct glg_est_config {
    double alpha, beta, kappa;
    int32_t meas_mask, reserved;
    double p0_std[28], q_std[28], r_std[7]; /* >= 0, finite; r_std > 0 for every measured entry */
} glg_est_config;
typedef struct glg_est glg_est;
/* GLG_ERR_ARG for NULLs, a bad configuration or num_envs * 57 > 4194304; GLG_ERR_STATE before the env has params and weather. */
int glg_est_create(glg_handle *h, const glg_est_config *cfg, glg_est **out);
void glg_est_destroy(glg_est *e);
/* x^ <- x0_dev (double [28][B] SoA; NULL = the env's x), P <- diag(p0_std^2), innovation 0, status 0, and the env's step_ctr
 * recorded.  GLG_ERR_STATE before the env's first glg_reset.  One launch. */
int glg_est_reset(glg_est *e, const double *x0_dev, void *stream);
/* After each step of the env: predict over the interval the env just took, then update with y_dev double [B][7] (entries in h
 * order; unmeasured ones are not read) or, when y_dev is NULL, predict only.  GLG_ERR_STATE before glg_est_reset.  Three launches:
 * the sigma kernel, glg_step_raw_control of the shadow handle, the UT kernel. */
int glg_est_update(glg_est *e, const double *y_dev, void *stream);
double *glg_est_mean_dev(glg_est *e);        /* [28][B], same layout as glg_state_dev */
double *glg_est_cov_dev(glg_est *e);         /* [B][28][28] */
double *glg_est_innovation_dev(glg_est *e);  /* [B][7]: y - ybar, 0 where not measured or not updated */
double *glg_est_sigma_dev(glg_est *e);       /* [28][B*57]: the propagated sigma points (the shadow handle's x) */
uint8_t *glg_est_status_dev(glg_est *e);     /* [B] */

/* ---- state smoothing: an unscented Rauch-Tung-Striebel smoother (URTS) over a recorded window of an estimator -----------------
 * A smoother belongs to one estimator and keeps, per env, a ring of W slots of the filter's forward quantities.  Recording does not
 * change a bit of the estimator's outputs (mean, cov, innovation, status).  Notation as in the filter contract above.
 * Smoother contract:
 *   Record: from the estimator's next glg_est_reset on.  Every glg_est_reset starts the record over and writes slot 0 (x^_0, P_0);
 *     each glg_est_update appends slot k+1 holding
 *       x^_{k+1}, P_{k+1}  the estimator's outputs after the update, bit for bit;
 *       xbar_{k+1}, P-_{k+1}  as the filter forms them, diag(q_std^2) included;
 *       D_{k+1} = sum_{i=1..2n} Wc_i (chi_i - x^_k)(chi'_i - xbar_{k+1})^T in ascending i, with chi_i - x^_k the offset
 *         +-gamma L[:, i-1] (the product the sigma points were formed with) and L the factor of P_k the update used;
 *       the env's status bits from this update and the env's timestep after its step.
 *     A slot that no one-interval prediction leads to (the reset slot, status 1, 4 or 8) holds xbar = P- = D = 0.  The ring keeps
 *     the last W estimates.
 *   Segments: slot k+1 starts a new segment when its status has bit 1, 4 or 8.  Status 2 and predict-only updates link to the slot
 *     before.  No gain crosses a segment start; the last slot of each segment is smoothed to its filtered value and its gain is 0.
 *   Deterministic states: a state j with p0_std[j] = q_std[j] = 0 (x27, the day counter, with the defaults) is left out: row and
 *     column j of G are 0, xs_j = x^_j, and row and column j of Ps are P's.  The rest of P- is factored by the filter's
 *     zero-column Cholesky rule.
 *   Backward pass, k from the newest slot down to the oldest in each segment:
 *     G_k = D_{k+1} (P-_{k+1})^-1: row i solves P- g_i = d_i by forward substitution through the factor and back substitution
 *       through its transpose; a component whose column of the factor is zero is 0.
 *     xs_k = x^_k + G_k (xs_{k+1} - xbar_{k+1}),  Ps_k = sym(P_k + G_k (Ps_{k+1} - P-_{k+1}) G_k^T).
 *     Sums run in ascending index order, without atomics: the result is deterministic.  The record is only read, so the smoother
 *     can run again as the window moves (run after every update: fixed-lag smoothing).  The lag-one cross-covariance EM needs is
 *     Ps_{k+1} G_k^T.
 * The smoother's memory is its own.  Destroy the smoother before its estimator; a smoother whose estimator is gone can only be
 * destroyed (glg_smooth_run returns GLG_ERR_STATE).  Errors are reported through glg_last_error of the env handle. */
typedef struct glg_smooth glg_smooth;
/* window >= 2 slots per env.  GLG_ERR_ARG for NULLs or a bad window, GLG_ERR_STATE if the estimator already has a smoother. */
int glg_smooth_create(glg_est *e, int32_t window, glg_smooth **out);
void glg_smooth_destroy(glg_smooth *s);
/* The backward pass over the valid slots into the output views.  GLG_ERR_STATE before the first recorded reset.  One launch. */
int glg_smooth_run(glg_smooth *s, void *stream);
int32_t glg_smooth_length(const glg_smooth *s);  /* valid slots: min(recorded, window) */
int32_t glg_smooth_first(const glg_smooth *s);   /* ring slot of the oldest valid estimate */
int64_t glg_smooth_bytes(const glg_smooth *s);   /* device bytes the smoother owns */
/* written by glg_smooth_run, oldest first (slot 0 is the oldest valid estimate) */
double *glg_smooth_mean_dev(glg_smooth *s);           /* [W][28][B] smoothed means */
double *glg_smooth_cov_dev(glg_smooth *s);            /* [W][B][28][28] smoothed covariances */
double *glg_smooth_gain_dev(glg_smooth *s);           /* [W][B][28][28] G_k; 0 at a segment's last slot */
/* the record, in ring order (glg_smooth_first names the oldest slot) */
double *glg_smooth_filtered_mean_dev(glg_smooth *s);  /* [W][28][B] x^ */
double *glg_smooth_filtered_cov_dev(glg_smooth *s);   /* [W][B][28][28] P */
double *glg_smooth_prior_mean_dev(glg_smooth *s);     /* [W][28][B] xbar */
double *glg_smooth_prior_cov_dev(glg_smooth *s);      /* [W][B][28][28] P- */
double *glg_smooth_cross_dev(glg_smooth *s);          /* [W][B][28][28] D */
uint8_t *glg_smooth_status_dev(glg_smooth *s);        /* [W][B] */
int32_t *glg_smooth_timestep_dev(glg_smooth *s);      /* [W][B] */

/* Noise settings that can change: p0_std, q_std, r_std (host arrays of 28, 28 and 7 doubles; NULL keeps a setting), validated as
 * in glg_est_create.  They are staged and take effect at the next glg_est_reset, so one record never mixes two noise models; that
 * reset also recomputes the smoother's deterministic-state mask.  GLG_ERR_ARG for a NULL estimator or a bad setting. */
int glg_est_set_noise(glg_est *e, const double *p0_std, const double *q_std, const double *r_std);

/* ---- noise identification: the E-step of an EM fit of the estimator's diagonal Q and R over a smoother's window -----------------
 * An EM object belongs to one smoother, as the smoother belongs to an estimator.  Notation as in the filter and smoother contracts.
 *   Log: from the estimator's next glg_est_reset on, per ring slot of the smoother and env: the controls the env applied (double
 *     [W][6][B]; 0 at a reset slot), the env's weather table ([W][B]), the measurement y_dev as given ([W][7][B]; 0 where not
 *     measured or y_dev is NULL), flags ([W][B]: bit 0 y_dev was non-NULL, bit 1 the update was applied: y_dev non-NULL and status
 *     0), and l = -(v^T S^-1 v + log det S + m log 2 pi) / 2 from the UT kernel's Cholesky of S and the innovation v (0 where no
 *     update was applied).  Logging does not change a bit of the estimator's outputs or of the smoother's record.
 *   E-step (glg_em_estep), over the smoother's output of its last glg_smooth_run (ms, Ps, G, oldest first); L is a factor by the
 *     filter's zero-column rule, the weights and gamma are the estimator's.
 *     Q term, for every slot k whose predecessor k-1 is in the window and linked to it (no status bit 1, 4 or 8 at k):
 *       chi_i: the sigma points of (ms_{k-1}, Ps_{k-1}); f_i one interval of the env's nominal model from chi_i with slot k's
 *       logged controls and table at pre-step timestep timestep_k - 1 (weather row min(k, rows - Np - 1)): the interval the
 *       filter's update stepped.  fbar = sum Wm_i f_i, Phi = sum Wc_i (f_i - fbar)(f_i - fbar)^T in ascending i;
 *       Delta_j = Wi gamma (f_{j+} - f_{j-}) (row j), Z = L^-T Delta by back substitution (a component whose column of L is zero is
 *       0), C = (Ps_k G_{k-1}^T) Z;  E_k = diag[Ps_k + (ms_k - fbar)(ms_k - fbar)^T + Phi - C - C^T].
 *       E_k is the expectation of (x_k - f(x_{k-1}))^2 under the smoothed joint of (x_{k-1}, x_k), with the cross term from the
 *       Gaussian regression of x_k on x_{k-1}; for f(x) = A x it is Shumway-Stoffer's.  A transition whose stepped point is
 *       non-finite (its EM env done before the season's end) is left out.
 *     R term, for every slot with the applied flag: the sigma points of (ms_k, Ps_k) through h;
 *       E_r = (y_r - hbar_r)^2 + sum Wc_i (h_ir - hbar_r)^2 for each measured entry r.
 *     Sums: per env in ascending slot order, then pooled in ascending env order; no atomics, so the result is deterministic.
 *   The points of all (env, slot) pairs are stepped by the unchanged step kernels of an internal handle (the EM handle, created
 *   like the estimator's shadow handle) in balanced chunks of at most max_points points, each stepped as a batch of exactly its
 *   own points (no padding, also while the window is not yet full): per chunk the sigma kernel, the step and the expectation
 *   kernel; then two reduction kernels.  The M-step (q_j^2 = pooled E_j / transitions, r_r^2 = pooled R_r /
 *   measured slots) is the caller's: glgym.estimation.DeviceNoiseEM.
 * Destroy the EM object before its smoother; one whose smoother or estimator is gone can only be destroyed (glg_em_estep returns
 * GLG_ERR_STATE).  glg_set_weather on the env makes glg_em_estep return GLG_ERR_STATE.  Errors are reported through glg_last_error
 * of the env handle. */
typedef struct glg_em glg_em;
/* max_points: sigma points per launch, 0 = 4194304, else 57 .. 4194304 (it bounds the EM handle's memory).  GLG_ERR_ARG for NULLs
 * or a bad max_points, GLG_ERR_STATE if the smoother already has an EM object or its estimator is gone. */
int glg_em_create(glg_smooth *s, int64_t max_points, glg_em **out);
void glg_em_destroy(glg_em *m);
/* The E-step over the smoother's output.  GLG_ERR_STATE before the first logged reset, or when the record changed since the last
 * glg_smooth_run.  Launches: 3 per chunk, then 2. */
int glg_em_estep(glg_em *m, void *stream);
int64_t glg_em_bytes(const glg_em *m);        /* device bytes of the log, the outputs and the EM envs' controls (not the EM handle) */
int64_t glg_em_logged(const glg_em *m);       /* slots logged since the estimator's last reset (more than W: the oldest are gone) */
int32_t glg_em_chunk_pairs(const glg_em *m);  /* most (env, slot) pairs per launch: min(B W, max_points / 57) */
/* the log, in the smoother's ring order (glg_smooth_first names the oldest slot) */
double *glg_em_controls_dev(glg_em *m);       /* [W][6][B] */
int32_t *glg_em_table_dev(glg_em *m);         /* [W][B] */
double *glg_em_measurements_dev(glg_em *m);   /* [W][7][B] */
uint8_t *glg_em_flags_dev(glg_em *m);         /* [W][B] */
double *glg_em_loglik_dev(glg_em *m);         /* [W][B] l */
/* written by glg_em_estep, oldest first */
double *glg_em_expectation_dev(glg_em *m);    /* [W][B][35]: E_k (28), then the R terms (7); 0 where a slot enters no sum */
double *glg_em_prediction_dev(glg_em *m);     /* [W][28][B] fbar: the smoothed one-step prediction; 0 where no transition */
uint8_t *glg_em_used_dev(glg_em *m);          /* [W][B] bit 0: the slot's transition entered the Q sums; bit 1: its R terms */
double *glg_em_env_stats_dev(glg_em *m);      /* [B][38] per env: the 35 sums, transitions, measured slots, sum of l */
double *glg_em_totals_dev(glg_em *m);         /* [38] pooled over the envs */

/* Multi-GPU episode statistics (SURVEY 8e): the step path has no collective; the one exchange is a sum of the 16-entry
 * statistics vector over the ranks' handles, once per logging interval -- ncclAllReduce on the handle's device buffer.
 * NCCL is bound at run time (dlopen of libnccl.so.2, the copy torch already loaded when there is one), so libglgym.so has no
 * link-time dependency on it.  Protocol: rank 0 calls glg_nccl_unique_id and broadcasts the 128 bytes by any means
 * (torch.distributed, MPI, a file); every rank calls glg_nccl_init with its rank; then glg_allreduce_stats enqueues the
 * all-reduce (in place, sum, float64 x 16) on `stream`.  The communicator is destroyed with the handle. */
int glg_nccl_unique_id(uint8_t id_out[128]);
int glg_nccl_init(glg_handle *h, const uint8_t id[128], int32_t rank, int32_t world_size);
int glg_allreduce_stats(glg_handle *h, void *stream);

/* evalF for a batch (pure function; replaces B calls of GreenLight::evalF, greenlight_model.cpp:96-120).
 * Row-major device arrays x[B][28], u[B][6], d[B][10], p[B][208] (p_stride = 208) or one shared p (p_stride = 0),
 * x_next[B][28].  bad_dev: optional uint8[B], 1 where the result is not finite. */
int glg_evalf_batch(const double *x_dev, const double *u_dev, const double *d_dev, const double *p_dev, int32_t p_stride,
                    double *x_next_dev, uint8_t *bad_dev, int32_t B, double dt, int32_t n_sub, int32_t device, void *stream);
/* Same with the integrator choice of glg_config.integrator (0 fixed-step, 1 graded). */
int glg_evalf_batch_ex(const double *x_dev, const double *u_dev, const double *d_dev, const double *p_dev, int32_t p_stride,
                       double *x_next_dev, uint8_t *bad_dev, int32_t B, double dt, int32_t n_sub, int32_t integrator,
                       int32_t device, void *stream);

/* Linearisation by forward-mode differentiation of the model (exact up to rounding, fp64).  All matrices are row-major float64,
 * J[b][i][j] = d out_i / d in_j; inputs as glg_evalf_batch_ex (x[B][28], u[B][6], d[B][10], p shared (p_stride = 0) or [B][208]).
 * Non-smooth points: fabs'(0) = 0; fmin / fmax / branches take the derivative of the branch the value takes; step-count decisions
 * (harvest micro-steps, graded splits) are frozen at the values, so the result is the Jacobian of the map on the executed grid.
 * Continuous-time RHS and its Jacobians: f_dev [B][28], jx_dev [B][28][28], ju_dev [B][28][6]; f_dev and ju_dev may be NULL. */
int glg_rhs_jacobian_batch(const double *x_dev, const double *u_dev, const double *d_dev, const double *p_dev, int32_t p_stride,
                           double *f_dev, double *jx_dev, double *ju_dev, int32_t B, int32_t device, void *stream);
/* Derivative of glg_evalf_batch_ex: x_next_dev [B][28], jx_dev [B][28][28], ju_dev [B][28][6], bad_dev uint8 [B];
 * x_next_dev, ju_dev and bad_dev may be NULL. */
int glg_evalf_jacobian_batch(const double *x_dev, const double *u_dev, const double *d_dev, const double *p_dev, int32_t p_stride,
                             double *x_next_dev, double *jx_dev, double *ju_dev, uint8_t *bad_dev, int32_t B, double dt,
                             int32_t n_sub, int32_t integrator, int32_t device, void *stream);
/* Linearise the step glg_step_raw_control(h, controls, NULL) would take, for every env of the handle, from its current state:
 * controls_dev double [B][6] (NULL: the env's current u), the weather row the step reads, the handle's nominal parameters,
 * dt, n_sub and integrator.  Always fp64 and the nominal model (also on a precision = 1 handle and under uncertainty_scale > 0).
 * x_next_dev [B][28] and ju_dev [B][28][6] may be NULL.  Writes nothing of the handle's; one launch.  GLG_ERR_ARG on a NULL
 * handle or NULL jx_dev, GLG_ERR_STATE before the first glg_reset. */
int glg_linearize(glg_handle *h, const double *controls_dev, double *x_next_dev, double *jx_dev, double *ju_dev, void *stream);

/* Number of kernels this handle has launched so far (bench.py's gpu_launches). */
int64_t glg_launch_count(const glg_handle *h);
/* Measured FP64 FMA throughput of the device [FLOP/s] (dependent-chain-free DFMA loop, all SMs); the roofline
 * denominator for this FP64-pipe-bound path. Synchronous. */
int glg_measure_fp64_peak(int32_t device, double *flops_per_s);
int glg_measure_fp32_peak(int32_t device, double *flops_per_s);

/* Accuracy probe of the kernel's branch-free fp64 math (csrc/glg_math.h): out[i] = f_op(in[i]) on the device.
 * op: 0 exp, 1 log, 2 rcp, 3 sqrt, 4 cbrt, 5 pow(x,0.66), 6 pow(x,0.32), 7 1/(1+exp(x)).  Tests only. */
int glg_debug_math(int32_t op, const double *in_dev, double *out_dev, int32_t n, void *stream);

#ifdef __cplusplus
}
#endif
#endif
