/*
 * fwgym.h — C-ABI of the B200-native batched fixed-wing simulator (libfwgym.so).
 *
 * This is the drop-in boundary for the hot path of eivindeb/fixed-wing-gym:
 *     FixedWingAircraft.step()  ->  PyFly.step()  ->  scipy solve_ivp(RK45)  ->  reward/target/observation
 * (reference: gym_fixed_wing/fixed_wing.py:338-437 "step", :287-336 "reset", :214-222 "seed").
 * The reference has no FFI of its own (pure Python); the binding a maintainer adds is the ctypes stub shown in
 * INTEGRATION.md.  Plain pointers and sizes only — no torch types.  All pointers marked "device" are CUDA device
 * pointers owned by the caller (e.g. torch CUDA tensors); every call is stream-ordered on the cudaStream_t passed
 * as `void* stream` (NULL = legacy default stream).  A handle is not thread-safe; distinct handles are independent.
 *
 * All functions return FW_OK (0) or a negative fw_status; fw_last_error() returns a message for the last failure
 * on the calling thread.
 */
#ifndef FWGYM_H
#define FWGYM_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define FW_ABI_VERSION 13

/* ---------------------------------------------------------------------------------------------- limits */
#define FW_MAX_OBS_VARS 32
#define FW_MAX_TARGETS 3
#define FW_N_ACT 3            /* elevator, aileron, throttle inputs (fixed_wing.py:39 forces actuation.inputs) */
#define FW_MAX_FACTORS 16
#define FW_N_FCLASS 3         /* linear, exponential, quadratic (fixed_wing.py:738-746) */
#define FW_MAX_GOAL_WORDS 8   /* success_streak_req <= 256 */
#define FW_N_SV 21            /* PyFly state variables, ids below */
#define FW_N_ODE 19           /* quat4, omega3, pos3, vel3, actuator value3, actuator dot3 */
#define FW_N_FILT 6           /* Dryden shaping filters u,v,w,p,q,r */
#define FW_FILT_MAXN 3
#define FW_N_PAR 53           /* == FW_PAR_N below (model parameters that can differ per env) */
#define FW_MAX_RAND 64        /* entries of simulator-parameter randomisation per reset */
#define FW_N_TURB_LEVELS 4    /* Dryden intensities of a mixed handle: 0 none, 1 light, 2 moderate, 3 severe */
#define FW_N_INERTIA 9        /* inertia terms of the right-hand side: gammas[1..8], inv_Jy */
#define FW_MAX_AIRCRAFT 53    /* per-env aircraft parameters: the live ones but ar, rho, g, Jx, Jy, Jz, Jxz */

/* PyFly state-variable ids (order of oracle/pyfly_restated.py REQUIRED_VARIABLES + elevons) */
enum fw_sv {
  FW_SV_ROLL = 0, FW_SV_PITCH, FW_SV_YAW, FW_SV_OMEGA_P, FW_SV_OMEGA_Q, FW_SV_OMEGA_R,
  FW_SV_POS_N, FW_SV_POS_E, FW_SV_POS_D, FW_SV_VEL_U, FW_SV_VEL_V, FW_SV_VEL_W,
  FW_SV_VA, FW_SV_ALPHA, FW_SV_BETA, FW_SV_ELEVATOR, FW_SV_AILERON, FW_SV_RUDDER, FW_SV_THROTTLE,
  FW_SV_ELEVON_L, FW_SV_ELEVON_R
};

/* Model parameters the right-hand side reads LIVE at every evaluation (PyFly.params[...] / PyFly.rho / PyFly.g), i.e.
 * the ones whose per-episode randomisation (fixed_wing.py:523-570) changes the dynamics.  The inertia entries are not
 * here: PyFly folds them into gammas at construction, so randomising them consumes a draw and changes nothing (a
 * per-env aircraft, fw_set_aircraft, does set them: see fw_air).  The last three are derived per env at reset (1/mass,
 * 1/(pi e AR), exp(2 M a_0)).  FW_PAR_MASS .. FW_PAR_C_N_DELTA_R are in the order of the fw_sim_t fields mass ..
 * C_n_delta_r. */
enum fw_par {
  FW_PAR_MASS = 0, FW_PAR_S_WING, FW_PAR_B, FW_PAR_C, FW_PAR_S_PROP, FW_PAR_K_MOTOR, FW_PAR_K_T_P, FW_PAR_K_OMEGA,
  FW_PAR_C_PROP, FW_PAR_E, FW_PAR_M, FW_PAR_A_0, FW_PAR_AR,
  FW_PAR_C_L_0, FW_PAR_C_L_ALPHA, FW_PAR_C_L_Q, FW_PAR_C_L_DELTA_E,
  FW_PAR_C_D_P, FW_PAR_C_D_0, FW_PAR_C_D_ALPHA1, FW_PAR_C_D_ALPHA2, FW_PAR_C_D_BETA1, FW_PAR_C_D_BETA2, FW_PAR_C_D_Q,
  FW_PAR_C_D_DELTA_E,
  FW_PAR_C_M_0, FW_PAR_C_M_ALPHA, FW_PAR_C_M_Q, FW_PAR_C_M_DELTA_E, FW_PAR_C_M_FP,
  FW_PAR_C_Y_0, FW_PAR_C_Y_BETA, FW_PAR_C_Y_P, FW_PAR_C_Y_R, FW_PAR_C_Y_DELTA_A, FW_PAR_C_Y_DELTA_R,
  FW_PAR_C_L_ROLL_0, FW_PAR_C_L_ROLL_BETA, FW_PAR_C_L_ROLL_P, FW_PAR_C_L_ROLL_R, FW_PAR_C_L_ROLL_DELTA_A,
  FW_PAR_C_L_ROLL_DELTA_R,
  FW_PAR_C_N_0, FW_PAR_C_N_BETA, FW_PAR_C_N_P, FW_PAR_C_N_R, FW_PAR_C_N_DELTA_A, FW_PAR_C_N_DELTA_R,
  FW_PAR_RHO, FW_PAR_G,
  FW_PAR_INV_MASS, FW_PAR_INV_PI_E_AR, FW_PAR_EXP_2MA0,
  FW_PAR_N
};

/* Ids of the per-env aircraft parameters (fw_sim_t.air_id): a fw_par id for the live parameters but FW_PAR_AR (always
 * b^2 / S_wing) and the derived ones, and these four for the inertia, which reaches the right-hand side only through
 * gammas[1..8] and inv_Jy (FW_AIR_JX == FW_PAR_N). */
enum fw_air { FW_AIR_JX = 53, FW_AIR_JY, FW_AIR_JZ, FW_AIR_JXZ };

enum fw_status {
  FW_OK = 0, FW_ERR_ARG = -1, FW_ERR_CUDA = -2, FW_ERR_CONFIG = -3, FW_ERR_ALLOC = -4, FW_ERR_ABI = -5,
  FW_ERR_WATCHDOG = -6   /* an env-kernel block gave up waiting for its aircraft: the handle refuses to step until a full
                          * fw_reset (or fw_set_state); see fw_step */
};

/* termination codes written to term_code_out (fixed_wing.py:366-368,383-385,409-416) */
#define FW_TERM_NONE 0
#define FW_TERM_STEPS 1
#define FW_TERM_SUCCESS 2
#define FW_TERM_NUMERIC 3      /* the integration left the representable range (non-finite state or step size: scipy's RK45
                                * loop would never return, rk.py:111-147 with a NaN h_abs) or needed more dopri5 attempts
                                * than fw_sim_t.max_attempts allows; handled like a constraint failure (done, step_fail
                                * reward); info["termination"] = "numeric" */
#define FW_TERM_FAIL_BASE 16   /* FW_TERM_FAIL_BASE + fw_sv id of the variable whose constraint was violated */

/* variable condition flags (PyFly Variable.apply_conditions) */
#define FW_VC_VMIN 1u
#define FW_VC_VMAX 2u
#define FW_VC_CMIN 4u
#define FW_VC_CMAX 8u
#define FW_VC_WRAP 16u

typedef struct {
  double vmin, vmax, cmin, cmax;   /* value clip and hard constraint, radians where applicable */
  double lo, hi, clo, chi;         /* same with missing bounds as -inf/+inf (branch-free device code) */
  double init_min, init_max;       /* uniform init range after curriculum scaling (fixed_wing.py:233-245) */
  uint32_t flags;
  uint32_t _pad;
} fw_var_t;

typedef struct {
  int32_t n;                        /* filter order 1..3 */
  int32_t stream;                   /* which of the 4 white-noise streams drives it */
  double Ad[FW_FILT_MAXN * FW_FILT_MAXN];   /* x' = x*Ad + u_prev*Bd0 + u*Bd1 (scipy lsim row-vector form) */
  double Bd0[FW_FILT_MAXN], Bd1[FW_FILT_MAXN], C[FW_FILT_MAXN];
  double D;
} fw_filter_t;

typedef struct {
  int32_t type;        /* 0 state, 1 target, 2 action (fixed_wing.py:797-830) */
  int32_t ref;         /* fw_sv id | target index | action index */
  int32_t value_kind;  /* target: 0 relative, 1 absolute, 2 integrator */
  int32_t window;      /* action: window_size */
  int32_t norm;        /* apply (val-mean)/var */
  int32_t _pad;
  double mean, var;
} fw_obs_var_t;

typedef struct {
  int32_t sv;          /* fw_sv id of the controlled state */
  int32_t cls;         /* 0 constant, 1 linear, 2 sinusoidal, 3 compensate (fixed_wing.py:933-991) */
  int32_t wrap;        /* PyFly Variable.wrap of that state */
  int32_t has_delta, has_bound, to_radians;
  double low, high, delta, bound;                 /* already in radians when to_radians */
  double slope_low, slope_high, amp_low, amp_high, period_low, period_high;   /* raw config units */
} fw_target_t;

typedef struct {
  int32_t cls;         /* 0 action, 1 state, 2 success, 3 step, 4 goal */
  int32_t type;        /* action: 0 value 1 delta 2 bound | state: 0 value 1 error 2 int_error | goal: 0 per_state 1 all */
  int32_t fclass;      /* 0 linear, 1 exponential, 2 quadratic */
  int32_t ref;         /* state.value: fw_sv id ; state.error/int_error: target index */
  int32_t window, shaping, has_max, value_timesteps;
  double scaling, max, sign, value;
  /* reward.randomize_scaling (fixed_wing.py:330-334): a factor configured with scaling = [low, high] draws a new
   * scaling at every reset; scale_slot1 = 1 + per-env scaling row, 0 = the fixed `scaling` above */
  int32_t scale_slot1, _pad;
  double scale_low, scale_high;
} fw_factor_t;

/* Flat configuration, compiled on the host from the reference's JSON files (config.py) */
/* simulator half: what PyFly holds (passed to the dynamics kernel as a __grid_constant__ parameter) */
typedef struct {
  double dt, rho, g;
  double rtol, atol;              /* scipy RK45 defaults 1e-3 / 1e-6 */
  double mass, S_wing, b, c, S_prop, k_motor, k_T_P, k_Omega, C_prop, e, M, a_0, ar;
  double C_L_0, C_L_alpha, C_L_q, C_L_delta_e;
  double C_D_p, C_D_0, C_D_alpha1, C_D_alpha2, C_D_beta1, C_D_beta2, C_D_q, C_D_delta_e;
  double C_m_0, C_m_alpha, C_m_q, C_m_delta_e, C_m_fp;
  double C_Y_0, C_Y_beta, C_Y_p, C_Y_r, C_Y_delta_a, C_Y_delta_r;
  double C_l_0, C_l_beta, C_l_p, C_l_r, C_l_delta_a, C_l_delta_r;
  double C_n_0, C_n_beta, C_n_p, C_n_r, C_n_delta_a, C_n_delta_r;
  double gammas[9];
  double Jy, inv_Jy, inv_mass, inv_pi_e_ar;   /* host-computed reciprocals (1 ulp from the divisions they replace) */
  double exp_2Ma0;                /* exp(2 M a_0) = e1*e2 of the stall blending function (one exp per RHS, dynamics.cuh) */
  int32_t drag_model;             /* 0 induced (1-sigma)CL^2/(pi e AR) + flat plate, 1 polynomial */
  int32_t turbulence;             /* Dryden gusts on */
  int32_t wind_enabled;           /* steady wind may be non-zero */
  int32_t max_attempts;           /* opt-in cap on dopri5 step attempts per env step (sim_config_kw "dopri5_max_attempts");
                                   * 0 = none, the reference's behaviour (a hang guard of 20000 remains) */
  double wind_mag_min, wind_mag_max;
  double turb_noise_scale;        /* sqrt(pi/dt) */
  fw_filter_t filt[FW_N_FILT];
  fw_var_t var[FW_N_SV];
  double act_coef[FW_N_ACT][6];   /* per dynamics actuator (elevon_l, elevon_r, throttle): c00 c01 c02 c10 c11 c12 */
  double act_dot_max[FW_N_ACT];
  int32_t act_has_dot_max[FW_N_ACT];
  int32_t _pad1;
  /* action scaling happens at the head of the dynamics kernel (fixed_wing.py:349-354,439-459) */
  int32_t scale_actions, has_scale_low, has_scale_high, _pad2;
  double scale_low, scale_high;
  double act_to_low[FW_N_ACT], act_to_high[FW_N_ACT];
  /* per-env model parameters (simulator-parameter randomisation): par_slot1[id] = 1 + row (relative to the handle's
   * parameter rows) holding that parameter for every env, 0 = the same for all envs (the value above) */
  int32_t par_slot1[FW_N_PAR];
  /* per-env Dryden intensity ("mixed" handle, sim_config_kw turbulence_intensity = {"values", "probabilities"}).  Ad /
   * Bd0 / Bd1 of filt[] do not depend on the intensity; the output rows C / D do, one set per level (level 0 = none is
   * all zero).  An env's level is chosen at its reset: its requested level (fw_set_turbulence_levels) when >= 0, else
   * the first l with u < turb_cdf[l] for one uniform u of Philox stream FW_RS_TURBLVL.  0 everywhere when not mixed. */
  int32_t turb_mixed, _pad;
  double turb_cdf[FW_N_TURB_LEVELS];
  double turb_C[FW_N_TURB_LEVELS][FW_N_FILT][FW_FILT_MAXN];
  double turb_D[FW_N_TURB_LEVELS][FW_N_FILT];
  /* per-env aircraft (fw_env_t.n_aircraft > 0, fw_set_aircraft): aircraft request row j sets parameter air_id[j]
   * (fw_air) at each reset; a NaN request flies the nominal value (the field above, or Jx / Jy / Jz / Jxz).  Listed
   * parameters, ar (when b or S_wing is listed), the derived rows and the inertia terms live in per-env parameter rows:
   * inertia_slot1[k] = 1 + row of gammas[1 + k] (k < 8) / inv_Jy (k = 8), 0 = the constant above.  All zero when no
   * aircraft parameter is listed. */
  double Jx, Jz, Jxz;
  int32_t air_id[FW_MAX_AIRCRAFT];
  int32_t inertia_slot1[FW_N_INERTIA];
  /* keeps sizeof(fw_sim_t) congruent to its earlier size (ABI 10) modulo 32, so every kernel parameter after it, also
   * behind the float image of the fp32 dynamics kernels (1.5x), keeps its 16-byte alignment and the compiler its
   * 128-bit constant loads: the kernels of existing configurations compile to the same instructions */
  int32_t _pad_air[2];
} fw_sim_t;

/* One draw of FixedWingAircraft.sample_simulator_parameters (fixed_wing.py:523-570), in the reference's order.
 * dist 0: gaussian  v = normal(orig, var), then np.clip(v, orig - clip, orig + clip) when has_clip
 * dist 1: uniform   v = uniform(orig - var, orig + var)
 * dist 2: uniform   v = uniform(orig, var)                     (simulator attributes given as low / high)
 * var / clip are absolute (the host applies var_type "relative": var * |orig|, clip * orig - signed, as the reference).
 * slot1: 1 + parameter row that receives v, 0 = drawn and discarded (a parameter the dynamics never read). */
typedef struct {
  int32_t par;         /* fw_par id, -1 when slot1 == 0 */
  int32_t dist, has_clip, slot1;
  double orig, var, clip;
} fw_rand_t;

/* env half: what FixedWingAircraft holds (passed to the env/reset kernels) */
typedef struct {
  int32_t steps_max, integration_window;
  int32_t obs_len, obs_step, obs_nvar, obs_shape, obs_norm, obs_noise;
  double obs_noise_mean, obs_noise_std;
  fw_obs_var_t obs[FW_MAX_OBS_VARS];
  int32_t has_bounds;
  int32_t n_aircraft;             /* per-env aircraft parameters: double state rows "aircraft_req" (fw_set_aircraft) */
  double bounds_min[FW_N_ACT], bounds_max[FW_N_ACT];
  int32_t n_targets, resample_every, streak_req, on_success;   /* on_success: 0 none, 1 done, 2 new */
  double streak_fraction;
  fw_target_t tgt[FW_MAX_TARGETS];
  int32_t n_factors, potential, step_fail_timesteps, n_terms;
  double step_fail_value;
  int32_t term_fclass[FW_N_FCLASS];
  double term_weight[FW_N_FCLASS];
  fw_factor_t fac[FW_MAX_FACTORS];
  /* episode metrics (FixedWingAircraft.get_metric, fixed_wing.py:1095-1162), streamed on the device when enabled */
  int32_t metrics_enabled, _pad4;
  double rise_low, rise_high;     /* rise_time thresholds (fractions of the initial error; config "metrics") */
  /* simulator-parameter randomisation at every reset (SURVEY §8f row 4) */
  int32_t n_rand, n_par_rows;     /* draws per reset; per-env parameter rows (randomised + derived) */
  fw_rand_t rand[FW_MAX_RAND];
  int32_t n_scale_rows;           /* per-env reward-scaling rows (reward.randomize_scaling) */
  int32_t bank_enabled;           /* the handle keeps the scenario-bank rows "bank_next" / "bank_scenario" (fw_set_bank) */
} fw_env_t;

typedef struct {
  int32_t abi_version;
  int32_t precision;              /* 0 = fp64 dynamics (parity mode), 1 = fp32 dynamics (opt-in) */
  fw_sim_t sim;
  fw_env_t env;
} fw_config_t;

typedef struct {
  uint64_t env_steps;        /* env steps executed since creation / last reset of counters */
  uint64_t attempts;         /* dopri5 step attempts (k summed over env steps) */
  uint64_t accepted;         /* accepted dopri5 steps */
  uint64_t warp_max_attempts;/* warp passes of the attempt kernel: each pass is one dopri5 attempt for up to 32 lanes (cost) */
  uint64_t warp_steps;       /* lane attempts executed in those passes (useful work); lane efficiency = this / (32 * passes) */
  uint64_t failures;         /* env steps that ended in a constraint failure */
  uint64_t resets;           /* auto + explicit episode resets */
  uint64_t rhs_evals;        /* RHS evaluations = 2*env_steps + 6*attempts */
  uint64_t watchdog;         /* env-kernel blocks that gave up waiting for their chunk's aircraft (must stay 0) */
} fw_counters_t;

typedef struct fw_handle_s* fw_handle;

/* Handle lifetime.  Replaces FixedWingAircraft.__init__ (fixed_wing.py:14-212) x n_envs; global_env_offset makes
 * RNG streams sharding-invariant (SURVEY §8e). */
int fw_create(const fw_config_t* cfg, int64_t n_envs, int64_t global_env_offset, int device, fw_handle* out);
int fw_destroy(fw_handle h);
const char* fw_last_error(void);
int fw_abi_version(void);
int64_t fw_config_sizeof(void);   /* sizeof(fw_config_t) as compiled, checked by the ctypes mirror */

/* Replaces FixedWingAircraft.seed (fixed_wing.py:214-222): Philox key for every env of the handle; the per-env draw
 * counters (ticks) restart, so seed(s) followed by a full reset reproduces the same episodes. */
int fw_seed(fw_handle h, uint64_t seed);

/* Replace the compiled configuration (set_curriculum_level / set_attr paths, fixed_wing.py:224-285). */
int fw_set_config(fw_handle h, const fw_config_t* cfg);

/* Replaces FixedWingAircraft.reset (fixed_wing.py:287-336) for the envs selected by `mask` (device uint8[N], NULL =
 * all).  init_state: optional device double [FW_N_SV + 3, N] (SoA; NaN entries = "sample it"; the last three rows are
 * the steady wind n, e, d), init_target: optional device double [FW_MAX_TARGETS, N] (NaN = sampled target kept).
 * turb_noise: optional device double [4, turb_len, N] = PyFly.reset(turbulence_noise=...) forwarded by
 * fixed_wing.py:287,308: the UNSCALED standard-normal samples of the four Dryden noise streams for the episode that
 * starts now (sim step s reads column s mod turb_len); the buffer must stay valid until those episodes end; envs that
 * auto-reset later go back to their Philox streams.  obs_out: device float [N, obs_dim] (rows of the envs not
 * selected are left untouched); obs64_out: optional device double copy for parity checks. */
int fw_reset(fw_handle h, const uint8_t* mask, const double* init_state, const double* init_target,
             const double* turb_noise, int64_t turb_len, float* obs_out, double* obs64_out, void* stream);

/* Replaces FixedWingAircraft.step (fixed_wing.py:338-437) + SubprocVecEnv auto-reset for all N envs.
 * actions: device [N, FW_N_ACT] row-major, float (actions_f64 = 0) or double (actions_f64 = 1).
 * obs_out float [N, obs_dim] (post-reset observation for envs that finished), rew_out float [N], done_out uint8 [N],
 * term_out int32 [N] (FW_TERM_*).  Optional (may be NULL): obs64_out / rew64_out double copies; term_obs_out float
 * [N, obs_dim] terminal observation of finished envs (rows of others untouched). auto_reset = 0 leaves finished envs
 * un-reset (single-env facade semantics).
 * Errors are sticky where they must be: the env kernel starts while the attempt kernel is still running and each of its
 * blocks waits for its 128 aircraft; a block that gives up (~1 s: a lost update, never observed) commits NOTHING for
 * its envs (their outputs are NaN / done = 0 / term = -1), raises a flag in host-visible memory, and from then on
 * fw_step, fw_host_submit, fw_host_wait and fw_counters return FW_ERR_WATCHDOG until a full fw_reset or fw_set_state
 * re-arms the step queue. */
int fw_step(fw_handle h, const void* actions, int actions_f64, float* obs_out, float* rew_out, uint8_t* done_out,
            int32_t* term_out, double* obs64_out, double* rew64_out, float* term_obs_out, int auto_reset,
            void* stream);

/* Host-buffer stepping: the call a policy living on the CPU makes (the reference's VecEnv.step takes and returns
 * host numpy arrays, train_rl_controller.py:223).  fw_host_open allocates `depth` slots of device staging and PINNED
 * host result buffers plus two copy streams.  fw_host_submit enqueues, without blocking on the GPU,
 *     H2D(actions_host) on the input copy stream -> fw_step on `stream` -> D2H(obs, reward, done, term) on the output
 *     copy stream,
 * and returns the slot; fw_host_wait blocks until that slot's results are on the host and returns pointers to them
 * (valid until the slot is submitted again: depth submissions later).  With depth >= 2 the PCIe traffic of step t
 * overlaps the kernels of step t+1.  actions_host: [N, FW_N_ACT] float32; pinned memory makes the upload asynchronous,
 * pageable memory is staged by the driver before the call returns.  Results: obs float [N, obs_dim], reward float
 * [N], done uint8 [N], term int32 [N] (FW_TERM_*), auto-reset semantics as fw_step(auto_reset = 1). */
int fw_host_open(fw_handle h, int depth);
/* zero_copy != 0: the result buffers are MAPPED pinned host memory and the env kernel writes observations (as coalesced
 * bursts through a shared-memory tile), rewards, dones and termination codes straight into them while the dynamics
 * kernels of the step are still finishing other chunks: no device -> host copy follows the step, fw_host_wait returns
 * when the env kernel has completed.  Results are identical. */
int fw_host_open_ex(fw_handle h, int depth, int zero_copy);
int fw_host_close(fw_handle h);
int fw_host_submit(fw_handle h, const float* actions_host, void* stream, int* slot_out);
int fw_host_wait(fw_handle h, int slot, const float** obs, const float** rew, const uint8_t** done,
                 const int32_t** term);

/* Per-env Dryden intensity of a mixed handle (fw_sim_t.turb_mixed): levels = device int32 [N], -1 = draw from the
 * handle's distribution at every reset, 0..3 = pinned (none, light, moderate, severe), any other value counts as -1;
 * NULL sets every env to -1.  Takes
 * effect at each env's next reset (explicit or automatic).  FW_ERR_ARG on a handle that is not mixed.  The requested
 * and active levels are the state rows "turb_level_req" / "turb_level" (fw_get_state / fw_set_state). */
int fw_set_turbulence_levels(fw_handle h, const int32_t* levels, void* stream);

/* Per-env aircraft (fw_env_t.n_aircraft > 0): values = device double [fw_aircraft_dim(h), N], row j = the requested value
 * of parameter fw_sim_t.air_id[j] for every env, NaN = the handle's nominal value; NULL sets every request to NaN.
 * Takes effect at each env's next reset (explicit or automatic): the reset writes the episode's parameters and
 * recomputes what PyFly derives from them at construction (ar = b^2 / S_wing, 1/mass, 1/(pi e ar), exp(2 M a_0),
 * gammas[1..8] and 1/Jy), so the running episode keeps its aircraft.  No random draw is added or moved.  FW_ERR_ARG on a
 * handle without aircraft parameters.  The requests are the state rows "aircraft_req" (fw_get_state / fw_set_state). */
int fw_set_aircraft(fw_handle h, const double* values, void* stream);
/* Number of per-env aircraft parameters of the handle (rows of fw_set_aircraft), 0 when none. */
int64_t fw_aircraft_dim(fw_handle h);

/* Scenario bank (handles created with fw_env_t.bank_enabled): a device table of S initial states / targets that resets
 * consume in order, with one result row per scenario.  Every env keeps two int32 state rows: "bank_next" (scenario id of
 * its next banked episode) and "bank_scenario" (scenario id of the running episode, -1 when it is not from the bank).
 * fw_set_bank sets bank_next = first + e for local env e (mod S when `cycle`) and bank_scenario = -1; every reset that
 * injects nothing (auto-resets, fw_reset with NULL init_state and init_target) while bank_next < S starts scenario
 * bank_next, exactly as fw_reset would with the scenario's columns as init_state / init_target (NaN = sample it), and
 * advances bank_next by `stride` (mod S when `cycle`, else saturating at S).  stride >= n_envs keeps any two envs off the
 * same scenario; sharded ranks pass first = their env offset and stride = the total env count.  An env past the bank
 * samples from the configured ranges; a reset with init_state or init_target leaves the cursor alone (bank_scenario = -1).
 * When a banked episode ends (with or without auto_reset) the env kernel writes the optional result rows at index
 * bank_scenario (only below S), counts it, and sets bank_scenario = -1.  The tables and result buffers must stay valid
 * while the bank is attached.  The cursor rows are state (fw_get_state / fw_set_state); the pointers are not: to resume a
 * checkpoint, attach the bank, then fw_set_state. */
typedef struct {
  const double* init_state;       /* optional device double [FW_N_SV + 3, S] (rows as fw_reset init_state) */
  const double* init_target;      /* optional device double [FW_MAX_TARGETS, S] */
  const int32_t* turb_level;      /* optional device int32 [S] (mixed handles only): >= 0 pins the episode's Dryden level
                                   * like fw_set_turbulence_levels, -1 keeps the env's own rule */
  int64_t n_scenarios;            /* S: 1 .. INT32_MAX */
  int64_t first, stride;          /* assignment: env e flies first + e, then + stride per episode; stride >= n_envs */
  int32_t cycle;                  /* != 0: the cursor wraps modulo S (no outcome rows allowed, several envs share ids) */
  int32_t _pad;
  int32_t* term;                  /* optional device int32 [S]: termination code (FW_TERM_*) */
  int32_t* length;                /* optional device int32 [S]: episode length in env steps */
  double* ret;                    /* optional device double [S]: episode return */
  double* episode;                /* optional device double [S, fw_episode_dim] metric rows (metrics enabled only) */
  int32_t* episodes;              /* optional device int32 [S]: banked episodes ended per scenario (atomic counts) */
  int32_t* successes;             /* optional device int32 [S]: of those, episodes whose success streak was reached */
} fw_bank_t;
/* Attach (bank != NULL) or detach (NULL) a scenario bank.  FW_ERR_ARG: the handle was not created with bank_enabled,
 * S <= 0 or S > INT32_MAX, first < 0, stride < n_envs, an episode buffer without metrics, outcome rows (term / length /
 * ret / episode) together with cycle, or a level column on a handle that is not mixed.  Attaching or detaching also
 * detaches the aircraft column (fw_set_bank_aircraft). */
int fw_set_bank(fw_handle h, const fw_bank_t* bank, void* stream);
/* Aircraft column of the attached bank (handles with aircraft parameters): aircraft = device double [fw_aircraft_dim(h),
 * S], NULL = none.  A finite entry pins that parameter of the scenario's episodes like fw_set_aircraft; NaN keeps the
 * env's request.  The column must stay valid while it is attached; the next fw_set_bank detaches it.  FW_ERR_ARG: the
 * handle has no aircraft parameters, or no bank is attached. */
int fw_set_bank_aircraft(fw_handle h, const double* aircraft);

/* Rows [row0, row0 + nrows) of the state matrix below: device double [nrows, N] (e.g. the three target rows without
 * exporting the whole state). */
int fw_get_rows(fw_handle h, int64_t row0, int64_t nrows, double* out, void* stream);

/* Full per-env state for parity, checkpoint/resume: device double [fw_state_rows(h), N]. */
int64_t fw_state_rows(fw_handle h);
int fw_get_state(fw_handle h, double* out, void* stream);
int fw_set_state(fw_handle h, const double* in, void* stream);
/* name of row r of the state matrix ("q0", "omega_p", "steps_count", ...), NULL when out of range */
const char* fw_state_row_name(fw_handle h, int64_t r);

/* Per-env dopri5 attempt count of the last step (also for envs whose episode ended in it): device int32 [N]. */
int fw_last_attempts(fw_handle h, int32_t* out, void* stream);

/* Counters (synchronises the stream it was last used on). */
int fw_counters(fw_handle h, fw_counters_t* out);
int fw_reset_counters(fw_handle h);

/* Per-kernel device timing: when on, every fw_step records CUDA events around the dynamics and env kernels on the
 * launching stream; fw_profile() synchronises, returns the summed milliseconds and the number of steps, and clears. */
int fw_set_profiling(fw_handle h, int on);
int fw_profile(fw_handle h, double* dyn_ms, double* env_ms, int64_t* steps);

/* Episode metric sums for a caller-side NCCL all-reduce (SURVEY §8e): out double [FW_N_METRIC_SUMS] on the host. */
#define FW_N_METRIC_SUMS 8   /* episodes, successes, sum_return, sum_length, failures, steps_term, success_term, goal_steps */
int fw_metric_sums(fw_handle h, double* out_host);

/* Episode metrics (SURVEY §8f row 1).  With cfg.env.metrics_enabled the env kernel keeps streaming forms of every
 * FixedWingAircraft.get_metric quantity (fixed_wing.py:1095-1162, evaluated by the reference inside step() when an
 * episode ends, :417-419) and, for every env whose episode ended in a step, writes one row of fw_episode_dim(h)
 * doubles to the registered device buffer [N, dim] (rows of other envs untouched; done_out says which are fresh).
 * Row layout: return, length, control_variation, success_all, settling_time_all, success_time_frac_all, then per
 * target k: avg_error, total_error, end_error, rise_time, overshoot, success, settling_time, success_time_frac
 * (NaN where the reference yields nan / has no entry). */
int fw_episode_dim(fw_handle h);
int fw_set_episode_out(fw_handle h, double* ep_out);

/* PID baseline controller (SURVEY §8f row 2): pyfly/pid_controller.py as used by evaluate_controller.py:141-151,202.
 * One call = PIDController.set_reference(current targets) + get_action(roll, pitch, Va, omega) for every env, read
 * straight from the handle's state rows (the reference reads the same values out of the un-normalised, noise-free
 * observation vector of its evaluation config).  integ: device double [3, N] integrators (Va, roll, pitch), owned by
 * the caller; reset_mask: optional device uint8 [N], non-zero = PIDController.reset() first.  actions_out: device
 * double [N, 3] = (elevator, aileron, throttle) in physical units (use an env with action.scale_space = false). */
typedef struct {
  double k_p_V, k_i_V;
  double k_p_phi, k_i_phi, k_d_phi;
  double k_p_theta, k_i_theta, k_d_theta;
  double delta_a_min, delta_a_max, delta_e_min, delta_e_max, delta_t_min, delta_t_max;
} fw_pid_gains_t;
int fw_pid_step(fw_handle h, const fw_pid_gains_t* gains, double* integ, const uint8_t* reset_mask,
                double* actions_out, void* stream);

/* Introspection */
int64_t fw_num_envs(fw_handle h);
int fw_obs_dim(fw_handle h);
/* Kernel launches one fw_step issues: init, attempt and env kernel. */
int fw_launches_per_step(fw_handle h);
/* Which kernel instantiations this handle's configuration selected: "dyn=<shipped|generic|rand> env=<shape name|generic>"
 * (dynamics.cuh "kernel specialisation", env_shapes.h).  Valid until the next call on the calling thread. */
const char* fw_kernel_variant(fw_handle h);

/* Experiment hook (scheduling studies, DESIGN.md 4.4): `order` is a device int32 [N] permutation of the env ids, the
 * order in which the attempt kernel's warps adopt aircraft (NULL restores the natural order).  Results do not depend
 * on it; the time does.  The buffer must stay valid while it is set. */
int fw_debug_set_order(fw_handle h, const int32_t* order);

/* Test hook for the watchdog path: spin_limit = polls of the chunk counter before an env block gives up (0 restores the
 * default, ~1 s); starve != 0 makes block 0 of the NEXT step wait for one aircraft more than exist, so it must time out. */
int fw_debug_watchdog(fw_handle h, uint32_t spin_limit, int starve);

/* Experiment hook (library built with -DFW_TIMELINE only; otherwise the values never change): out8 = GPU global-timer
 * stamps in ns {init first start, init last end, attempt first start, attempt last end, env first start, env last end,
 * first env block past its chunk wait, sum of env block run times}; reset != 0 re-arms the buffer afterwards. */
int fw_debug_timeline(unsigned long long* out8, int reset);

/* Micro-benchmark: sustained DFMA throughput of this GPU in FLOP/s (roofline denominator, bench.py). */
int fw_dfma_peak(int device, double* flops_out, double* ms_out);

#ifdef __cplusplus
}
#endif
#endif /* FWGYM_H */
