// Structure-of-arrays state layout in HBM: one row per quantity, N (padded) contiguous envs per row, so that lane i
// of a warp touches element i of a row (fully coalesced 256 B per warp per row for doubles).
#pragma once
#include <stdint.h>
#include "../../include/fwgym.h"

// ---- double rows (fixed part) -------------------------------------------------------------------------------
enum {
  D_Q = 0,          // 4  quaternion (normalised at each env step, PyFly _set_states_from_ode_solution)
  D_OMEGA = 4,      // 3
  D_POS = 7,        // 3
  D_VEL = 10,       // 3
  D_ACT = 13,       // 3  elevon_left, elevon_right, throttle values
  D_ACTDOT = 16,    // 3
  D_ROLL = 19, D_PITCH = 20, D_YAW = 21, D_VA = 22, D_ALPHA = 23, D_BETA = 24, D_ELEV = 25, D_AIL = 26,
  D_CMD = 27,       // 3  constrained model commands (elevator, aileron, throttle) of the last step
  D_WIND = 30,      // 3  steady wind NED
  D_TX = 33,        // 18 Dryden filter states, 3 per filter
  D_TU = 51,        // 4  previous white-noise sample per stream (already scaled by sqrt(pi/dt))
  D_GUST = 55,      // 6  current gust: linear u,v,w then angular p,q,r
  D_TARGET = 61,    // 3
  D_TSLOPE = 64, D_TAMP = 67, D_TPERIOD = 70, D_TPHASE = 73, D_TBIAS = 76,   // 3 each
  D_PREVSHAPE = 79, // 3  prev_shaping per function class
  D_ERR0 = 82,      // 3  history["error"][k][0]
  D_EPRET = 85,     // episode return
  D_FIXED = 86
};

// ---- int32 rows (fixed part) --------------------------------------------------------------------------------
enum {
  I_STEPS = 0,      // steps_count
  I_STEPS_TGT,      // _steps_for_current_target
  I_HISTLEN,        // len(history["error"][k]) == len(PyFly Variable.history) (successful steps + 1)
  I_TICK,           // rng tick (next call uses this value)
  I_EPTICK,         // tick of the reset that started the episode (keys the turbulence stream)
  I_FLAGS,          // FWF_* bits
  I_GOALCNT,        // number of set bits among the last streak_req entries of the "all" goal history
  I_LASTK,          // dopri5 attempts of the last step
  I_STATUS,         // last sim step: 0 ok, else FW_TERM_FAIL_BASE + sv
  I_GOALRING,       // FW_MAX_GOAL_WORDS words
  I_FIXED = I_GOALRING + FW_MAX_GOAL_WORDS
};

#define FWF_GOAL_ACHIEVED 1u      // fixed_wing.py:51,382 latch (never cleared by reset)
#define FWF_HIST_VALID 2u         // self.history is not None (a previous episode exists)
#define FWF_PREVSHAPE_SHIFT 2     // 3 bits: prev_shaping[fclass] is not None
#define FWF_TCLS_SHIFT 8          // 2 bits per target: current class (reset(target=) may force constant)
#define FWF_EP_SUCCESS (1u << 16) // streak achieved in this episode (metric "success"["all"])
#define FWF_TURB_INJ (1u << 17)   // this episode's Dryden noise was injected at reset (fw_reset turb_noise), not drawn

// variable part, computed from the config by fw_layout_build below (host: make_layout in fwgym.cu; device: folded)
struct FwLayout {
  int64_t n;            // number of envs
  int64_t stride;       // padded row length (multiple of 32)
  int32_t d_rows, i_rows;
  int32_t act_depth, act_row;     // raw-action ring: act_depth x 3 rows starting at act_row (double)
  int32_t cmd_depth, cmd_row;     // constrained-command ring (only when scale_actions == 0)
  int32_t sv_depth, sv_row;       // observed-state ring: sv_depth x n_sv_obs rows
  int32_t n_sv_obs;
  int32_t err_depth, err_row;     // error ring: err_depth x n_targets
  int32_t tgt_depth, tgt_row;     // target ring: tgt_depth x n_targets
  int32_t goal_words;
  int32_t sv_slot[FW_MAX_OBS_VARS];   // obs var index -> column in the sv ring (-1 if not a state var)
  // episode metrics (only when fw_env_t.metrics_enabled): accumulator rows + the 50-entry error ring of end_error
  int32_t met, m_drow, m_irow, end_row;
  // per-env model parameters (simulator-parameter randomisation): n_par_rows rows starting at par_row
  int32_t par_row, n_par_rows;
  // per-env reward scalings (reward.randomize_scaling): n_rs_rows rows starting at rs_row
  int32_t rs_row, n_rs_rows;
  // per-env Dryden intensity (only when fw_sim_t.turb_mixed): int32 rows tl_row (requested level, -1 = draw at every
  // reset) and tl_row + 1 (level of the running episode); n_tl_rows = 0 or 2
  int32_t tl_row, n_tl_rows;
  // scenario bank (only when fw_env_t.bank_enabled): int32 rows bank_row (scenario id of the next banked episode) and
  // bank_row + 1 (scenario id of the running episode, -1: not from the bank); n_bank_rows = 0 or 2.  (These two fields
  // took the place of padding: the struct keeps its size, so no kernel parameter after it moves.)
  int32_t bank_row, n_bank_rows;
  // per-env aircraft (only when fw_env_t.n_aircraft > 0): double rows air_row .. air_row + n_air_rows - 1, the requested
  // value of each listed parameter (NaN = nominal).  16 bytes, so that every kernel parameter after it keeps its alignment.
  int32_t air_row, n_air_rows;
  int32_t _pad_air[2];
};

// metric accumulators, relative to FwLayout.m_drow (double) / m_irow (int32); k = target index
#define FW_END_WINDOW 50
enum { MD_SUME = 0, MD_SUMABS = 3, MD_MIN = 6, MD_MAX = 9, MD_PREVABS = 12, MD_CV = 15, MD_PREVCMD = 16, MD_ROWS = 19 };
enum { MI_RISE_LO = 0, MI_RISE_HI = 3, MI_SETTLE = 6 /* k, 3 = all */, MI_GSUM = 10 /* k, 3 = all */, MI_GCNT = 14,
       MI_GRING = 17 /* 3 x goal_words */ };
enum { EP_RETURN = 0, EP_LENGTH, EP_CV, EP_SUCCESS_ALL, EP_SETTLE_ALL, EP_STF_ALL, EP_PER_TARGET = 6,
       EPT_AVG = 0, EPT_TOTAL, EPT_END, EPT_RISE, EPT_OVERSHOOT, EPT_SUCCESS, EPT_SETTLE, EPT_STF, EPT_N = 8 };

// Layout of the variable part.  constexpr so that the SAME function sizes a handle on the host (make_layout, fwgym.cu)
// and folds the row numbers of a compile-time configuration shape into the specialised env kernels (env_shapes.h).
// Returns 0 or a 1-based error number (messages: fw_layout_error).
constexpr int fw_layout_build(const fw_env_t& E, int scale_actions, int64_t n, FwLayout& L, int turb_mixed = 0) {
  L = FwLayout{};
  L.n = n;
  L.stride = (n + 31) / 32 * 32;
  if (E.obs_len < 1 || E.obs_step < 1 || E.obs_nvar < 1 || E.obs_nvar > FW_MAX_OBS_VARS) return 1;
  if (E.n_targets < 0 || E.n_targets > FW_MAX_TARGETS) return 2;
  if (E.n_factors < 0 || E.n_factors > FW_MAX_FACTORS) return 3;
  if (E.streak_req > 32 * FW_MAX_GOAL_WORDS) return 4;
  const int imax = (E.obs_len - 1) * E.obs_step + 1;   // deepest history index used by an observation row
  int row = D_FIXED;
  int act_need = 0, win_obs = 0;
  bool need_err = false, need_tgt = false, integ = false;
  for (int v = 0; v < E.obs_nvar; ++v) {
    L.sv_slot[v] = -1;
    const fw_obs_var_t& ov = E.obs[v];
    if (ov.type == 0) L.sv_slot[v] = L.n_sv_obs++;
    if (ov.type == 1 && ov.value_kind == 0 && E.obs_len > 1) need_err = true;
    if (ov.type == 1 && ov.value_kind == 1 && E.obs_len > 1) need_tgt = true;
    if (ov.type == 1 && ov.value_kind == 2) { need_err = true; integ = true; }
    if (ov.type == 2) win_obs = ov.window > win_obs ? ov.window : win_obs;
  }
  if (win_obs > 0) act_need = win_obs + imax;
  bool int_err = false;
  for (int f = 0; f < E.n_factors; ++f) {
    const fw_factor_t& F = E.fac[f];
    if (F.cls == 0 && F.type == 1) act_need = F.window + 1 > act_need ? F.window + 1 : act_need;
    if (F.cls == 1 && F.type == 2) { need_err = true; int_err = true; }
  }
  if ((integ || int_err) && E.integration_window <= 0) return 5;
  if (act_need > 0) {
    const bool raw = scale_actions != 0;
    // reward "delta" always reads the raw action history; action observations read raw actions when scale_actions
    // and PyFly's constrained command history otherwise (fixed_wing.py:824-828)
    L.act_depth = act_need; L.act_row = row; row += act_need * FW_N_ACT;
    if (!raw && win_obs > 0) { L.cmd_depth = act_need; L.cmd_row = row; row += act_need * FW_N_ACT; }
  }
  if (E.obs_len > 1 && L.n_sv_obs > 0) { L.sv_depth = imax + 1; L.sv_row = row; row += L.sv_depth * L.n_sv_obs; }
  else L.sv_depth = 1;
  if (need_err) {
    L.err_depth = ((integ || int_err) ? E.integration_window : 0) + imax + 2;
    L.err_row = row; row += L.err_depth * E.n_targets;
  }
  if (need_tgt) { L.tgt_depth = imax + 1; L.tgt_row = row; row += L.tgt_depth * E.n_targets; }
  L.goal_words = (E.streak_req + 31) / 32;
  L.i_rows = I_FIXED;
  if (E.metrics_enabled) {
    L.met = 1;
    L.m_drow = row; row += MD_ROWS;
    L.end_row = row; row += FW_END_WINDOW * E.n_targets;
    L.m_irow = L.i_rows; L.i_rows += MI_GRING + 3 * L.goal_words;
  }
  if (turb_mixed) { L.tl_row = L.i_rows; L.n_tl_rows = 2; L.i_rows += 2; }
  if (E.bank_enabled) { L.bank_row = L.i_rows; L.n_bank_rows = 2; L.i_rows += 2; }
  if (E.n_rand < 0 || E.n_rand > FW_MAX_RAND || E.n_par_rows < 0 || E.n_par_rows > FW_N_PAR + FW_N_INERTIA) return 6;
  L.par_row = row;
  L.n_par_rows = E.n_par_rows;
  row += E.n_par_rows;
  if (E.n_scale_rows < 0 || E.n_scale_rows > FW_MAX_FACTORS) return 7;
  L.rs_row = row;
  L.n_rs_rows = E.n_scale_rows;
  row += E.n_scale_rows;
  if (E.n_aircraft < 0 || E.n_aircraft > FW_MAX_AIRCRAFT) return 8;
  if (E.n_aircraft) { L.air_row = row; L.n_air_rows = E.n_aircraft; row += E.n_aircraft; }
  L.d_rows = row;
  return 0;
}
inline const char* fw_layout_error(int code) {
  switch (code) {
    case 1: return "bad observation length/step/nvar";
    case 2: return "bad n_targets";
    case 3: return "bad n_factors";
    case 4: return "success_streak_req > 256 unsupported";
    case 5: return "integrator observation / int_error reward need integration_window > 0";
    case 6: return "bad simulator-parameter randomisation table";
    case 7: return "bad reward-scaling randomisation table";
    case 8: return "bad number of aircraft parameters";
  }
  return "";
}

