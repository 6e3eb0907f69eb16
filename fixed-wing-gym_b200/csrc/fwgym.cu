// libfwgym.so — kernels + C-ABI (include/fwgym.h).  sm_100a only.
//
//   fw_init_kernel    : one thread per aircraft, natural order: action scaling + command constraining, f(t0, y0) and
//                       scipy's initial step size (2 RHS evaluations), parked in carry rows.
//   fw_attempt_kernel : persistent warps, one aircraft per lane; every pass is one dopri5 step attempt (6 RHS
//                       evaluations, K stages in shared memory); lanes adopt the next waiting aircraft at attempt
//                       boundaries.  FP64-pipe / dependent-issue bound (DESIGN.md 4.2).
//   fw_env_kernel     : one thread per env, specialised on the configuration's shape (env_shapes.h): PyFly's state
//                       commit, Dryden filter advance, goal bits / streak, reward, target resample + advance, history
//                       rings, observation (+noise), done, metric sums, auto-reset.  Launched as a programmatic
//                       dependent of the attempt kernel; waits per chunk of 128 aircraft (DESIGN.md 4.3).
//   fw_reset_kernel   : explicit (masked) reset with optional injected initial states / targets.
//   host side         : handle, launches, host-buffer pipeline (fw_host_*), counters, profiling events.
#include <cuda_runtime.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <new>
#include <vector>
#include "../../include/fwgym.h"
#include "layout.h"
#include "philox.cuh"
#include "dynamics.cuh"
#include "env.cuh"

#define FW_DYN_BLOCK 32
#define FW_DYN_MIN_BLOCKS_F32 16
#define FW_DYN_MIN_BLOCKS 8
#define FW_ENV_BLOCK 128
#define FW_ENV_MIN_BLOCKS 4
#define FW_INIT_BLOCK 64
#define FW_INIT_MIN_BLOCKS 8   // 128 registers: one wave at 65536 envs (1024 blocks on 148 x 8 slots); 4 -> 8: init 18 -> 13 us

enum { CTR_ENV_STEPS = 0, CTR_ATTEMPTS, CTR_ACCEPTED, CTR_WARP_MAX, CTR_WARP_STEPS, CTR_FAILURES, CTR_RESETS, CTR_WATCHDOG, CTR_N };
enum { MS_EPISODES = 0, MS_SUCCESS, MS_RETURN, MS_LENGTH, MS_FAILURES, MS_STEPS_TERM, MS_SUCCESS_TERM, MS_GOAL_STEPS };

struct FwDynEntry;     // kernel instantiation tables ("kernel instantiations" below)
struct FwShapeEntry;

struct fw_handle_s {
  fw_config_t cfg;
  FwLayout L;
  int device;
  int64_t n, offset;
  uint64_t seed;
  double* d;
  int32_t* i;
  unsigned long long* ctr;   // CTR_N
  double* msum;              // FW_N_METRIC_SUMS
  cudaStream_t last_stream;
  int profiling;
  const FwDynEntry* dyn;         // dynamics kernel instantiation (select_kernels)
  int64_t q_len;                 // ints in `queue`: Q_N + chunks
  const int32_t* order;          // fw_debug_set_order
  const FwShapeEntry* shape;     // env / reset kernel instantiation (select_kernels)
  double* ep_out;                // caller's episode-metric buffer (fw_set_episode_out)
  const double* turb_noise;      // caller's injected Dryden noise [4, turb_len, n] (fw_reset), NULL: Philox streams
  int64_t turb_len;
  FwBank bank;                   // attached scenario bank (fw_set_bank; n = 0: none)
  int* err_flag_host;            // mapped pinned word the env kernel raises when a block's chunk wait times out
  int* err_flag_dev;             //   (device alias); non-zero = the handle refuses to step (FW_ERR_WATCHDOG)
  uint32_t spin_limit;           // polls before an env block gives up (fw_debug_watchdog; default ~1 s)
  int starve_next;               // test hook: block 0 of the next step waits for an aircraft that does not exist
  // init -> attempt -> env pipeline (see "dynamics kernels")
  double* carry_d;               // [CY_ROWS][stride]
  int32_t* carry_i;              // [CI_ROWS][stride]
  int32_t* long_list;            // [stride]
  int32_t* queue;                // [Q_N]
  int attempt_grid;              // persistent warps of the attempt kernel (resident capacity of the device)
  double long_div, long_h;       // priority threshold on the initial step size: long_h = dt / long_div
  std::vector<cudaEvent_t> ev;   // 3 events per profiled step: before dyn, between, after env
  // host-buffer pipeline (fw_host_*): `depth` slots of device staging + pinned host result buffers, copy streams
  struct HostSlot {
    float* d_act; float* d_obs; float* d_rew; uint8_t* d_done; int32_t* d_term;   // d_obs .. d_done: ONE block, one D2H copy
    float* h_obs; float* h_rew; uint8_t* h_done; int32_t* h_term;                   // likewise one pinned block
    size_t out_bytes;
    int zero_copy;   // results are written by the env kernel straight into mapped pinned host memory: no D2H copy
    cudaEvent_t e_in, e_step, e_out;
    int busy;
  };
  std::vector<HostSlot> hs;
  cudaStream_t hs_in, hs_out;
  int64_t hs_next;
};

static thread_local char g_err[512] = "";
static int fail(int code, const char* fmt, const char* a = "") {
  snprintf(g_err, sizeof(g_err), fmt, a);
  return code;
}
#define CK(x)                                                                                   \
  do {                                                                                          \
    cudaError_t e_ = (x);                                                                       \
    if (e_ != cudaSuccess) return fail(FW_ERR_CUDA, "CUDA error: %s", cudaGetErrorString(e_)); \
  } while (0)

// sticky watchdog error (fw_env_kernel): the flag lives in mapped pinned memory, so this is a plain host load
static bool poisoned(fw_handle h) { return *reinterpret_cast<volatile int*>(h->err_flag_host) != 0; }
#define CK_POISON(h)                                                                                             \
  do {                                                                                                           \
    if (poisoned(h))                                                                                             \
      return fail(FW_ERR_WATCHDOG, "an env-kernel block gave up waiting for its aircraft (fw_counters().watchdog): "  \
                                   "state of its envs was not advanced; call fw_reset (all envs) or fw_set_state%s", ""); \
  } while (0)

// ----------------------------------------------------------------------------------------------- dynamics kernels
// One env step of the simulator is three launches (DESIGN.md "pipeline"):
//   fw_init_kernel    natural order, one thread per aircraft: action -> commands, f(t0, y0) and scipy's initial step
//                     size (2 RHS evaluations), parked in the carry rows; aircraft that will need many attempts
//                     (tiny first step, e.g. right after a reset) are put on a priority list.
//   fw_attempt_kernel persistent warps (as many as fit the GPU), one aircraft per lane.  Each pass of a warp is ONE
//                     dopri5 step attempt (6 RHS evaluations) for all its lanes; a lane whose aircraft finished its
//                     env step parks the result and adopts the next waiting aircraft (priority list first, then the
//                     natural order), so warps stay full although aircraft need 2..8 attempts.  Attempt boundaries
//                     are the only points where an aircraft changes lanes, so all lanes of a warp are always in the
//                     same dopri5 stage.  Per-aircraft results do not depend on the lane assignment.
//   fw_env_kernel     natural order: PyFly's state commit + the env-side work (below).
enum {
  CY_K0 = 0, CY_KP = CY_K0 + FW_N_KC, CY_H = CY_KP + 3, CY_CMD, CY_RES = CY_CMD + 3,   // RES: 19 rows, final raw y
  CY_ROWS = CY_RES + FW_N_ODE
};
enum { CI_FAIL = 0, CI_ATTEMPTS, CI_ACCEPTED, CI_ROWS };
enum { Q_LONG_COUNT = 0, Q_LONG_CURSOR, Q_NAT_CURSOR, Q_N };
// Behind the Q_N queue counters the same buffer holds one "aircraft finished" counter per chunk of FW_ENV_BLOCK
// consecutive envs (zeroed with the queue at the start of every step).  The env kernel is launched as a programmatic
// dependent of the attempt kernel: its blocks become resident as attempt warps retire and each one waits for ITS chunk
// only, so the env-side work of the early chunks runs in the shadow of the attempt kernel's tail.
#define FW_CHUNK_DONE(q, env) ((q) + Q_N + (int)((env) / FW_ENV_BLOCK))

// Experiment build (-DFW_TIMELINE, scripts/gpu_timeline.py): first block start / last block end of the three kernels of a
// step on the GPU's global timer (ns), read back with fw_debug_timeline.
__device__ unsigned long long fw_timeline_buf[8];   // [6] first env block past its wait, [7] sum of env block run times
#ifdef FW_TIMELINE
__device__ __forceinline__ unsigned long long fw_gtime() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}
#define FW_TL_BEGIN(k) do { if (threadIdx.x == 0) atomicMin(&fw_timeline_buf[2 * (k)], fw_gtime()); } while (0)
#define FW_TL_END(k) do { if (threadIdx.x == 0) atomicMax(&fw_timeline_buf[2 * (k) + 1], fw_gtime()); } while (0)
#else
#define FW_TL_BEGIN(k) do { } while (0)
#define FW_TL_END(k) do { } while (0)
#endif

struct FwDynArgs {
  double* d;
  int32_t* i;
  int64_t stride, n;
  const void* actions;
  int actions_f64;
  unsigned long long* ctr;
  double* cd;          // carry rows [CY_ROWS][stride]
  int32_t* ci;         // carry int rows [CI_ROWS][stride]
  int32_t* long_list;  // [stride] aircraft to start first
  int32_t* q;          // [Q_N + chunks] queue counters + per-chunk finished counters; all zero between steps (fw_init_kernel)
  double long_h;       // initial step sizes below this go on the priority list
  int32_t par_row;     // first per-env model-parameter row of d (FwSpecRand)
  int32_t n_par_rows;
  const int32_t* order;   // experiment hook (fw_debug_set_order): adoption order of the natural queue, NULL = identity
  // ptxas allocates the attempt kernels' registers differently when this block changes size (at 120 or 128 bytes: fp64
  // FwSpecRand 253 -> 254 registers, fp32 FwSpecShipped 127 -> 128, fp32 FwSpecRand spills 60/56 -> 66/68 bytes):
  // padded to the 136 bytes they were tuned at
  int32_t _pad[6];
};
static_assert(sizeof(FwDynArgs) == 136, "see FwDynArgs._pad");

// ---- action -> actuator commands (fixed_wing.py:349-354,439-459; Actuation.set_and_constrain_commands) ----
__device__ __forceinline__ void fw_commands(const fw_sim_t& P, const FwDynArgs& a, const FwEnvCtx& c, double (&cmd)[3]) {
  double act[3];
  if (a.actions_f64) {
    const double* p = reinterpret_cast<const double*>(a.actions) + c.env * 3;
    act[0] = p[0]; act[1] = p[1]; act[2] = p[2];
  } else {
    const float* p = reinterpret_cast<const float*>(a.actions) + c.env * 3;
    act[0] = p[0]; act[1] = p[1]; act[2] = p[2];
  }
  if (P.scale_actions) {
#pragma unroll
    for (int j = 0; j < 3; ++j) {
      double x = act[j];
      if (P.has_scale_low) x = fmax(x, P.scale_low);
      if (P.has_scale_high) x = fmin(x, P.scale_high);
      act[j] = (P.act_to_high[j] - P.act_to_low[j]) * (x - P.scale_low) / (P.scale_high - P.scale_low) + P.act_to_low[j];
    }
  }
  int dummy = 0;
  const double er_c = -1.0 * act[1] + act[0], el_c = act[1] + act[0];
  cmd[0] = fw_cond<double>(P.var[FW_SV_ELEVON_L], FW_SV_ELEVON_L, el_c, dummy);
  cmd[1] = fw_cond<double>(P.var[FW_SV_ELEVON_R], FW_SV_ELEVON_R, er_c, dummy);
  cmd[2] = fw_cond<double>(P.var[FW_SV_THROTTLE], FW_SV_THROTTLE, act[2], dummy);
  c.D(D_CMD + 0) = fw_cond<double>(P.var[FW_SV_ELEVATOR], FW_SV_ELEVATOR, (cmd[1] + cmd[0]) / 2, dummy);
  c.D(D_CMD + 1) = fw_cond<double>(P.var[FW_SV_AILERON], FW_SV_AILERON, (-cmd[1] + cmd[0]) / 2, dummy);
  c.D(D_CMD + 2) = cmd[2];
}

template <typename T>
__device__ __forceinline__ void fw_load_gusts(const fw_sim_t& P, const FwEnvCtx& c, FwStepIn<T>& in) {
#pragma unroll
  for (int j = 0; j < 3; ++j) {
    in.gl[j] = P.turbulence ? (T)c.D(D_GUST + j) : (T)0;
    in.ga[j] = P.turbulence ? (T)c.D(D_GUST + 3 + j) : (T)0;
    in.wind[j] = P.wind_enabled ? (T)c.D(D_WIND + j) : (T)0;
  }
}

template <typename T, class Spec>
__global__ void __launch_bounds__(FW_INIT_BLOCK, FW_INIT_MIN_BLOCKS)
fw_init_kernel(const __grid_constant__ typename FwSimArg<T>::type Px, const FwDynArgs a) {
  const fw_sim_t& P = fw_sim_of(Px);
  FW_TL_BEGIN(0);
  const int64_t env = (int64_t)blockIdx.x * FW_INIT_BLOCK + threadIdx.x;
  const bool valid = env < a.n;
  bool is_long = false, init_failed = false;
  // Queue words are zeroed by the kernels instead of a memset node per step (one launch gap less): the two cursors,
  // which only the attempt kernel uses, here; the priority-list length and the chunk counters by the env kernel of the
  // previous step once it has consumed them (fw_create, a full fw_reset and fw_set_state zero everything).
  // Let the attempt kernel's warps take their places on the SMs as this kernel's blocks retire; they wait for this
  // grid's completion (griddepcontrol.wait) before they read anything
  asm volatile("griddepcontrol.launch_dependents;");
  if (blockIdx.x == 0 && threadIdx.x == 0) { a.q[Q_LONG_CURSOR] = 0; a.q[Q_NAT_CURSOR] = 0; }
  if (valid) {
    FwEnvCtx c{a.d, a.i, a.stride, env};
    double cmd[3];
    fw_commands(P, a, c, cmd);
    FwStepIn<T> in;
#pragma unroll
    for (int j = 0; j < 3; ++j) in.cmd[j] = (T)cmd[j];
    fw_load_gusts<T>(P, c, in);
    T y[FW_N_ODE], f0[FW_N_ODE], h_abs = 0;
#pragma unroll
    for (int j = 0; j < FW_N_ODE; ++j) y[j] = (T)c.D(j);
    const FwPar<T, Spec::rand ? FW_PAR_GLOBAL : FW_PAR_CONST> PP{P, a.d + (int64_t)a.par_row * a.stride + env, a.stride,
                                                                   nullptr};
    int failv = fw_ivp_init<T, Spec>(P, PP, in, y, f0, h_abs);
    if (!failv && !((double)h_abs * 0.0 == 0.0)) failv = FW_TERM_NUMERIC;   // non-finite first step: nothing to integrate
    double* cd = a.cd + env;
    int32_t* ci = a.ci + env;
#pragma unroll
    for (int kc = 0; kc < FW_N_KC; ++kc) cd[(CY_K0 + kc) * a.stride] = (double)f0[fw_kc_to_ode(kc)];
#pragma unroll
    for (int j = 0; j < 3; ++j) { cd[(CY_KP + j) * a.stride] = (double)f0[7 + j]; cd[(CY_CMD + j) * a.stride] = cmd[j]; }
    // Priority start (DESIGN.md 4.4): a tiny first step (the 1e-6 start after a reset).  Membership is carried by the
    // SIGN of the parked step size, so the attempt kernel's natural-order visit can skip list members without a load.
    is_long = !failv && (double)h_abs > 0.0 && (double)h_abs < a.long_h;
    cd[CY_H * a.stride] = is_long ? -(double)h_abs : (double)h_abs;
    ci[CI_FAIL * a.stride] = failv;     // != 0: ConstraintException inside RK45.__init__; nothing left to integrate
    ci[CI_ATTEMPTS * a.stride] = 0;
    ci[CI_ACCEPTED * a.stride] = 0;
    init_failed = failv != 0;
  }
  const unsigned full = 0xffffffffu;
  // aircraft that raised inside RK45.__init__ are finished as far as the env kernel is concerned (a warp's envs are
  // consecutive and FW_ENV_BLOCK is a multiple of 32: one chunk, one atomic)
  const unsigned fm = __ballot_sync(full, valid && init_failed);
  if (fm && (threadIdx.x & 31) == 0) atomicAdd(FW_CHUNK_DONE(a.q, env), __popc(fm));
  // priority list: one atomic per warp
  const unsigned lm = __ballot_sync(full, is_long);
  if (lm) {
    const int lane = threadIdx.x & 31;
    int base = 0;
    if (lane == 0) base = atomicAdd(a.q + Q_LONG_COUNT, __popc(lm));
    base = __shfl_sync(full, base, 0);
    if (is_long) a.long_list[base + __popc(lm & ((1u << lane) - 1u))] = (int32_t)env;
  }
  FW_TL_END(0);
}

// fp32 aircraft need half the registers and half the K-stage shared memory: twice the resident warps
template <typename T, class Spec>
__global__ void __launch_bounds__(FW_DYN_BLOCK, sizeof(T) == 4 ? FW_DYN_MIN_BLOCKS_F32 : FW_DYN_MIN_BLOCKS)
fw_attempt_kernel(const __grid_constant__ typename FwSimArg<T>::type Px, const FwDynArgs a) {
  const fw_sim_t& P = fw_sim_of(Px);
  FW_TL_BEGIN(1);
  extern __shared__ __align__(16) unsigned char smem_raw[];
  FwKStore<T, FW_DYN_BLOCK> K{reinterpret_cast<T*>(smem_raw)};
  // Every warp of this (fully resident) grid is on an SM by now: let the env kernel's blocks queue up behind us.  They
  // synchronise on the per-chunk counters below, not on this kernel's completion.
  asm volatile("griddepcontrol.wait;" ::: "memory");   // the init kernel has completed and its writes are visible
  // (The priority-list length is read first and the release depends on it: env block 0 zeroes it for the next step.)
  const int n_long = a.q[Q_LONG_COUNT];     // final: the init kernel has completed
  asm volatile("griddepcontrol.launch_dependents;" :: "r"(n_long) : "memory");
  const unsigned full = 0xffffffffu;
  const int lane = threadIdx.x & 31;
  const int n_nat = (int)a.n;
  FwIvp<T> S;
  FwStepIn<T> in;
  int64_t env = -1;
  const double* par_base = a.d;   // FwSpecRand: the adopted aircraft's element of parameter row 0
  // FwSpecRand: parameter cache behind the K stages, [n_par_rows][32]
  T* par_cache = reinterpret_cast<T*>(smem_raw) + 6 * FW_N_KC * FW_DYN_BLOCK + threadIdx.x;
  S.status = FW_STATUS_FINISHED;
  S.fail = 0; S.rejected = 0; S.attempts = 0; S.accepted = 0; S.t = 0; S.h_abs = 0;
#pragma unroll
  for (int j = 0; j < FW_N_ODE; ++j) S.y[j] = 0;
#pragma unroll
  for (int j = 0; j < 3; ++j) { S.k0pos[j] = 0; in.cmd[j] = 0; in.gl[j] = 0; in.ga[j] = 0; in.wind[j] = 0; }
  bool long_left = n_long > 0, nat_left = true;
  unsigned long long passes = 0, lane_attempts = 0;
  for (;;) {
    // ---- lanes without an aircraft adopt the next waiting ones (priority list first) ----
    const unsigned idle = __ballot_sync(full, S.status != FW_STATUS_RUNNING);
    if (idle && (long_left || nat_left)) {
      const int want = __popc(idle);
      const int rank = __popc(idle & ((1u << lane) - 1u));
      int got_long = 0, got_nat = 0, base_long = 0, base_nat = 0;
      if (long_left) {
        if (lane == 0) base_long = atomicAdd(a.q + Q_LONG_CURSOR, want);
        base_long = __shfl_sync(full, base_long, 0);
        got_long = min(want, max(0, n_long - base_long));
        if (base_long + want >= n_long) long_left = false;
      }
      if (got_long < want && nat_left) {
        const int need = want - got_long;
        if (lane == 0) base_nat = atomicAdd(a.q + Q_NAT_CURSOR, need);
        base_nat = __shfl_sync(full, base_nat, 0);
        got_nat = min(need, max(0, n_nat - base_nat));
        if (base_nat + need >= n_nat) nat_left = false;
      }
      if (S.status != FW_STATUS_RUNNING) {
        const bool from_long = rank < got_long;
        int64_t e = -1;
        if (from_long) e = a.long_list[base_long + rank];
        else if (rank - got_long < got_nat) {
          e = (int64_t)base_nat + (rank - got_long);
          if (a.order) e = a.order[e];
        }
        env = -1;
        if (e >= 0) {
          const double* cd = a.cd + e;
          const int32_t* ci = a.ci + e;
          const double h0s = cd[CY_H * a.stride];   // negative: on the priority list
          const double h0 = fabs(h0s);
          const int failv = ci[CI_FAIL * a.stride];
          // skipped: aircraft that raised inside RK45.__init__ (the init kernel parked that result), and the
          // natural-order visit of an aircraft that is on the priority list
          const bool skip = failv != 0 || (!from_long && h0s < 0.0);
          // this lane holds no aircraft, so its registers and K slot 0 are free: every load of the candidate is issued
          // before `skip` (which depends on two of them) is known - one dependent L2 round trip less per refill
          {
            par_base = a.d + (int64_t)a.par_row * a.stride + e;
            if constexpr (Spec::rand)
              for (int r = 0; r < a.n_par_rows; ++r) par_cache[r * 32] = (T)par_base[(int64_t)r * a.stride];
            FwEnvCtx c{a.d, a.i, a.stride, e};
#pragma unroll
            for (int j = 0; j < FW_N_ODE; ++j) S.y[j] = (T)c.D(j);
#pragma unroll
            for (int kc = 0; kc < FW_N_KC; ++kc) K.at(0, kc) = (T)cd[(CY_K0 + kc) * a.stride];
#pragma unroll
            for (int j = 0; j < 3; ++j) { S.k0pos[j] = (T)cd[(CY_KP + j) * a.stride]; in.cmd[j] = (T)cd[(CY_CMD + j) * a.stride]; }
            fw_load_gusts<T>(P, c, in);
            S.t = 0; S.h_abs = (T)h0; S.rejected = 0; S.attempts = 0; S.accepted = 0; S.fail = 0;
          }
          if (!skip) {
            env = e;
            S.status = FW_STATUS_RUNNING;
          }
        }
      }
    }
    const unsigned running = __ballot_sync(full, S.status == FW_STATUS_RUNNING);
    if (!running) {
      if (!long_left && !nat_left) break;
      continue;   // everything adopted in this round was a skip; draw again
    }
    // ---- one dopri5 step attempt for every lane that holds an aircraft ----
    ++passes;
    if (S.status == FW_STATUS_RUNNING) {
      ++lane_attempts;
      const FwPar<T, Spec::rand ? FW_PAR_SMEM : FW_PAR_CONST> PP{P, par_base, a.stride, par_cache};
      fw_ivp_attempt<T, Spec, FW_DYN_BLOCK>(P, PP, in, S, K);
      if (S.status != FW_STATUS_RUNNING) {   // env step finished (or raised): park the result for the env kernel
        double* cd = a.cd + env;
        int32_t* ci = a.ci + env;
#pragma unroll
        for (int j = 0; j < FW_N_ODE; ++j) cd[(CY_RES + j) * a.stride] = (double)S.y[j];
        ci[CI_FAIL * a.stride] = S.fail;
        ci[CI_ATTEMPTS * a.stride] = S.attempts;
        ci[CI_ACCEPTED * a.stride] = S.accepted;
        __threadfence();                               // results before the count (release)
        atomicAdd(FW_CHUNK_DONE(a.q, env), 1);
      }
    }
  }
  // ---- counters: warp passes (cost) and lane attempts (useful work) ----
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) lane_attempts += __shfl_xor_sync(full, lane_attempts, o);
  if (lane == 0 && passes) {
    atomicAdd(a.ctr + CTR_WARP_MAX, passes);
    atomicAdd(a.ctr + CTR_WARP_STEPS, lane_attempts);
  }
  FW_TL_END(1);
}

// ---- PyFly._set_states_from_ode_solution(save=True) + airspeed factors + next gust column (env kernel prologue) ----
// PyFly Variable.apply_conditions with the variable's condition FLAGS taken from the shape (a literal in a fixed
// shape: variables without a constraint / clip cost nothing) and the bounds from the runtime configuration.
template <bool WRAP>
__device__ __forceinline__ double fw_cond_s(uint32_t vflags, const fw_var_t& v, int sv, double x, int& fail) {
  if (vflags & (FW_VC_CMIN | FW_VC_CMAX)) {
    const bool bad = (x < v.clo) | (x > v.chi);
    if (bad && !fail) fail = FW_TERM_FAIL_BASE + sv;
  }
  if (vflags & (FW_VC_VMIN | FW_VC_VMAX)) {
    x = x < v.lo ? v.lo : x;     // compares keep NaN, like np.clip
    x = x > v.hi ? v.hi : x;
  }
  if (WRAP && (vflags & FW_VC_WRAP)) {
    const double ax = fabs(x);
    if (ax > CUDART_PI) {   // np.sign(v) * (|v| % pi - pi)
      const double s = x > 0 ? 1.0 : -1.0;
      x = s * (fmod(ax, CUDART_PI) - CUDART_PI);
    }
  }
  return x;
}

template <class SH>
__device__ __forceinline__ void fw_commit_step(const fw_sim_t& P, const FwEnvCtx& c, const double* __restrict__ cd,
                                               const int32_t* __restrict__ ci, int64_t stride, uint32_t k0, uint32_t k1,
                                               uint32_t genv, const FwTurbInject ti, const double* un_pre,
                                               int& attempts_out, int& accepted_out, int tlvl = 0) {
  const fw_sim_t& Ps = SH::sim(P);
#define FW_CS(SV, X) fw_cond_s<false>(Ps.var[SV].flags, P.var[SV], SV, X, failv)
#define FW_CSW(SV, X) fw_cond_s<true>(Ps.var[SV].flags, P.var[SV], SV, X, failv)
  // carry rows: written by the attempt kernel, which may still be running on other chunks -> read past L1 (ld.cg)
  int failv = __ldcg(ci + CI_FAIL * stride);
  attempts_out = __ldcg(ci + CI_ATTEMPTS * stride);
  accepted_out = __ldcg(ci + CI_ACCEPTED * stride);
  if (!failv) {
    double yd[FW_N_ODE];
#pragma unroll
    for (int j = 0; j < FW_N_ODE; ++j) yd[j] = __ldcg(cd + (CY_RES + j) * stride);
    {   // a state that left the representable range ends the episode (FW_TERM_NUMERIC) instead of feeding NaNs back;
        // the checks below keep the first failure and the state rows are only written when there is none
      double chk = 0.0;
#pragma unroll
      for (int j = 0; j < FW_N_ODE; ++j) chk = fma(yd[j], 0.0, chk);
      if (chk != 0.0) failv = FW_TERM_NUMERIC;
    }
    double roll = 0, pitch = 0, yaw = 0, Va = 0, alpha = 0, beta = 0, elev = 0, ail = 0;
    // quaternion / |quaternion|, Euler angles: fwmath routines (asin(x) = atan2(x, sqrt((1 - x)(1 + x))))
    double qn, iqn;
    fwm_sqrt_rsqrt(yd[0] * yd[0] + yd[1] * yd[1] + yd[2] * yd[2] + yd[3] * yd[3], &qn, &iqn);
    const double e0 = yd[0] * iqn, e1 = yd[1] * iqn, e2 = yd[2] * iqn, e3 = yd[3] * iqn;
    yd[0] = e0; yd[1] = e1; yd[2] = e2; yd[3] = e3;
    roll = fwm_atan2(2 * (e0 * e1 + e2 * e3), e0 * e0 + e3 * e3 - e1 * e1 - e2 * e2);
    const double sp = 2 * (e0 * e2 - e1 * e3);
    pitch = fwm_atan2(sp, fwm_sqrt((1 - sp) * (1 + sp)));
    yaw = fwm_atan2(2 * (e0 * e3 + e1 * e2), e0 * e0 + e1 * e1 - e2 * e2 - e3 * e3);
    roll = FW_CSW(FW_SV_ROLL, roll);
    pitch = FW_CSW(FW_SV_PITCH, pitch);
    yaw = FW_CSW(FW_SV_YAW, yaw);
#pragma unroll
    for (int j = 0; j < 9; ++j) yd[4 + j] = FW_CS(FW_SV_OMEGA_P + j, yd[4 + j]);
    yd[13] = FW_CS(FW_SV_ELEVON_L, yd[13]);
    yd[14] = FW_CS(FW_SV_ELEVON_R, yd[14]);
    yd[15] = FW_CS(FW_SV_THROTTLE, yd[15]);
#pragma unroll
    for (int j = 0; j < 3; ++j)
      if (Ps.act_has_dot_max[j]) yd[16 + j] = fmin(fmax(yd[16 + j], -P.act_dot_max[j]), P.act_dot_max[j]);
    ail = FW_CS(FW_SV_AILERON, (-yd[14] + yd[13]) / 2);
    elev = FW_CS(FW_SV_ELEVATOR, (yd[14] + yd[13]) / 2);
    double wb[3] = {0, 0, 0};
    if (Ps.wind_enabled) {
      const double wv[3] = {c.D(D_WIND + 0), c.D(D_WIND + 1), c.D(D_WIND + 2)};
      fw_rot_euler(roll, pitch, yaw, wv, wb);
    }
    double gl[3] = {0, 0, 0};
    if (Ps.turbulence) { gl[0] = c.D(D_GUST + 0); gl[1] = c.D(D_GUST + 1); gl[2] = c.D(D_GUST + 2); }
    const double ur = yd[10] - (wb[0] + gl[0]), vr = yd[11] - (wb[1] + gl[1]), wr = yd[12] - (wb[2] + gl[2]);
    const double hxz2 = ur * ur + wr * wr;
    Va = fwm_sqrt(hxz2 + vr * vr);
    alpha = fwm_atan2(wr, ur);
    beta = fwm_atan2(vr, fwm_sqrt(hxz2));   // asin(vr / Va)
    Va = FW_CS(FW_SV_VA, Va);
    alpha = FW_CS(FW_SV_ALPHA, alpha);
    beta = FW_CS(FW_SV_BETA, beta);
    if (!failv) {
#pragma unroll
      for (int j = 0; j < FW_N_ODE; ++j) c.D(j) = yd[j];
      c.D(D_ROLL) = roll; c.D(D_PITCH) = pitch; c.D(D_YAW) = yaw;
      c.D(D_VA) = Va; c.D(D_ALPHA) = alpha; c.D(D_BETA) = beta;
      c.D(D_ELEV) = elev; c.D(D_AIL) = ail;
      // gust column for the next sim step (cur_sim_step + 1); a mixed handle's level-0 episodes keep their zero gusts
      if (SH::mixed ? tlvl != 0 : Ps.turbulence != 0) {
        double un[4];
        if (ti.noise && ((uint32_t)c.I(I_FLAGS) & FWF_TURB_INJ)) fw_turb_noise_injected(P, ti, c.env, c.I(I_STEPS) + 1, un);
        else if (un_pre) { un[0] = un_pre[0]; un[1] = un_pre[1]; un[2] = un_pre[2]; un[3] = un_pre[3]; }
        else fw_turb_noise<SH::fixed>(P, k0, k1, genv, (uint32_t)c.I(I_EPTICK), c.I(I_STEPS) + 1, un);
        fw_turb_advance<SH>(P, c, un, tlvl);
      }
    }
  }
  c.I(I_STATUS) = failv;
  c.I(I_LASTK) = attempts_out;
#undef FW_CS
#undef FW_CSW
}

// ---------------------------------------------------------------------------------------------------- env kernel
// Observation tile of an env block (dynamic shared memory, only when FwEnvArgs.stage_obs): zero-copy host results write
// observations straight into MAPPED PINNED host memory, and 14 floats per thread at a 56-byte stride would cross PCIe as
// 4-byte writes; staged, a block's rows (contiguous in the output) leave as 16-byte stores, 512 B per warp instruction.
extern __shared__ __align__(16) float fw_env_tile[];

struct FwEnvArgs {
  double* d;
  int32_t* i;
  int64_t n;
  const void* actions;
  int actions_f64;
  uint32_t k0, k1, env_offset;
  float* obs_out;
  float* rew_out;
  uint8_t* done_out;
  int32_t* term_out;
  double* obs64_out;
  double* rew64_out;
  float* term_obs_out;
  int auto_reset;
  int obs_dim;
  unsigned long long* ctr;
  double* msum;
  const double* cd;    // carry rows written by the init / attempt kernels
  const int32_t* ci;
  double* ep_out;      // [N, ep_dim] episode-metric rows (NULL: not requested)
  int ep_dim;
  int32_t* q;          // queue buffer of the dynamics kernels: per-chunk finished counters behind Q_N
  FwTurbInject ti;     // injected Dryden noise of the running episodes (fw_reset turb_noise)
  int* err_flag;       // host-visible sticky error word (watchdog)
  uint32_t spin_limit;
  int32_t starve;      // test hook (fw_debug_watchdog)
  int32_t stage_obs;   // float32 observations through a shared-memory tile (dynamic smem: FW_ENV_BLOCK * obs_dim floats)
  FwBank bank;         // scenario bank (bank shapes only; appended: no earlier parameter moves)
};

// Env-side work of one env step for env `env` (fixed_wing.py:338-437 after the simulator call).  Episode-metric
// contributions are returned in m[] / n_reset and summed per warp by the caller (one atomic per warp and metric).
// Random draws of a step that depend on nothing the integration produces (keyed by counters the previous step left):
// the gust noise of the next sim step and the observation-noise normals.  fw_env_kernel draws them BEFORE it waits for its
// chunk's aircraft, in the shadow of the attempt kernel (Philox + Box-Muller are ~40 % of the env step's instructions).
template <int NZ>
struct FwEnvPre {
  bool have_un;
  int nz;                      // normals drawn: 0 or NZ
  double un[4];                // scaled gust noise of the next sim step
  double z[NZ > 0 ? NZ : 1];   // standard normals of the env stream of this tick
};
// observation-noise normals a fixed shape draws ahead (a 5 x 12 matrix observation would need 120 registers: none)
template <class SH>
__host__ __device__ constexpr int fw_env_nz() {
  if constexpr (SH::fixed) {
    const int n = SH::cenv.obs_noise ? ((SH::cenv.obs_len * SH::cenv.obs_nvar + 1) / 2) * 2 : 0;
    return n <= 16 ? n : 0;
  } else {
    return 0;
  }
}
template <class SH>
__device__ __forceinline__ void fw_env_step(const fw_env_t& E, const fw_sim_t& P, const FwLayout& L, const FwEnvArgs& a,
                                            int64_t env, const FwEnvPre<fw_env_nz<SH>()>& pre,
                                            double (&m)[FW_N_METRIC_SUMS], int& n_reset, int& attempts, int& accepted,
                                            int& failed, bool& need_reset) {
  FW_SHAPE_REFS;
  FwEnvCtx c{a.d, a.i, L.stride, env};
  fw_commit_step<SH>(P, c, a.cd + env, a.ci + env, L.stride, a.k0, a.k1, a.env_offset + (uint32_t)env, a.ti,
                     pre.have_un ? pre.un : nullptr, attempts, accepted, SH::mixed ? c.I(Ls.tl_row + 1) : 0);
  failed = c.I(I_STATUS) != 0;
  uint32_t flags = (uint32_t)c.I(I_FLAGS);
  int steps = c.I(I_STEPS);
  const int status = c.I(I_STATUS);
  double ar[3];
  if (a.actions_f64) {
    const double* p = reinterpret_cast<const double*>(a.actions) + env * 3;
    ar[0] = p[0]; ar[1] = p[1]; ar[2] = p[2];
  } else {
    const float* p = reinterpret_cast<const float*>(a.actions) + env * 3;
    ar[0] = p[0]; ar[1] = p[1]; ar[2] = p[2];
  }
  // history["action"].append(action) happens before the simulator step (fixed_wing.py:345)
  if (Ls.act_depth > 0)
    for (int j = 0; j < 3; ++j) fw_ring_put(c, Ls.act_row, Ls.act_depth, FW_N_ACT, j, steps, ar[j]);
  if (Ls.cmd_depth > 0)
    for (int j = 0; j < 3; ++j) fw_ring_put(c, Ls.cmd_row, Ls.cmd_depth, FW_N_ACT, j, steps, c.D(D_CMD + j));
  steps += 1;
  if (Ls.met) fw_metrics_command(L, c, steps);
  int steps_tgt = c.I(I_STEPS_TGT) + 1;
  c.I(I_STEPS_TGT) = steps_tgt;
  const uint32_t tick = (uint32_t)c.I(I_TICK);
  c.I(I_TICK) = (int32_t)(tick + 1u);
  const uint32_t genv = a.env_offset + (uint32_t)env;
  constexpr int NZ = fw_env_nz<SH>();
  FwEnvRngT<SH::fixed, NZ> rng{FwRng{a.k0, a.k1, genv, tick}, 0u, 0u, 0.0, pre.nz};
  if constexpr (NZ > 0) {
#pragma unroll
    for (int j = 0; j < NZ; ++j) rng.zpre[j] = pre.z[j];
  }

  bool done = false;
  int term = FW_TERM_NONE;
  if (E.steps_max > 0 && steps >= E.steps_max) { done = true; term = FW_TERM_STEPS; }
  double reward;
  int hist_len = c.I(I_HISTLEN);
  // a.stage_obs: float32 observations go to the block's shared-memory tile and leave in one coalesced burst (fw_env_kernel)
  FwObsWriter ow{a.stage_obs ? fw_env_tile : a.obs_out, a.obs64_out, env * (int64_t)a.obs_dim,
                 a.stage_obs ? (int64_t)threadIdx.x * a.obs_dim : (int64_t)-1};
  if (status == 0) {
    const uint32_t gb = fw_goal_status<SH>(E, c);
    bool achieved_on_step = false, resample = false;
    if (Es.streak_req > 0) {
      const int slot = hist_len % Es.streak_req;
      const int wd = slot >> 5, bit = slot & 31;
      uint32_t word = (uint32_t)c.I(I_GOALRING + wd);
      const int oldb = (word >> bit) & 1u, newb = (int)(gb >> 31);
      word = (word & ~(1u << bit)) | ((uint32_t)newb << bit);
      c.I(I_GOALRING + wd) = (int32_t)word;
      const int cnt = c.I(I_GOALCNT) + newb - oldb;
      c.I(I_GOALCNT) = cnt;
      if (newb) m[MS_GOAL_STEPS] += 1.0;
      if (steps_tgt >= Es.streak_req && (double)cnt / (double)Es.streak_req >= E.streak_fraction) {
        achieved_on_step = !(flags & FWF_GOAL_ACHIEVED);
        flags |= FWF_GOAL_ACHIEVED | FWF_EP_SUCCESS;
        // (on_success is a runtime number in every instantiation: env_shapes.h does not compare it)
        if (E.on_success == 1) { done = true; term = FW_TERM_SUCCESS; }
        else if (E.on_success == 2) resample = true;
      }
    }
    if (Ls.met) fw_metrics_goal(E, L, c, gb, hist_len);
    reward = fw_reward<SH>(E, P, L, c, flags, ar, achieved_on_step, steps, hist_len, gb);
    if (resample || (Es.resample_every && steps_tgt >= Es.resample_every)) {
      fw_sample_target<SH>(E, c, rng, flags, steps);
      steps_tgt = 0;
    }
    double nt[FW_MAX_TARGETS];
    fw_next_targets<SH>(E, P, c, flags, steps, steps_tgt, nt);
    fw_loop<SH, FW_CNT(n_targets)>(Es.n_targets, [&](int k) FW_LAMBDA_INLINE {
      c.D(D_TARGET + k) = nt[k];
      if (Ls.tgt_depth > 0) fw_ring_put(c, Ls.tgt_row, Ls.tgt_depth, Es.n_targets, k, hist_len, nt[k]);
      if (Ls.err_depth > 0 || Ls.met) {
        const double err = fw_error(Es.tgt[k].wrap, nt[k], fw_sv<SH>(c, Es.tgt[k].sv));
        if (Ls.err_depth > 0) fw_ring_put(c, Ls.err_row, Ls.err_depth, Es.n_targets, k, hist_len, err);
        if (Ls.met) fw_metrics_error(E, L, c, k, err, hist_len);
      }
    });
    if (Ls.sv_depth > 1)
      fw_loop<SH, FW_CNT(obs_nvar)>(Es.obs_nvar, [&](int v) FW_LAMBDA_INLINE {
        if (Es.obs[v].type == 0)
          fw_ring_put(c, Ls.sv_row, Ls.sv_depth, Ls.n_sv_obs, Ls.sv_slot[v], hist_len, fw_sv<SH>(c, Es.obs[v].ref));
      });
    hist_len += 1;
    c.I(I_HISTLEN) = hist_len;
  } else {
    done = true;
    reward = Es.step_fail_timesteps ? (double)(steps - E.steps_max) : E.step_fail_value;
    term = status;
  }
  c.I(I_STEPS) = steps;
  const bool do_reset = done && a.auto_reset;
  if (!do_reset || a.term_obs_out) {
    // an env that is about to be reset writes its terminal observation (float32 only) to term_obs_out instead
    const FwObsWriter w{do_reset ? a.term_obs_out : ow.o32, do_reset ? nullptr : a.obs64_out, ow.base,
                        do_reset ? (int64_t)-1 : ow.base32};
    fw_observation<SH>(E, P, L, c, rng, flags, steps, hist_len, false, w);
  }
  c.I(I_FLAGS) = (int32_t)flags;
  const double epret = c.D(D_EPRET) + reward;
  c.D(D_EPRET) = epret;
  a.rew_out[env] = (float)reward;
  if (a.rew64_out) a.rew64_out[env] = reward;
  a.done_out[env] = done ? 1 : 0;
  a.term_out[env] = term;
  if (done) {
    if (Ls.met && a.ep_out) fw_metrics_finish(E, P, L, c, hist_len, steps, epret, a.ep_out + env * (int64_t)a.ep_dim);
    m[MS_EPISODES] += 1.0;
    m[MS_RETURN] += epret;
    m[MS_LENGTH] += (double)steps;
    if (flags & FWF_EP_SUCCESS) m[MS_SUCCESS] += 1.0;
    if (term >= FW_TERM_FAIL_BASE) m[MS_FAILURES] += 1.0;
    if (term == FW_TERM_STEPS) m[MS_STEPS_TERM] += 1.0;
    if (term == FW_TERM_SUCCESS) m[MS_SUCCESS_TERM] += 1.0;
  }
  if constexpr (SH::bank) {   // a banked episode ended: its scenario's result rows (never at or beyond n)
    if (done) {
      const int32_t scen = c.I(Ls.bank_row + 1);
      if (scen >= 0) {
        const FwBank& b = a.bank;
        if (scen < b.n) {
          if (b.term) b.term[scen] = term;
          if (b.length) b.length[scen] = steps;
          if (b.ret) b.ret[scen] = epret;
          if (Ls.met && b.episode) fw_metrics_finish(E, P, L, c, hist_len, steps, epret, b.episode + scen * (int64_t)a.ep_dim);
          if (b.episodes) atomicAdd(b.episodes + scen, 1);
          if (b.successes && (flags & FWF_EP_SUCCESS)) atomicAdd(b.successes + scen, 1);
        }
        c.I(Ls.bank_row + 1) = -1;
      }
    }
  }
  if (do_reset) n_reset += 1;
  need_reset = do_reset;   // the reset itself is run by the whole warp together (fw_env_kernel)
}

// per-warp sum of the metric contributions, then one atomic per non-zero metric (all 32 lanes must call)
__device__ __forceinline__ void fw_flush_metrics(const FwEnvArgs& a, double (&m)[FW_N_METRIC_SUMS], int n_reset) {
  const unsigned full = 0xffffffffu;
  bool any = n_reset != 0;
#pragma unroll
  for (int k = 0; k < FW_N_METRIC_SUMS; ++k) any |= m[k] != 0.0;
  if (!__any_sync(full, any)) return;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
#pragma unroll
    for (int k = 0; k < FW_N_METRIC_SUMS; ++k) m[k] += __shfl_xor_sync(full, m[k], o);
    n_reset += __shfl_xor_sync(full, n_reset, o);
  }
  if ((threadIdx.x & 31) == 0) {
#pragma unroll
    for (int k = 0; k < FW_N_METRIC_SUMS; ++k)
      if (m[k] != 0.0) atomicAdd(a.msum + k, m[k]);
    if (n_reset) atomicAdd(a.ctr + CTR_RESETS, (unsigned long long)n_reset);
  }
}

template <class SH>
__global__ void __launch_bounds__(FW_ENV_BLOCK, FW_ENV_MIN_BLOCKS)
fw_env_kernel(const __grid_constant__ fw_env_t E, const __grid_constant__ fw_sim_t P, const __grid_constant__ FwLayout L,
              const __grid_constant__ FwEnvArgs a) {
  const int64_t env = (int64_t)blockIdx.x * FW_ENV_BLOCK + threadIdx.x;
  FW_TL_BEGIN(2);
  // ---- before the wait: this step's random draws (FwEnvPre).  Everything read here was written by the env / reset
  // kernels of EARLIER launches (tick counters), never by the dynamics kernels that may still be running.
  constexpr int NZ = fw_env_nz<SH>();
  FwEnvPre<NZ> pre;
  pre.have_un = false;
  pre.nz = 0;
  if constexpr (SH::fixed) {
    const fw_sim_t& Ps = SH::sim(P);
    if (env < a.n) {
      const uint32_t genv = a.env_offset + (uint32_t)env;
      const int32_t* ip = a.i + env;
      if (Ps.turbulence)
        fw_turb_noise<true>(P, a.k0, a.k1, genv, (uint32_t)ip[(int64_t)I_EPTICK * L.stride], ip[(int64_t)I_STEPS * L.stride] + 1,
                            pre.un);
      if constexpr (NZ > 0) {
        const FwRng g{a.k0, a.k1, genv, (uint32_t)ip[(int64_t)I_TICK * L.stride]};
#pragma unroll
        for (int j = 0; j < NZ / 2; ++j) fw_normal2_inl(g, FW_RS_ENV_N, (uint32_t)j, pre.z[2 * j], pre.z[2 * j + 1]);
      }
    }
    // compile-time for a fixed shape: the draw-in-place paths (fw_commit_step, FwEnvRngT::normal) fold away
    pre.have_un = Ps.turbulence != 0;
    pre.nz = NZ;
  }
  // Wait until every aircraft of this block's chunk has been parked by the dynamics kernels (acquire side of the
  // release in fw_attempt_kernel).  One polling thread per block; the others sleep on the barrier.  The attempt kernel
  // never waits for anything, so this cannot deadlock; the watchdog turns a lost update into an error flag
  // (fw_counters reports it) instead of a hung GPU.
  int timed_out = 0;   // (block-wide OR below: no shared variable, which would turn every access of the kernel generic)
  if (threadIdx.x == 0) {
    const int64_t first = (int64_t)blockIdx.x * FW_ENV_BLOCK;
    int need = (int)((a.n - first) < FW_ENV_BLOCK ? (a.n - first) : FW_ENV_BLOCK);
    if (a.starve && blockIdx.x == 0) need += 1;
    const volatile int32_t* cnt = FW_CHUNK_DONE(a.q, first);
    unsigned spins = 0;
    bool ok = true;
    while (*cnt < need) {
      __nanosleep(256);
      if (++spins > a.spin_limit) { ok = false; break; }
    }
    __threadfence();
    timed_out = ok ? 0 : 1;
    if (ok) {
      // consumed: zero it for the next step (nothing adds to a complete chunk); block 0 also zeroes the priority-list
      // length, which every attempt warp read before this kernel could start
      *FW_CHUNK_DONE(a.q, first) = 0;
      if (blockIdx.x == 0) a.q[Q_LONG_COUNT] = 0;
    } else {
      // Gave up: the carry rows of this chunk may be stale or partial, so NOTHING is committed for its envs, the
      // counter is left alone (late arrivals would corrupt the next step's count) and the handle is poisoned: the host
      // sees the flag and refuses to step until the queue has been re-armed (fw_reset / fw_set_state).
      atomicAdd(a.ctr + CTR_WATCHDOG, 1ull);
      *reinterpret_cast<volatile int*>(a.err_flag) = 1;
      __threadfence_system();
    }
  }
  if (__syncthreads_or(timed_out)) {
    if (env < a.n) {
      const float nanf_ = __int_as_float(0x7fc00000);
      if (a.obs_out) for (int j = 0; j < a.obs_dim; ++j) a.obs_out[env * (int64_t)a.obs_dim + j] = nanf_;
      a.rew_out[env] = nanf_;
      a.done_out[env] = 0;
      a.term_out[env] = -1;
    }
    return;
  }
#ifdef FW_TIMELINE
  const unsigned long long tl_go = fw_gtime();
  if (threadIdx.x == 0) atomicMin(&fw_timeline_buf[6], tl_go);
#endif
  double m[FW_N_METRIC_SUMS];
#pragma unroll
  for (int k = 0; k < FW_N_METRIC_SUMS; ++k) m[k] = 0.0;
  int n_reset = 0, attempts = 0, accepted = 0, failed = 0, nv = 0;
  bool need_reset = false;
  if (env < a.n) { fw_env_step<SH>(E, P, L, a, env, pre, m, n_reset, attempts, accepted, failed, need_reset); nv = 1; }
  // ---- auto-resets, one env at a time, by the WHOLE warp (env.cuh, fw_reset_env<SH, true>): a reset used to be one lane
  // running ~4 500 instructions (60 % of them Philox blocks) while 31 lanes waited, and in the stationary episode mix
  // half of the env blocks contain one (+10 us of mean block run time, profiles/r2_step_timeline.txt).
  {
    const unsigned fullm = 0xffffffffu;
    const int lane = threadIdx.x & 31;
    unsigned rm = __ballot_sync(fullm, need_reset);
    while (rm) {
      const int leader = __ffs((int)rm) - 1;
      rm &= rm - 1u;
      const int64_t env_l = __shfl_sync(fullm, env, leader);
      const int tid_l = (int)(threadIdx.x & ~31u) + leader;
      FwEnvCtx c{a.d, a.i, L.stride, env_l};
      FwObsWriter ow{a.stage_obs ? fw_env_tile : a.obs_out, a.obs64_out, env_l * (int64_t)a.obs_dim,
                     a.stage_obs ? (int64_t)tid_l * a.obs_dim : (int64_t)-1};
      ow.commit = lane == leader;
      if constexpr (SH::bank)
        fw_reset_env_body<SH, true>(E, P, L, c, a.k0, a.k1, a.env_offset + (uint32_t)env_l, nullptr, nullptr, 0,
                                    FwTurbInject{nullptr, 0, 0}, ow, a.bank);
      else
        fw_reset_env_body<SH, true>(E, P, L, c, a.k0, a.k1, a.env_offset + (uint32_t)env_l, nullptr, nullptr, 0,
                                    FwTurbInject{nullptr, 0, 0}, ow);
      __syncwarp();
    }
  }
  if (a.stage_obs) {
    __syncthreads();
    const int64_t first = (int64_t)blockIdx.x * FW_ENV_BLOCK;
    const int nval = (int)((a.n - first) < FW_ENV_BLOCK ? (a.n - first) : FW_ENV_BLOCK);
    const int nfl = nval * a.obs_dim;                 // this block's rows: contiguous floats of obs_out, 512-byte aligned
    float* dst = a.obs_out + first * a.obs_dim;
    const int n4 = nfl >> 2;
    for (int i = threadIdx.x; i < n4; i += FW_ENV_BLOCK)
      reinterpret_cast<float4*>(dst)[i] = reinterpret_cast<const float4*>(fw_env_tile)[i];
    for (int i = (n4 << 2) + threadIdx.x; i < nfl; i += FW_ENV_BLOCK) dst[i] = fw_env_tile[i];
  }
  fw_flush_metrics(a, m, n_reset);
  // dopri5 counters (fw_counters): one atomic per warp
  const unsigned full = 0xffffffffu;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    attempts += __shfl_xor_sync(full, attempts, o);
    accepted += __shfl_xor_sync(full, accepted, o);
    failed += __shfl_xor_sync(full, failed, o);
    nv += __shfl_xor_sync(full, nv, o);
  }
  if ((threadIdx.x & 31) == 0 && nv) {
    atomicAdd(a.ctr + CTR_ENV_STEPS, (unsigned long long)nv);
    atomicAdd(a.ctr + CTR_ATTEMPTS, (unsigned long long)attempts);
    atomicAdd(a.ctr + CTR_ACCEPTED, (unsigned long long)accepted);
    if (failed) atomicAdd(a.ctr + CTR_FAILURES, (unsigned long long)failed);
  }
#ifdef FW_TIMELINE
  __syncthreads();
  if (threadIdx.x == 0) atomicAdd(&fw_timeline_buf[7], fw_gtime() - tl_go);
#endif
  FW_TL_END(2);
}


struct FwResetArgs {
  double* d;
  int32_t* i;
  int64_t n;
  const uint8_t* mask;
  const double* init_state;
  const double* init_target;
  uint32_t k0, k1, env_offset;
  float* obs_out;
  double* obs64_out;
  int obs_dim;
  unsigned long long* ctr;
  FwTurbInject ti;
};
// the explicit reset of a bank shape: the same arguments and the scenario bank (a struct of its own, so that the reset
// kernels of the other shapes keep their parameter block and their code)
struct FwResetBankArgs {
  FwResetArgs r;
  FwBank bank;
};

template <class SH>
__global__ void __launch_bounds__(FW_ENV_BLOCK)
fw_reset_kernel(const __grid_constant__ fw_env_t E, const __grid_constant__ fw_sim_t P, const __grid_constant__ FwLayout L,
                const FwResetArgs a) {
  const int64_t env = (int64_t)blockIdx.x * FW_ENV_BLOCK + threadIdx.x;
  if (env >= a.n) return;
  if (a.mask && !a.mask[env]) return;
  FwEnvCtx c{a.d, a.i, L.stride, env};
  FwObsWriter ow{a.obs_out, a.obs64_out, env * (int64_t)a.obs_dim, -1};
  atomicAdd(a.ctr + CTR_RESETS, 1ull);
  fw_reset_env<SH>(E, P, L, c, a.k0, a.k1, a.env_offset + (uint32_t)env, a.init_state, a.init_target, a.n, a.ti, ow);
}
template <class SH>
__global__ void __launch_bounds__(FW_ENV_BLOCK)
fw_reset_bank_kernel(const __grid_constant__ fw_env_t E, const __grid_constant__ fw_sim_t P,
                     const __grid_constant__ FwLayout L, const FwResetBankArgs ab) {
  const FwResetArgs& a = ab.r;
  const int64_t env = (int64_t)blockIdx.x * FW_ENV_BLOCK + threadIdx.x;
  if (env >= a.n) return;
  if (a.mask && !a.mask[env]) return;
  FwEnvCtx c{a.d, a.i, L.stride, env};
  FwObsWriter ow{a.obs_out, a.obs64_out, env * (int64_t)a.obs_dim, -1};
  atomicAdd(a.ctr + CTR_RESETS, 1ull);
  fw_reset_env_bank<SH>(E, P, L, c, a.k0, a.k1, a.env_offset + (uint32_t)env, a.init_state, a.init_target, a.n, a.ti, ow,
                        ab.bank);
}

// Kernel parameters are limited to 32 764 bytes (CUDA 12.1+ on Volta and later).  The configuration travels as
// __grid_constant__ parameters, so its size is bounded here (the per-level Dryden tables of fw_sim_t count against it);
// 64 bytes cover the alignment padding between the parameters.
static_assert(sizeof(fw_env_t) + sizeof(fw_sim_t) + sizeof(FwLayout) + sizeof(FwEnvArgs) + 64 <= 32764,
              "env kernel parameters exceed the 32 764-byte limit");
static_assert(sizeof(fw_env_t) + sizeof(fw_sim_t) + sizeof(FwLayout) + sizeof(FwResetBankArgs) + 64 <= 32764,
              "reset kernel parameters exceed the 32 764-byte limit");
static_assert(sizeof(FwSimX) + sizeof(FwDynArgs) + 64 <= 32764, "fp32 dynamics kernel parameters exceed the 32 764-byte limit");
static_assert(sizeof(fw_sim_t) + sizeof(FwDynArgs) + 64 <= 32764, "fp64 dynamics kernel parameters exceed the 32 764-byte limit");
// the per-level Dryden tables were appended without moving any later kernel parameter off its 16-byte alignment
static_assert(sizeof(fw_sim_t) % 32 == 24 && sizeof(FwLayout) % 16 == 8, "see fw_sim_t._pad_air / FwLayout._pad_air");

// ---- PID baseline controller (pyfly/pid_controller.py; evaluate_controller.py:141-151) ---------------------------
__global__ void fw_pid_kernel(const double* __restrict__ d, int64_t stride, int64_t n, const fw_pid_gains_t g, double dt,
                              int k_roll, int k_pitch, int k_va, double* __restrict__ integ,
                              const uint8_t* __restrict__ reset_mask, double* __restrict__ actions) {
  const int64_t env = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (env >= n) return;
  auto D = [&](int row) FW_LAMBDA_INLINE { return d[(int64_t)row * stride + env]; };
  double i_va = integ[env], i_roll = integ[n + env], i_pitch = integ[2 * n + env];
  if (reset_mask && reset_mask[env]) i_va = i_roll = i_pitch = 0.0;
  const double e_va = D(D_VA) - D(D_TARGET + k_va);
  const double e_phi = D(D_ROLL) - D(D_TARGET + k_roll);
  const double e_th = D(D_PITCH) - D(D_TARGET + k_pitch);
  i_va = i_va + dt * e_va;
  i_roll = i_roll + dt * e_phi;
  i_pitch = i_pitch + dt * e_th;
  double dt_ = 0.0 - g.k_p_V * e_va - g.k_i_V * i_va;
  double da = -g.k_p_phi * e_phi - g.k_i_phi * i_roll - g.k_d_phi * D(D_OMEGA + 0);
  double de = 0.0 - g.k_p_theta * e_th - g.k_i_theta * i_pitch - g.k_d_theta * D(D_OMEGA + 1);
  dt_ = fmin(fmax(dt_, g.delta_t_min), g.delta_t_max);
  da = fmin(fmax(da, g.delta_a_min), g.delta_a_max);
  de = fmin(fmax(de, g.delta_e_min), g.delta_e_max);
  integ[env] = i_va; integ[n + env] = i_roll; integ[2 * n + env] = i_pitch;
  actions[env * 3 + 0] = de;
  actions[env * 3 + 1] = da;
  actions[env * 3 + 2] = dt_;
}

// ---- state import: [rows_d + rows_i, N] doubles (export: fw_export_rows_kernel) -------------------------------
__global__ void fw_import_kernel(double* d, int32_t* i, int64_t stride, int64_t n, int rows_d, int rows_i,
                                 const double* in) {
  const int64_t env = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (env >= n) return;
  for (int r = 0; r < rows_d; ++r) d[(int64_t)r * stride + env] = in[(int64_t)r * n + env];
  for (int r = 0; r < rows_i; ++r) i[(int64_t)r * stride + env] = (int32_t)(long long)in[(int64_t)(rows_d + r) * n + env];
}
// requested Dryden levels of a mixed handle (fw_set_turbulence_levels); NULL or a value outside -1..3 = -1 (draw)
__global__ void fw_set_levels_kernel(int32_t* row, int64_t n, const int32_t* __restrict__ levels) {
  const int64_t env = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (env >= n) return;
  const int32_t v = levels ? levels[env] : -1;
  row[env] = (v < -1 || v > 3) ? -1 : v;
}
// scenario-bank cursors at attach: bank_next = first + e (mod n when cycling, else at most n), no running scenario
__global__ void fw_bank_attach_kernel(int32_t* next, int32_t* scen, int64_t n_envs, int64_t first, int64_t n_scen,
                                      int cycle) {
  const int64_t env = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (env >= n_envs) return;
  const int64_t c = first + env;
  next[env] = (int32_t)(n_scen <= 0 ? 0 : cycle ? c % n_scen : (c < n_scen ? c : n_scen));
  scen[env] = -1;
}
__global__ void fw_gather_i32_kernel(const int32_t* i, int64_t stride, int64_t n, int row, int32_t* out) {
  const int64_t env = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (env < n) out[env] = i[(int64_t)row * stride + env];
}

// DFMA peak micro-benchmark: 8 independent FMA chains per thread, all SMs, 32 resident warps per SM
__global__ void __launch_bounds__(256) fw_dfma_kernel(double* out, int iters, double seed) {
  double a0 = seed, a1 = seed + 1, a2 = seed + 2, a3 = seed + 3, a4 = seed + 4, a5 = seed + 5, a6 = seed + 6, a7 = seed + 7;
  const double m = 1.0000001, b = 1e-9;
  for (int i = 0; i < iters; ++i) {
#pragma unroll
    for (int u = 0; u < 8; ++u) {
      a0 = fma(a0, m, b); a1 = fma(a1, m, b); a2 = fma(a2, m, b); a3 = fma(a3, m, b);
      a4 = fma(a4, m, b); a5 = fma(a5, m, b); a6 = fma(a6, m, b); a7 = fma(a7, m, b);
    }
  }
  const double s = a0 + a1 + a2 + a3 + a4 + a5 + a6 + a7;
  if (s == 12345.678) out[0] = s;
}

// ------------------------------------------------------------------------------------------------------- host side
static int blocks(int64_t n, int per_block) { return (int)((n + per_block - 1) / per_block); }

// pdl: programmatic dependent launch - the kernel may start while the preceding kernel of the stream is still running
template <typename... P, typename... A>
static cudaError_t launch(void (*kernel)(P...), int grid, int block, size_t smem, cudaStream_t s, bool pdl,
                          const A&... args) {
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[0].val.programmaticStreamSerializationAllowed = 1;
  cudaLaunchConfig_t lc = {};
  lc.gridDim = dim3((unsigned)grid);
  lc.blockDim = dim3((unsigned)block);
  lc.dynamicSmemBytes = smem;
  lc.stream = s;
  lc.attrs = at;
  lc.numAttrs = pdl ? 1 : 0;
  return cudaLaunchKernelEx(&lc, kernel, args...);
}

static int make_layout(const fw_config_t& cfg, int64_t n, FwLayout& L) {
  if (cfg.sim.turb_mixed && !cfg.sim.turbulence)
    return fail(FW_ERR_CONFIG, "per-env turbulence levels (turb_mixed) need turbulence on");
  const int rc = fw_layout_build(cfg.env, cfg.sim.scale_actions, n, L, cfg.sim.turb_mixed);
  if (rc) return fail(FW_ERR_CONFIG, "%s", fw_layout_error(rc));
  // the reset writes aircraft parameters through these tables without checks of its own
  const fw_sim_t& S = cfg.sim;
  const int np = cfg.env.n_par_rows;
  auto row_ok = [&](int s1) { return s1 >= 1 && s1 <= np; };
  bool inertia = false;
  for (int j = 0; j < cfg.env.n_aircraft; ++j) {
    const int id = S.air_id[j];
    const bool live = id >= 0 && id < FW_PAR_N && id != FW_PAR_AR && id < FW_PAR_INV_MASS;
    if (!live && !(id >= FW_AIR_JX && id <= FW_AIR_JXZ))
      return fail(FW_ERR_CONFIG, "aircraft parameters: bad air_id%s", "");
    if (live && !row_ok(S.par_slot1[id])) return fail(FW_ERR_CONFIG, "aircraft parameters: a live entry has no parameter row%s", "");
    inertia |= !live;
  }
  for (int k = 0; k < FW_N_INERTIA; ++k)
    if (S.inertia_slot1[k] ? !(inertia && row_ok(S.inertia_slot1[k])) : inertia)
      return fail(FW_ERR_CONFIG, "aircraft parameters: per-env inertia needs a parameter row for every inertia term%s", "");
  if (cfg.env.n_aircraft && cfg.env.n_rand)
    return fail(FW_ERR_CONFIG, "aircraft parameters together with simulator-parameter randomisation%s", "");
  return FW_OK;
}

// dynamic shared memory of one attempt warp: 6 K stages x 16 components (+ the parameter cache of FwSpecRand)
template <typename T, class Spec>
static int fw_attempt_smem(int n_par_rows) {
  return (6 * FW_N_KC + (Spec::rand ? n_par_rows : 0)) * FW_DYN_BLOCK * (int)sizeof(T);
}

template <typename T, class Spec>
static cudaError_t launch_dyn(const fw_sim_t& sim_in, const FwDynArgs& da, int attempt_grid, cudaStream_t s) {
  typename FwSimArg<T>::type sim;
  if constexpr (sizeof(T) == 8) sim = sim_in;
  else {   // fp32 kernels: the configuration + its float image (dynamics.cuh, FwSimX)
    sim.P = sim_in;
    const double* src = reinterpret_cast<const double*>(&sim_in);
    for (size_t k = 0; k < sizeof(fw_sim_t) / 8; ++k) sim.F.v[k] = (float)src[k];
  }
  fw_init_kernel<T, Spec><<<blocks(da.n, FW_INIT_BLOCK), FW_INIT_BLOCK, 0, s>>>(sim, da);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return e;
  const int warps = blocks(da.n, FW_DYN_BLOCK);
  return launch(fw_attempt_kernel<T, Spec>, warps < attempt_grid ? warps : attempt_grid, FW_DYN_BLOCK,
                (size_t)fw_attempt_smem<T, Spec>(da.n_par_rows), s, true, sim, da);
}
// per device (called from fw_create): opt in to the K-stage shared memory and size the persistent grid
template <typename T, class Spec>
static cudaError_t prepare_dyn(int sm_count, int n_par_rows, int* grid_out) {
  const int smem = fw_attempt_smem<T, Spec>(n_par_rows);
  cudaError_t e = cudaFuncSetAttribute(fw_attempt_kernel<T, Spec>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
  if (e != cudaSuccess) return e;
  int per_sm = 0;
  e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, fw_attempt_kernel<T, Spec>, FW_DYN_BLOCK, smem);
  if (e != cudaSuccess) return e;
  if (grid_out) *grid_out = per_sm * sm_count;
  return cudaSuccess;
}

// ---- kernel instantiations: chosen once per configuration (select_kernels), launched through these entries --------
// name: what fw_kernel_variant reports
struct FwDynEntry {
  const char* name;
  cudaError_t (*launch)(const fw_sim_t& sim, const FwDynArgs& da, int attempt_grid, cudaStream_t s);
  cudaError_t (*prepare)(int sm_count, int n_par_rows, int* grid_out);
};
enum { DYN_SHIPPED = 0, DYN_GENERIC, DYN_RAND };   // dynamics.cuh "kernel specialisation"
#define FW_DYN_ENTRY(T, SPEC, NAME) {NAME, launch_dyn<T, SPEC>, prepare_dyn<T, SPEC>}
static const FwDynEntry kDynKernels[2][3] = {   // [fw_config_t.precision: fp64, fp32][DYN_*]
    {FW_DYN_ENTRY(double, FwSpecShipped, "shipped"), FW_DYN_ENTRY(double, FwSpecGeneric, "generic"),
     FW_DYN_ENTRY(double, FwSpecRand, "rand")},
    {FW_DYN_ENTRY(float, FwSpecShipped, "shipped"), FW_DYN_ENTRY(float, FwSpecGeneric, "generic"),
     FW_DYN_ENTRY(float, FwSpecRand, "rand")}};
#undef FW_DYN_ENTRY

using FwResetKernel = void (*)(fw_env_t, fw_sim_t, FwLayout, FwResetArgs);
using FwResetBankKernel = void (*)(fw_env_t, fw_sim_t, FwLayout, FwResetBankArgs);
struct FwShapeEntry {
  const char* name;
  void (*env)(fw_env_t, fw_sim_t, FwLayout, FwEnvArgs);
  FwResetKernel reset;             // shapes without a bank
  FwResetBankKernel reset_bank;    // bank shapes
};
template <class SH>
constexpr FwShapeEntry fw_shape_entry(const char* name) {
  if constexpr (SH::bank) return {name, fw_env_kernel<SH>, nullptr, fw_reset_bank_kernel<SH>};
  else return {name, fw_env_kernel<SH>, fw_reset_kernel<SH>, nullptr};
}
// FW_SHAPE_LIST in fw_find_shape's order, then the four table-walking instantiations (env_shapes.h)
#define FW_SHAPE_ENTRY(NAME) fw_shape_entry<FwShape_##NAME>(#NAME),
static const FwShapeEntry kShapeKernels[] = {
    FW_SHAPE_LIST(FW_SHAPE_ENTRY)
    fw_shape_entry<FwShapeGeneric>("generic"),
    fw_shape_entry<FwShapeGenericMixed>("generic"),
    fw_shape_entry<FwShapeGenericBank>("generic_bank"),
    fw_shape_entry<FwShapeGenericMixedBank>("generic_bank")};
#undef FW_SHAPE_ENTRY
// first of the four table-walking entries: + 1 mixed, + 2 bank
static constexpr int kShapeGeneric = sizeof(kShapeKernels) / sizeof(kShapeKernels[0]) - 4;

struct FwKernels {
  const FwDynEntry* dyn;
  const FwShapeEntry* shape;
};
// The leanest instantiations that cover this configuration.  FWGYM_FORCE_GENERIC=1 selects the table-walking kernels
// even for a shipped configuration; per-env model parameters still need FwSpecRand.
static FwKernels select_kernels(const fw_config_t& cfg) {
  static const int rank_sv[FW_R_BETA + 1] = {FW_SV_OMEGA_P, FW_SV_OMEGA_Q, FW_SV_OMEGA_R, FW_SV_VEL_U, FW_SV_VEL_V,
                                             FW_SV_VEL_W, FW_SV_ELEVON_L, FW_SV_ELEVON_R, FW_SV_THROTTLE,
                                             FW_SV_AILERON, FW_SV_ELEVATOR, FW_SV_VA, FW_SV_ALPHA, FW_SV_BETA};
  const fw_sim_t& S = cfg.sim;
  const char* force_env = getenv("FWGYM_FORCE_GENERIC");
  const bool force = force_env && force_env[0] == '1';
  bool rand = false;   // per-env model parameters
  for (int i = 0; i < FW_PAR_N; ++i)
    if (S.par_slot1[i]) rand = true;
  for (int k = 0; k < FW_N_INERTIA; ++k)
    if (S.inertia_slot1[k]) rand = true;
  uint32_t clip = 0, cons = 0;
  for (int r = 0; r <= FW_R_BETA; ++r) {
    const uint32_t f = S.var[rank_sv[r]].flags;
    if (f & (FW_VC_VMIN | FW_VC_VMAX)) clip |= FW_RB(r);
    if (f & (FW_VC_CMIN | FW_VC_CMAX)) cons |= FW_RB(r);
  }
  for (int i = 0; i < FW_N_ACT; ++i)
    if (S.act_has_dot_max[i]) clip |= FW_RB(FW_R_AD0 + i);
  const bool shipped_covers = !(clip & ~FwSpecShipped::clip) && !(cons & ~FwSpecShipped::cons) && !S.wind_enabled &&
                              S.drag_model == 0;
  const int spec = rand ? DYN_RAND : (force || !shipped_covers) ? DYN_GENERIC : DYN_SHIPPED;
  const int shape = force ? -1 : fw_find_shape(cfg.env, cfg.sim);
  return {&kDynKernels[cfg.precision != 0][spec],
          &kShapeKernels[shape >= 0 ? shape : kShapeGeneric + (S.turb_mixed != 0) + 2 * (cfg.env.bank_enabled != 0)]};
}

// persistent grid of the handle's attempt kernel: its resident capacity on the device, or FWGYM_ATTEMPT_WARPS_PER_SM
// warps per SM; one warp per SM if the occupancy query reports none
static int size_attempt_grid(fw_handle h) {
  int sms = 0, g = 0;
  CK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, h->device));
  CK(h->dyn->prepare(sms, h->L.n_par_rows, &g));
  const char* e = getenv("FWGYM_ATTEMPT_WARPS_PER_SM");
  if (e && atoi(e) > 0) g = atoi(e) * sms;
  h->attempt_grid = g > 0 ? g : sms;
  return FW_OK;
}

template <typename T>
static bool alloc_zeroed(T** p, size_t count) {
  return cudaMalloc(p, count * sizeof(T)) == cudaSuccess && cudaMemset(*p, 0, count * sizeof(T)) == cudaSuccess;
}

extern "C" {

static void host_free(fw_handle h);

const char* fw_last_error(void) { return g_err; }
int fw_abi_version(void) { return FW_ABI_VERSION; }
int64_t fw_config_sizeof(void) { return (int64_t)sizeof(fw_config_t); }

// buffers and launch choices of a value-initialised handle; on failure fw_create hands the partly built handle to
// fw_destroy
static int init_handle(fw_handle h) {
  int rc = make_layout(h->cfg, h->n, h->L);
  if (rc) return rc;
  const size_t st = (size_t)h->L.stride;
  h->q_len = Q_N + blocks(h->L.stride, FW_ENV_BLOCK);
  if (!alloc_zeroed(&h->d, h->L.d_rows * st) || !alloc_zeroed(&h->i, h->L.i_rows * st) ||
      !alloc_zeroed(&h->ctr, CTR_N) || !alloc_zeroed(&h->msum, FW_N_METRIC_SUMS))
    return fail(FW_ERR_ALLOC, "cudaMalloc failed: %s", cudaGetErrorString(cudaGetLastError()));
  // from here on the kernels keep the queue zeroed (fw_init_kernel)
  if (!alloc_zeroed(&h->carry_d, CY_ROWS * st) || !alloc_zeroed(&h->carry_i, CI_ROWS * st) ||
      !alloc_zeroed(&h->long_list, st) || !alloc_zeroed(&h->queue, (size_t)h->q_len))
    return fail(FW_ERR_ALLOC, "cudaMalloc (carry) failed: %s", cudaGetErrorString(cudaGetLastError()));
  if (cudaHostAlloc(&h->err_flag_host, sizeof(int), cudaHostAllocMapped) != cudaSuccess ||
      cudaHostGetDevicePointer(&h->err_flag_dev, h->err_flag_host, 0) != cudaSuccess)
    return fail(FW_ERR_ALLOC, "cudaHostAlloc (error flag) failed: %s", cudaGetErrorString(cudaGetLastError()));
  *h->err_flag_host = 0;
  if (h->L.n_tl_rows)   // requested levels start at -1: every env draws its level at each reset
    CK(cudaMemset(h->i + (size_t)h->L.tl_row * st, 0xff, st * sizeof(int32_t)));
  if (h->L.n_air_rows)  // aircraft requests start as NaN (all bits set): the nominal aircraft
    CK(cudaMemset(h->d + (size_t)h->L.air_row * st, 0xff, h->L.n_air_rows * st * sizeof(double)));
  // aircraft whose first dopri5 step is below dt / FWGYM_LONG_DIV need the most attempts (e.g. the 1e-6 start after a
  // reset): they are started first so that they do not become the tail of the attempt kernel
  const char* e = getenv("FWGYM_LONG_DIV");
  h->long_div = e ? atof(e) : 32.0;
  h->long_h = h->long_div > 0 ? h->cfg.sim.dt / h->long_div : 0.0;
  const FwKernels k = select_kernels(h->cfg);
  h->dyn = k.dyn;
  h->shape = k.shape;
  return size_attempt_grid(h);
}

int fw_create(const fw_config_t* cfg, int64_t n_envs, int64_t global_env_offset, int device, fw_handle* out) {
  if (!cfg || !out || n_envs <= 0) return fail(FW_ERR_ARG, "fw_create: bad argument");
  if (cfg->abi_version != FW_ABI_VERSION) return fail(FW_ERR_ABI, "fw_create: config ABI version mismatch");
  CK(cudaSetDevice(device));
  fw_handle_s* h = new (std::nothrow) fw_handle_s();
  if (!h) return fail(FW_ERR_ALLOC, "out of host memory");
  h->cfg = *cfg;
  h->device = device;
  h->n = n_envs;
  h->offset = global_env_offset;
  h->spin_limit = 1u << 22;   // x 256 ns: ~1 s
  const int rc = init_handle(h);
  if (rc) { fw_destroy(h); return rc; }
  *out = h;
  return FW_OK;
}

// also frees the partly built handle of a failed fw_create: any of its buffers may still be null
int fw_destroy(fw_handle h) {
  if (!h) return FW_OK;
  cudaSetDevice(h->device);
  cudaFree(h->d); cudaFree(h->i); cudaFree(h->ctr); cudaFree(h->msum);
  cudaFree(h->carry_d); cudaFree(h->carry_i); cudaFree(h->long_list); cudaFree(h->queue);
  if (h->err_flag_host) cudaFreeHost(h->err_flag_host);
  host_free(h);
  for (cudaEvent_t e : h->ev) cudaEventDestroy(e);
  delete h;
  return FW_OK;
}

int fw_seed(fw_handle h, uint64_t seed) {
  if (!h) return fail(FW_ERR_ARG, "null handle");
  h->seed = seed;
  // the per-env draw counters restart with the key (FixedWingAircraft.seed reseeds np_random and the simulator):
  // seed(s) + reset() reproduces the same episodes on a live handle
  CK(cudaSetDevice(h->device));
  CK(cudaMemsetAsync(h->i + (size_t)I_TICK * h->L.stride, 0, (size_t)h->L.stride * sizeof(int32_t), h->last_stream));
  return FW_OK;
}

int fw_set_config(fw_handle h, const fw_config_t* cfg) {
  if (!h || !cfg) return fail(FW_ERR_ARG, "null argument");
  if (cfg->abi_version != FW_ABI_VERSION) return fail(FW_ERR_ABI, "config ABI version mismatch");
  FwLayout L;
  int rc = make_layout(*cfg, h->n, L);
  if (rc) return rc;
  if (L.d_rows != h->L.d_rows || memcmp(&L, &h->L, sizeof(L)) != 0)
    return fail(FW_ERR_CONFIG, "fw_set_config: new config changes the state layout; create a new handle");
  h->cfg = *cfg;
  const FwKernels k = select_kernels(h->cfg);
  h->shape = k.shape;
  if (k.dyn != h->dyn) {
    h->dyn = k.dyn;
    CK(cudaSetDevice(h->device));
    rc = size_attempt_grid(h);
    if (rc) return rc;
  }
  h->long_h = h->long_div > 0 ? h->cfg.sim.dt / h->long_div : 0.0;
  return FW_OK;
}

int64_t fw_num_envs(fw_handle h) { return h ? h->n : 0; }
int fw_obs_dim(fw_handle h) { return h ? h->cfg.env.obs_len * h->cfg.env.obs_nvar : 0; }
int fw_pid_step(fw_handle h, const fw_pid_gains_t* gains, double* integ, const uint8_t* reset_mask, double* actions_out,
                void* stream) {
  if (!h || !gains || !integ || !actions_out) return fail(FW_ERR_ARG, "fw_pid_step: null argument");
  int k_roll = -1, k_pitch = -1, k_va = -1;
  for (int k = 0; k < h->cfg.env.n_targets; ++k) {
    if (h->cfg.env.tgt[k].sv == FW_SV_ROLL) k_roll = k;
    if (h->cfg.env.tgt[k].sv == FW_SV_PITCH) k_pitch = k;
    if (h->cfg.env.tgt[k].sv == FW_SV_VA) k_va = k;
  }
  if (k_roll < 0 || k_pitch < 0 || k_va < 0)
    return fail(FW_ERR_CONFIG, "fw_pid_step: the PID controller needs roll, pitch and Va targets");
  CK(cudaSetDevice(h->device));
  fw_pid_kernel<<<blocks(h->n, 128), 128, 0, (cudaStream_t)stream>>>(h->d, h->L.stride, h->n, *gains, h->cfg.sim.dt,
                                                                     k_roll, k_pitch, k_va, integ, reset_mask, actions_out);
  CK(cudaGetLastError());
  return FW_OK;
}
int fw_episode_dim(fw_handle h) {
  return (h && h->cfg.env.metrics_enabled) ? EP_PER_TARGET + EPT_N * h->cfg.env.n_targets : 0;
}
int fw_set_episode_out(fw_handle h, double* ep_out) {
  if (!h) return fail(FW_ERR_ARG, "null handle");
  if (ep_out && !h->cfg.env.metrics_enabled) return fail(FW_ERR_CONFIG, "fw_set_episode_out: metrics are not enabled in this handle's configuration");
  h->ep_out = ep_out;
  return FW_OK;
}
int fw_launches_per_step(fw_handle h) { return h ? 3 : 0; }
const char* fw_kernel_variant(fw_handle h) {
  static thread_local char buf[96];
  if (!h) return "";
  snprintf(buf, sizeof(buf), "dyn=%s env=%s", h->dyn->name, h->shape->name);
  return buf;
}
int64_t fw_state_rows(fw_handle h) { return h ? h->L.d_rows + h->L.i_rows : 0; }

const char* fw_state_row_name(fw_handle h, int64_t r) {
  static const char* dn[D_FIXED] = {
      "q0", "q1", "q2", "q3", "omega_p", "omega_q", "omega_r", "position_n", "position_e", "position_d", "velocity_u",
      "velocity_v", "velocity_w", "elevon_left", "elevon_right", "throttle", "elevon_left_dot", "elevon_right_dot",
      "throttle_dot", "roll", "pitch", "yaw", "Va", "alpha", "beta", "elevator", "aileron", "cmd_elevator", "cmd_aileron",
      "cmd_throttle", "wind_n", "wind_e", "wind_d", "tx0", "tx1", "tx2", "tx3", "tx4", "tx5", "tx6", "tx7", "tx8", "tx9",
      "tx10", "tx11", "tx12", "tx13", "tx14", "tx15", "tx16", "tx17", "tu0", "tu1", "tu2", "tu3", "gust_u", "gust_v",
      "gust_w", "gust_p", "gust_q", "gust_r", "target0", "target1", "target2", "tslope0", "tslope1", "tslope2", "tamp0",
      "tamp1", "tamp2", "tperiod0", "tperiod1", "tperiod2", "tphase0", "tphase1", "tphase2", "tbias0", "tbias1", "tbias2",
      "prev_shaping0", "prev_shaping1", "prev_shaping2", "err0_0", "err0_1", "err0_2", "episode_return"};
  static const char* in[I_GOALRING + 1] = {"steps_count", "steps_for_target", "hist_len", "rng_tick", "episode_tick",
                                           "flags", "goal_count", "last_attempts", "sim_status", "goal_ring"};
  if (!h || r < 0) return nullptr;
  if (r < D_FIXED) return dn[r];
  if (h->L.n_par_rows > 0 && r >= h->L.par_row && r < h->L.par_row + h->L.n_par_rows) return "param";
  if (h->L.n_rs_rows > 0 && r >= h->L.rs_row && r < h->L.rs_row + h->L.n_rs_rows) return "reward_scaling";
  if (h->L.n_air_rows > 0 && r >= h->L.air_row && r < h->L.air_row + h->L.n_air_rows) return "aircraft_req";
  if (r < h->L.d_rows) return "ring";
  r -= h->L.d_rows;
  if (r < I_GOALRING) return in[r];
  if (h->L.n_tl_rows && r == h->L.tl_row) return "turb_level_req";
  if (h->L.n_tl_rows && r == h->L.tl_row + 1) return "turb_level";
  if (h->L.n_bank_rows && r == h->L.bank_row) return "bank_next";
  if (h->L.n_bank_rows && r == h->L.bank_row + 1) return "bank_scenario";
  if (r < h->L.i_rows) return in[I_GOALRING];
  return nullptr;
}

// A full reset and fw_set_state recover from a watchdog error and re-arm the step queue (the kernels keep it zeroed
// between steps; this covers a step that was abandoned half-way, e.g. after an error)
static int recover_and_rearm(fw_handle h, cudaStream_t s) {
  if (poisoned(h)) {
    CK(cudaDeviceSynchronize());   // nothing of the abandoned step may still be running
    *h->err_flag_host = 0;
  }
  CK(cudaMemsetAsync(h->queue, 0, (size_t)h->q_len * sizeof(int32_t), s));
  return FW_OK;
}

int fw_reset(fw_handle h, const uint8_t* mask, const double* init_state, const double* init_target,
             const double* turb_noise, int64_t turb_len, float* obs_out, double* obs64_out, void* stream) {
  if (!h) return fail(FW_ERR_ARG, "null handle");
  if (turb_noise && turb_len <= 0) return fail(FW_ERR_ARG, "fw_reset: turb_noise needs turb_len > 0");
  CK(cudaSetDevice(h->device));
  cudaStream_t s = (cudaStream_t)stream;
  if (mask) {
    CK_POISON(h);   // only a FULL reset recovers from a watchdog error
  } else {
    const int rc = recover_and_rearm(h, s);
    if (rc) return rc;
  }
  // injected Dryden noise: kept for the episodes that start here (a partial reset without noise keeps the buffer the
  // other envs may still be reading; a full reset without noise drops it)
  if (turb_noise) { h->turb_noise = turb_noise; h->turb_len = turb_len; }
  else if (!mask) { h->turb_noise = nullptr; h->turb_len = 0; }
  FwResetArgs a{h->d, h->i, h->n, mask, init_state, init_target, (uint32_t)h->seed, (uint32_t)(h->seed >> 32),
                (uint32_t)h->offset, obs_out, obs64_out, fw_obs_dim(h), h->ctr,
                FwTurbInject{turb_noise, turb_len, h->n}};
  if (h->shape->reset_bank)
    h->shape->reset_bank<<<blocks(h->n, FW_ENV_BLOCK), FW_ENV_BLOCK, 0, s>>>(h->cfg.env, h->cfg.sim, h->L,
                                                                             FwResetBankArgs{a, h->bank});
  else
    h->shape->reset<<<blocks(h->n, FW_ENV_BLOCK), FW_ENV_BLOCK, 0, s>>>(h->cfg.env, h->cfg.sim, h->L, a);
  CK(cudaGetLastError());
  h->last_stream = s;
  return FW_OK;
}

// stage_obs: obs_out is mapped pinned HOST memory (fw_host_open zero-copy mode): observations leave the env kernel as
// coalesced bursts through a shared-memory tile
static int step_impl(fw_handle h, const void* actions, int actions_f64, float* obs_out, float* rew_out, uint8_t* done_out,
                     int32_t* term_out, double* obs64_out, double* rew64_out, float* term_obs_out, int auto_reset,
                     void* stream, int stage_obs) {
  if (!h || !actions || !rew_out || !done_out || !term_out) return fail(FW_ERR_ARG, "fw_step: null argument");
  if (!obs_out && !obs64_out) return fail(FW_ERR_ARG, "fw_step: no observation buffer");
  CK_POISON(h);
  CK(cudaSetDevice(h->device));
  cudaStream_t s = (cudaStream_t)stream;
  const uint32_t k0 = (uint32_t)h->seed, k1 = (uint32_t)(h->seed >> 32);
  FwDynArgs da{h->d, h->i, h->L.stride, h->n, actions, actions_f64, h->ctr, h->carry_d, h->carry_i, h->long_list,
               h->queue, h->long_h, h->L.par_row, h->L.n_par_rows, h->order};
  cudaEvent_t pe[3] = {nullptr, nullptr, nullptr};
  if (h->profiling) {
    for (int k = 0; k < 3; ++k) { CK(cudaEventCreate(&pe[k])); h->ev.push_back(pe[k]); }
    CK(cudaEventRecord(pe[0], s));
  }
  CK(h->dyn->launch(h->cfg.sim, da, h->attempt_grid, s));
  if (h->profiling) CK(cudaEventRecord(pe[1], s));
  FwEnvArgs ea{h->d, h->i, h->n, actions, actions_f64, k0, k1, (uint32_t)h->offset, obs_out, rew_out, done_out,
               term_out, obs64_out, rew64_out, term_obs_out, auto_reset, fw_obs_dim(h), h->ctr, h->msum, h->carry_d,
               h->carry_i, h->ep_out, fw_episode_dim(h), h->queue, FwTurbInject{h->turb_noise, h->turb_len, h->n},
               h->err_flag_dev, h->spin_limit, h->starve_next,
               (stage_obs && obs_out && (size_t)FW_ENV_BLOCK * fw_obs_dim(h) * sizeof(float) <= 48 * 1024) ? 1 : 0,
               h->bank};
  h->starve_next = 0;
  // a programmatic dependent of the attempt kernel: it synchronises on the per-chunk counters.  With per-kernel
  // profiling on, an event sits between the two kernels, so they are serialised anyway.
  CK(launch(h->shape->env, blocks(h->n, FW_ENV_BLOCK), FW_ENV_BLOCK,
            ea.stage_obs ? (size_t)FW_ENV_BLOCK * ea.obs_dim * sizeof(float) : 0, s, !h->profiling, h->cfg.env,
            h->cfg.sim, h->L, ea));
  if (h->profiling) CK(cudaEventRecord(pe[2], s));
  h->last_stream = s;
  return FW_OK;
}

int fw_step(fw_handle h, const void* actions, int actions_f64, float* obs_out, float* rew_out, uint8_t* done_out,
            int32_t* term_out, double* obs64_out, double* rew64_out, float* term_obs_out, int auto_reset,
            void* stream) {
  return step_impl(h, actions, actions_f64, obs_out, rew_out, done_out, term_out, obs64_out, rew64_out, term_obs_out,
                   auto_reset, stream, 0);
}

// ---- host-buffer stepping ---------------------------------------------------------------------------------------
static void host_free(fw_handle h) {
  for (auto& sl : h->hs) {
    cudaFree(sl.d_act);
    if (!sl.zero_copy) cudaFree(sl.d_obs);
    cudaFreeHost(sl.h_obs);
    if (sl.e_in) cudaEventDestroy(sl.e_in);
    if (sl.e_step) cudaEventDestroy(sl.e_step);
    if (sl.e_out) cudaEventDestroy(sl.e_out);
  }
  if (!h->hs.empty()) { cudaStreamDestroy(h->hs_in); cudaStreamDestroy(h->hs_out); }
  h->hs.clear();
}

// results of a step in one block [obs | reward | termination code | done]: one device -> host copy per step
static void carve_results(float* obs, size_t n, size_t od, float** rew, int32_t** term, uint8_t** done) {
  *rew = obs + n * od;
  *term = reinterpret_cast<int32_t*>(*rew + n);
  *done = reinterpret_cast<uint8_t*>(*term + n);
}

int fw_host_open(fw_handle h, int depth) { return fw_host_open_ex(h, depth, 0); }

int fw_host_open_ex(fw_handle h, int depth, int zero_copy) {
  if (!h || depth < 1 || depth > 8) return fail(FW_ERR_ARG, "fw_host_open: bad argument");
  CK(cudaSetDevice(h->device));
  host_free(h);
  const size_t n = (size_t)h->n, od = (size_t)fw_obs_dim(h);
  CK(cudaStreamCreateWithFlags(&h->hs_in, cudaStreamNonBlocking));
  CK(cudaStreamCreateWithFlags(&h->hs_out, cudaStreamNonBlocking));
  h->hs_next = 0;
  for (int k = 0; k < depth; ++k) {
    fw_handle_s::HostSlot sl = {};
    h->hs.push_back(sl);
    fw_handle_s::HostSlot& r = h->hs.back();
    r.out_bytes = n * (od * sizeof(float) + sizeof(float) + sizeof(int32_t) + 1);
    r.zero_copy = zero_copy ? 1 : 0;
    bool ok = cudaMalloc(&r.d_act, n * FW_N_ACT * sizeof(float)) == cudaSuccess;
    if (ok && zero_copy)    // the device alias of the pinned block is what the env kernel writes
      ok = cudaHostAlloc(&r.h_obs, r.out_bytes, cudaHostAllocMapped) == cudaSuccess &&
           cudaHostGetDevicePointer(&r.d_obs, r.h_obs, 0) == cudaSuccess;
    else if (ok)
      ok = cudaMalloc(&r.d_obs, r.out_bytes) == cudaSuccess && cudaMallocHost(&r.h_obs, r.out_bytes) == cudaSuccess;
    if (!ok ||
        cudaEventCreateWithFlags(&r.e_in, cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&r.e_step, cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&r.e_out, cudaEventDisableTiming) != cudaSuccess) {
      const char* msg = cudaGetErrorString(cudaGetLastError());
      host_free(h);
      return fail(FW_ERR_ALLOC, "fw_host_open: allocation failed: %s", msg);
    }
    carve_results(r.d_obs, n, od, &r.d_rew, &r.d_term, &r.d_done);
    carve_results(r.h_obs, n, od, &r.h_rew, &r.h_term, &r.h_done);
  }
  return FW_OK;
}

int fw_host_close(fw_handle h) {
  if (!h) return FW_OK;
  cudaSetDevice(h->device);
  host_free(h);
  return FW_OK;
}

int fw_host_submit(fw_handle h, const float* actions_host, void* stream, int* slot_out) {
  if (!h || !actions_host || !slot_out) return fail(FW_ERR_ARG, "fw_host_submit: null argument");
  if (h->hs.empty()) return fail(FW_ERR_ARG, "fw_host_submit: call fw_host_open first");
  const int k = (int)(h->hs_next % (int64_t)h->hs.size());
  fw_handle_s::HostSlot& sl = h->hs[k];
  if (sl.busy) return fail(FW_ERR_ARG, "fw_host_submit: every slot is in flight; fw_host_wait the oldest one first");
  CK_POISON(h);
  CK(cudaSetDevice(h->device));
  cudaStream_t s = (cudaStream_t)stream;
  const size_t n = (size_t)h->n, od = (size_t)fw_obs_dim(h);
  CK(cudaMemcpyAsync(sl.d_act, actions_host, n * FW_N_ACT * sizeof(float), cudaMemcpyHostToDevice, h->hs_in));
  CK(cudaEventRecord(sl.e_in, h->hs_in));
  CK(cudaStreamWaitEvent(s, sl.e_in, 0));
  int rc = step_impl(h, sl.d_act, 0, sl.d_obs, sl.d_rew, sl.d_done, sl.d_term, nullptr, nullptr, nullptr, 1, stream,
                     sl.zero_copy);
  if (rc) return rc;
  if (sl.zero_copy) {
    CK(cudaEventRecord(sl.e_out, s));       // the results are in host memory when the env kernel has completed
  } else {
    CK(cudaEventRecord(sl.e_step, s));
    CK(cudaStreamWaitEvent(h->hs_out, sl.e_step, 0));
    CK(cudaMemcpyAsync(sl.h_obs, sl.d_obs, sl.out_bytes, cudaMemcpyDeviceToHost, h->hs_out));
    CK(cudaEventRecord(sl.e_out, h->hs_out));
  }
  sl.busy = 1;
  h->hs_next += 1;
  *slot_out = k;
  return FW_OK;
}

int fw_host_wait(fw_handle h, int slot, const float** obs, const float** rew, const uint8_t** done,
                 const int32_t** term) {
  if (!h || slot < 0 || slot >= (int)h->hs.size()) return fail(FW_ERR_ARG, "fw_host_wait: bad slot");
  fw_handle_s::HostSlot& sl = h->hs[slot];
  if (!sl.busy) return fail(FW_ERR_ARG, "fw_host_wait: slot was not submitted");
  CK(cudaEventSynchronize(sl.e_out));
  sl.busy = 0;
  CK_POISON(h);
  if (obs) *obs = sl.h_obs;
  if (rew) *rew = sl.h_rew;
  if (done) *done = sl.h_done;
  if (term) *term = sl.h_term;
  return FW_OK;
}

int fw_debug_set_order(fw_handle h, const int32_t* order) {
  if (!h) return fail(FW_ERR_ARG, "null handle");
  h->order = order;
  return FW_OK;
}

int fw_debug_timeline(unsigned long long* out8, int reset) {
  if (out8 && cudaMemcpyFromSymbol(out8, fw_timeline_buf, sizeof(unsigned long long) * 8) != cudaSuccess)
    return fail(FW_ERR_CUDA, "timeline read");
  if (reset) {
    const unsigned long long z[8] = {~0ull, 0, ~0ull, 0, ~0ull, 0, ~0ull, 0};
    if (cudaMemcpyToSymbol(fw_timeline_buf, z, sizeof(z)) != cudaSuccess) return fail(FW_ERR_CUDA, "timeline reset");
  }
  return FW_OK;
}

int fw_set_profiling(fw_handle h, int on) {
  if (!h) return fail(FW_ERR_ARG, "null handle");
  h->profiling = on;
  return FW_OK;
}

int fw_profile(fw_handle h, double* dyn_ms, double* env_ms, int64_t* steps) {
  if (!h || !dyn_ms || !env_ms || !steps) return fail(FW_ERR_ARG, "null argument");
  CK(cudaSetDevice(h->device));
  CK(cudaStreamSynchronize(h->last_stream));
  double d = 0, e = 0;
  const size_t n = h->ev.size() / 3;
  for (size_t k = 0; k < n; ++k) {
    float a = 0, b = 0;
    CK(cudaEventElapsedTime(&a, h->ev[3 * k], h->ev[3 * k + 1]));
    CK(cudaEventElapsedTime(&b, h->ev[3 * k + 1], h->ev[3 * k + 2]));
    d += a; e += b;
  }
  for (cudaEvent_t ev : h->ev) cudaEventDestroy(ev);
  h->ev.clear();
  *dyn_ms = d; *env_ms = e; *steps = (int64_t)n;
  return FW_OK;
}

__global__ void fw_export_rows_kernel(const double* d, const int32_t* i, int64_t stride, int64_t n, int rows_d, int64_t row0,
                                      int64_t nrows, double* out) {
  const int64_t env = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (env >= n) return;
  for (int64_t r = 0; r < nrows; ++r) {
    const int64_t row = row0 + r;
    out[r * n + env] = row < rows_d ? d[row * stride + env] : (double)i[(row - rows_d) * stride + env];
  }
}

int fw_get_rows(fw_handle h, int64_t row0, int64_t nrows, double* out, void* stream) {
  if (!h || !out) return fail(FW_ERR_ARG, "null argument");
  if (row0 < 0 || nrows < 0 || row0 + nrows > h->L.d_rows + h->L.i_rows) return fail(FW_ERR_ARG, "fw_get_rows: row range");
  CK(cudaSetDevice(h->device));
  fw_export_rows_kernel<<<blocks(h->n, 256), 256, 0, (cudaStream_t)stream>>>(h->d, h->i, h->L.stride, h->n, h->L.d_rows,
                                                                             row0, nrows, out);
  CK(cudaGetLastError());
  return FW_OK;
}

int fw_debug_watchdog(fw_handle h, uint32_t spin_limit, int starve) {
  if (!h) return fail(FW_ERR_ARG, "null handle");
  h->spin_limit = spin_limit ? spin_limit : (1u << 22);
  h->starve_next = starve;
  return FW_OK;
}

int fw_get_state(fw_handle h, double* out, void* stream) {
  return fw_get_rows(h, 0, fw_state_rows(h), out, stream);
}

int fw_set_state(fw_handle h, const double* in, void* stream) {
  if (!h || !in) return fail(FW_ERR_ARG, "null argument");
  CK(cudaSetDevice(h->device));
  const int rc = recover_and_rearm(h, (cudaStream_t)stream);
  if (rc) return rc;
  fw_import_kernel<<<blocks(h->n, 256), 256, 0, (cudaStream_t)stream>>>(h->d, h->i, h->L.stride, h->n, h->L.d_rows,
                                                                        h->L.i_rows, in);
  CK(cudaGetLastError());
  return FW_OK;
}

int fw_set_turbulence_levels(fw_handle h, const int32_t* levels, void* stream) {
  if (!h) return fail(FW_ERR_ARG, "null handle");
  if (!h->L.n_tl_rows)
    return fail(FW_ERR_ARG, "fw_set_turbulence_levels: the handle flies one turbulence intensity (configure "
                            "turbulence_intensity as {\"values\": [...], \"probabilities\": [...]})");
  CK(cudaSetDevice(h->device));
  fw_set_levels_kernel<<<blocks(h->n, 256), 256, 0, (cudaStream_t)stream>>>(h->i + (size_t)h->L.tl_row * h->L.stride, h->n, levels);
  CK(cudaGetLastError());
  return FW_OK;
}

int fw_set_aircraft(fw_handle h, const double* values, void* stream) {
  if (!h) return fail(FW_ERR_ARG, "null handle");
  if (!h->L.n_air_rows)
    return fail(FW_ERR_ARG, "fw_set_aircraft: the handle has no aircraft parameters (fw_env_t.n_aircraft)%s", "");
  CK(cudaSetDevice(h->device));
  const size_t st = (size_t)h->L.stride;
  double* rows = h->d + (size_t)h->L.air_row * st;
  if (values)
    CK(cudaMemcpy2DAsync(rows, st * sizeof(double), values, (size_t)h->n * sizeof(double), (size_t)h->n * sizeof(double),
                         (size_t)h->L.n_air_rows, cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
  else
    CK(cudaMemsetAsync(rows, 0xff, (size_t)h->L.n_air_rows * st * sizeof(double), (cudaStream_t)stream));
  return FW_OK;
}

int64_t fw_aircraft_dim(fw_handle h) { return h ? h->L.n_air_rows : 0; }

int fw_set_bank(fw_handle h, const fw_bank_t* b, void* stream) {
  if (!h) return fail(FW_ERR_ARG, "null handle");
  if (!h->L.n_bank_rows)
    return fail(FW_ERR_ARG, "fw_set_bank: the handle was not created with a scenario bank (fw_env_t.bank_enabled)%s", "");
  FwBank k{};
  if (b) {
    if (b->n_scenarios <= 0 || b->n_scenarios > INT32_MAX) return fail(FW_ERR_ARG, "fw_set_bank: n_scenarios out of 1..INT32_MAX%s", "");
    if (b->first < 0) return fail(FW_ERR_ARG, "fw_set_bank: first < 0%s", "");
    if (b->stride < h->n) return fail(FW_ERR_ARG, "fw_set_bank: stride < n_envs (two envs could fly one scenario)%s", "");
    if (b->episode && !h->cfg.env.metrics_enabled)
      return fail(FW_ERR_ARG, "fw_set_bank: an episode buffer needs metrics enabled in the configuration%s", "");
    if (b->cycle && (b->term || b->length || b->ret || b->episode))
      return fail(FW_ERR_ARG, "fw_set_bank: a cycling bank has no per-scenario outcome rows (only the counters)%s", "");
    if (b->turb_level && !h->L.n_tl_rows)
      return fail(FW_ERR_ARG, "fw_set_bank: a level column needs a handle with per-env turbulence levels%s", "");
    k = FwBank{b->init_state, b->init_target, b->turb_level, b->n_scenarios, b->stride, b->cycle ? 1 : 0, 0,
               b->term, b->length, b->ret, b->episode, b->episodes, b->successes, nullptr};
  }
  CK(cudaSetDevice(h->device));
  const size_t st = (size_t)h->L.stride;
  fw_bank_attach_kernel<<<blocks(h->n, 256), 256, 0, (cudaStream_t)stream>>>(
      h->i + (size_t)h->L.bank_row * st, h->i + (size_t)(h->L.bank_row + 1) * st, h->n, b ? b->first : 0, k.n, k.cycle);
  CK(cudaGetLastError());
  h->bank = k;
  return FW_OK;
}

int fw_set_bank_aircraft(fw_handle h, const double* aircraft) {
  if (!h) return fail(FW_ERR_ARG, "null handle");
  if (aircraft && !h->L.n_air_rows)
    return fail(FW_ERR_ARG, "fw_set_bank_aircraft: an aircraft column needs a handle with aircraft parameters%s", "");
  if (aircraft && h->bank.n == 0) return fail(FW_ERR_ARG, "fw_set_bank_aircraft: no scenario bank is attached%s", "");
  h->bank.aircraft = aircraft;
  return FW_OK;
}

int fw_last_attempts(fw_handle h, int32_t* out, void* stream) {
  if (!h || !out) return fail(FW_ERR_ARG, "null argument");
  CK(cudaSetDevice(h->device));
  // the carry row, not I_LASTK: an env that finished in the step was reset on the spot (I_LASTK = 0), the carry row still
  // holds the attempts of the step that ended its episode (incl. the attempt a ConstraintException cut short)
  fw_gather_i32_kernel<<<blocks(h->n, 256), 256, 0, (cudaStream_t)stream>>>(h->carry_i, h->L.stride, h->n, CI_ATTEMPTS, out);
  CK(cudaGetLastError());
  return FW_OK;
}

int fw_counters(fw_handle h, fw_counters_t* out) {
  if (!h || !out) return fail(FW_ERR_ARG, "null argument");
  CK(cudaSetDevice(h->device));
  unsigned long long c[CTR_N];
  CK(cudaStreamSynchronize(h->last_stream));
  CK(cudaMemcpy(c, h->ctr, sizeof(c), cudaMemcpyDeviceToHost));
  out->env_steps = c[CTR_ENV_STEPS];
  out->attempts = c[CTR_ATTEMPTS];
  out->accepted = c[CTR_ACCEPTED];
  out->warp_max_attempts = c[CTR_WARP_MAX];
  out->warp_steps = c[CTR_WARP_STEPS];
  out->failures = c[CTR_FAILURES];
  out->resets = c[CTR_RESETS];
  out->rhs_evals = 2 * c[CTR_ENV_STEPS] + 6 * c[CTR_ATTEMPTS];
  out->watchdog = c[CTR_WATCHDOG];
  CK_POISON(h);   // (the counters above are filled in either way)
  return FW_OK;
}

int fw_reset_counters(fw_handle h) {
  if (!h) return fail(FW_ERR_ARG, "null handle");
  CK(cudaSetDevice(h->device));
  CK(cudaStreamSynchronize(h->last_stream));
  CK(cudaMemset(h->ctr, 0, CTR_N * sizeof(unsigned long long)));
  CK(cudaMemset(h->msum, 0, FW_N_METRIC_SUMS * sizeof(double)));
  return FW_OK;
}

int fw_metric_sums(fw_handle h, double* out_host) {
  if (!h || !out_host) return fail(FW_ERR_ARG, "null argument");
  CK(cudaSetDevice(h->device));
  CK(cudaStreamSynchronize(h->last_stream));
  CK(cudaMemcpy(out_host, h->msum, FW_N_METRIC_SUMS * sizeof(double), cudaMemcpyDeviceToHost));
  return FW_OK;
}

int fw_dfma_peak(int device, double* flops_out, double* ms_out) {
  if (!flops_out) return fail(FW_ERR_ARG, "null argument");
  CK(cudaSetDevice(device));
  cudaDeviceProp prop;
  CK(cudaGetDeviceProperties(&prop, device));
  double* d;
  CK(cudaMalloc(&d, 8));
  const int blocks = prop.multiProcessorCount * 4, threads = 256, iters = 4096;
  cudaEvent_t e0, e1;
  CK(cudaEventCreate(&e0));
  CK(cudaEventCreate(&e1));
  fw_dfma_kernel<<<blocks, threads>>>(d, 64, 1.0);   // warm-up
  float best = 1e30f;
  for (int rep = 0; rep < 5; ++rep) {
    CK(cudaEventRecord(e0));
    fw_dfma_kernel<<<blocks, threads>>>(d, iters, 1.0);
    CK(cudaEventRecord(e1));
    CK(cudaEventSynchronize(e1));
    float ms;
    CK(cudaEventElapsedTime(&ms, e0, e1));
    best = ms < best ? ms : best;
  }
  CK(cudaGetLastError());
  const double fl = 2.0 * 64.0 * (double)iters * (double)blocks * (double)threads;
  *flops_out = fl / (best * 1e-3);
  if (ms_out) *ms_out = best;
  cudaEventDestroy(e0); cudaEventDestroy(e1); cudaFree(d);
  return FW_OK;
}

}  // extern "C"
