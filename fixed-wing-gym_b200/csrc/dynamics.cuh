// 6-DOF Skywalker-X8 right-hand side and scipy-RK45-equivalent adaptive dopri5 driver, one thread per aircraft.
//
// What it replaces (SURVEY §8a): PyFly.step / PyFly._dynamics / _forces / _f_* (pyfly 0.1.2, restated in
// oracle/pyfly_restated.py) and scipy.integrate.solve_ivp(RK45) (scipy/integrate/_ivp/rk.py:14-176,
// common.py:63-134, base.py:179-210) as called once per env step from fixed_wing.py:358.
#pragma once
#include <math_constants.h>
#include "layout.h"
#include "fwmath.cuh"

#define FW_STATUS_RUNNING 0
#define FW_STATUS_FINISHED 1
#define FW_STATUS_TOO_SMALL 2
// Hang guard: a healthy env step takes 2..10 attempts; the worst finite case observed (a sideways-sliding aircraft
// sitting on the atan2(w, u) singularity of alpha, turbulence off) 4 300.  Beyond the guard are only states that have
// left physics (unconstrained body rates of 1e150 rad/s: step sizes of 1e-17 s, i.e. 1e15 attempts in scipy).
#define FW_MAX_ATTEMPTS 20000

template <typename T> struct FwMath;
// fp64: the branch-free routines of fwmath.cuh (straight-line, Estrin polynomials, constant-bank coefficients) so
// that ptxas can interleave the independent chains of one right-hand side.  sincos stays libdevice: it is only
// reached when alpha/beta carry a clip (not in any shipped configuration).
template <> struct FwMath<double> {
  static __device__ __forceinline__ double sqrt_(double x) { return fwm_sqrt(x); }
  static __device__ __forceinline__ void sqrt_rsqrt(double x, double* s, double* rs) { fwm_sqrt_rsqrt(x, s, rs); }
  static __device__ __forceinline__ double exp_(double x) { return fwm_exp(x); }
  static __device__ __forceinline__ double atan2_(double y, double x) { return fwm_atan2(y, x); }
  static __device__ __forceinline__ double pow_(double x, double y) { return fwm_pow(x, y); }
  static __device__ __forceinline__ double div_(double a, double b) { return fwm_div(a, b); }
  static __device__ __forceinline__ double rcp_(double x) { return fwm_rcp(x); }
  static __device__ __forceinline__ void sincos_(double x, double* s, double* c) { sincos(x, s, c); }
  // nextafter(x, +inf) for finite x >= 0 (the integrator's t)
  static __device__ __forceinline__ double next_up(double x) { return __longlong_as_double(__double_as_longlong(x) + 1); }
};
// fp32 (opt-in mode, reported separately from the fp64 parity claim): hardware approximations (MUFU.RCP / RSQ / EX2 /
// LG2, ~1-2 ulp) and a straight-line atan2 — no libdevice slow paths, so the right-hand side stays one basic block
// like the fp64 one.  Inputs are finite physical numbers; zero arguments of sqrt / atan2 are handled.
template <> struct FwMath<float> {
  static __device__ __forceinline__ float rcp_(float x) { float r; asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x)); return r; }
  static __device__ __forceinline__ float sqrt_(float x) { float r; asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x)); return r; }
  static __device__ __forceinline__ void sqrt_rsqrt(float x, float* s, float* rs) {
    float r;
    asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    *rs = r;
    *s = x > 0.0f ? x * r : 0.0f;
  }
  static __device__ __forceinline__ float exp_(float x) { return __expf(x); }
  static __device__ __forceinline__ float div_(float a, float b) { return a * rcp_(b); }
  static __device__ __forceinline__ float pow_(float x, float y) { return __powf(x, y); }
  // atan(t) = t * R(t^2) on [0, 1] (degree 8, max abs error 1.1e-7), octant / quadrant fix-ups by selects
  static __device__ __forceinline__ float atan2_(float y, float x) {
    const float ax = fabsf(x), ay = fabsf(y);
    const float mx = fmaxf(ax, ay), mn = fminf(ax, ay);
    const float t = mx > 0.0f ? mn * rcp_(mx) : 0.0f;
    const float z = t * t, z2 = z * z, z4 = z2 * z2;
    const float p01 = fmaf(-0.3333306610584259f, z, 1.0f), p23 = fmaf(-0.14202570915222168f, z, 0.19992484152317047f);
    const float p45 = fmaf(-0.07495445758104324f, z, 0.10636754333972931f);
    const float p67 = fmaf(-0.016005029901862144f, z, 0.042587608098983765f);
    const float lo = fmaf(p23, z2, p01), hi = fmaf(p67, z2, p45);
    float r = t * fmaf(fmaf(0.0028340641874819994f, z4, hi), z4, lo);
    r = ay > ax ? 1.5707963267948966f - r : r;
    r = x < 0.0f ? 3.141592653589793f - r : r;
    return copysignf(r, y);
  }
  static __device__ __forceinline__ void sincos_(float x, float* s, float* c) { sincosf(x, s, c); }
  static __device__ __forceinline__ float next_up(float x) { return __int_as_float(__float_as_int(x) + 1); }
};

// ---- fp32 kernels read the model's numbers as FLOATS ----
// fw_sim_t holds doubles; converting one at its point of use is an F2F.F32.F64 (FP64 pipe) per read, ~190 per attempt
// body.  An fp32 dynamics kernel therefore receives FwSimX = the configuration + a float image of it: element k of the
// image is the float value of the k-th 8-byte slot of fw_sim_t (slots that are not doubles hold garbage and are never
// read).  fw_rd<T>(P, P.field) returns the field itself for double and the image element for float; after inlining
// both are constant-bank operands at fixed offsets of the kernel parameter.  P must be the FwSimX's own member.
struct FwSimF { float v[sizeof(fw_sim_t) / 8]; };
struct FwSimX { fw_sim_t P; FwSimF F; };
static_assert(sizeof(fw_sim_t) % 8 == 0, "fw_sim_t must be a whole number of 8-byte slots");
template <typename T> struct FwSimArg { typedef fw_sim_t type; };
template <> struct FwSimArg<float> { typedef FwSimX type; };
__device__ __forceinline__ const fw_sim_t& fw_sim_of(const fw_sim_t& p) { return p; }
__device__ __forceinline__ const fw_sim_t& fw_sim_of(const FwSimX& p) { return p.P; }
template <typename T>
__device__ __forceinline__ T fw_rd(const fw_sim_t& P, const double& field) {
  if constexpr (sizeof(T) == 8) return field;
  else return reinterpret_cast<const FwSimX*>(&P)->F.v[&field - reinterpret_cast<const double*>(&P)];
}

// PyFly Variable.apply_conditions: constraint check -> clip -> (wrap).  `fail` keeps the FIRST violated variable.
// The host stores every missing bound as +-inf (lo/hi for the clip, clo/chi for the constraint), so the body is
// branch-free compares/selects; variables without any condition skip it on one warp-uniform test.
template <typename T>
__device__ __forceinline__ T fw_cond(const fw_var_t& v, int sv, T x, int& fail) {
  if (v.flags == 0u) return x;
  const bool bad = (x < (T)v.clo) | (x > (T)v.chi);
  if (bad && !fail) fail = FW_TERM_FAIL_BASE + sv;
  x = x < (T)v.lo ? (T)v.lo : x;     // compares keep NaN, like np.clip
  x = x > (T)v.hi ? (T)v.hi : x;
  return x;
}

// + the wrap of angle variables (roll, yaw); only needed when a state is stored, never inside the RHS
template <typename T>
__device__ __forceinline__ T fw_cond_wrap(const fw_var_t& v, int sv, T x, int& fail) {
  x = fw_cond<T>(v, sv, x, fail);
  if (v.flags & FW_VC_WRAP) {
    T ax = fabs(x);
    if (ax > (T)CUDART_PI) {   // np.sign(v) * (|v| % pi - pi)
      T s = x > 0 ? (T)1 : (T)-1;
      x = s * (fmod(ax, (T)CUDART_PI) - (T)CUDART_PI);
    }
  }
  return x;
}

// per-step inputs that are constant during one env step
template <typename T> struct FwStepIn {
  T cmd[3];      // constrained setpoints for elevon_left, elevon_right, throttle
  T gl[3];       // linear gust (body); zero when turbulence is off
  T ga[3];       // angular gust; zero when turbulence is off
  T wind[3];     // steady wind NED
};

// ---- kernel specialisation -------------------------------------------------------------------------------------
// Every conditioned variable of the right-hand side has a RANK = its position in PyFly's evaluation order (the first
// violated one names the failure).  A kernel instantiation carries two compile-time rank masks: which variables it
// clips and which it constraint-checks.  Doing MORE than a configuration asks for is harmless (absent bounds are
// +-inf), so the host picks the leanest instantiation whose masks cover the configuration's:
//   FwSpecShipped : what every shipped fixed_wing_config*.json needs (constraints on omega_p/q/r and Va, clips on Va,
//                   the elevons, throttle, elevator, aileron and the elevon rates), no steady wind, induced drag.
//                   The RHS body is one straight-line block.
//   FwSpecGeneric : every variable, runtime wind / drag-model switches.
enum {
  FW_R_P = 0, FW_R_Q, FW_R_R, FW_R_U, FW_R_V, FW_R_W, FW_R_EL, FW_R_ER, FW_R_TH, FW_R_AIL, FW_R_ELEV, FW_R_VA,
  FW_R_ALPHA, FW_R_BETA, FW_R_AD0, FW_R_AD1, FW_R_AD2, FW_R_N
};
#define FW_RB(r) (1u << (r))
__constant__ int c_rank_sv[FW_R_BETA + 1] = {FW_SV_OMEGA_P, FW_SV_OMEGA_Q, FW_SV_OMEGA_R, FW_SV_VEL_U, FW_SV_VEL_V,
                                             FW_SV_VEL_W, FW_SV_ELEVON_L, FW_SV_ELEVON_R, FW_SV_THROTTLE,
                                             FW_SV_AILERON, FW_SV_ELEVATOR, FW_SV_VA, FW_SV_ALPHA, FW_SV_BETA};
struct FwSpecShipped {
  static constexpr uint32_t clip = FW_RB(FW_R_EL) | FW_RB(FW_R_ER) | FW_RB(FW_R_TH) | FW_RB(FW_R_AIL) |
                                   FW_RB(FW_R_ELEV) | FW_RB(FW_R_VA) | FW_RB(FW_R_AD0) | FW_RB(FW_R_AD1);
  static constexpr uint32_t cons = FW_RB(FW_R_P) | FW_RB(FW_R_Q) | FW_RB(FW_R_R) | FW_RB(FW_R_VA);
  static constexpr bool generic = false;
  static constexpr bool rand = false;
};
struct FwSpecGeneric {
  static constexpr uint32_t clip = 0xffffffffu, cons = 0xffffffffu;
  static constexpr bool generic = true;
  static constexpr bool rand = false;
};
//   FwSpecRand    : FwSpecGeneric + model parameters that differ per aircraft (simulator-parameter randomisation,
//                   fixed_wing.py:523-570): every live parameter is read through FwPar below.
struct FwSpecRand {
  static constexpr uint32_t clip = 0xffffffffu, cons = 0xffffffffu;
  static constexpr bool generic = true;
  static constexpr bool rand = true;
};

// ---- live model parameters ---------------------------------------------------------------------------------------
// (fw_par id, fw_sim_t field).  PyFly reads these from its params dict / attributes at every RHS evaluation, so
// FixedWingAircraft.sample_simulator_parameters can change them per episode.  RAND = false: the shared value, a
// constant-bank operand.  RAND = true: parameters the configuration randomises live in per-env rows
// (P.par_slot1[id] - 1, a warp-uniform test per read); the others still come from the constant bank.
#define FW_LIVE_PARAMS(X)                                                                                             \
  X(MASS, mass) X(S_WING, S_wing) X(B, b) X(C, c) X(S_PROP, S_prop) X(K_MOTOR, k_motor) X(K_T_P, k_T_P)               \
  X(K_OMEGA, k_Omega) X(C_PROP, C_prop) X(E, e) X(M, M) X(A_0, a_0) X(AR, ar)                                         \
  X(C_L_0, C_L_0) X(C_L_ALPHA, C_L_alpha) X(C_L_Q, C_L_q) X(C_L_DELTA_E, C_L_delta_e)                                 \
  X(C_D_P, C_D_p) X(C_D_0, C_D_0) X(C_D_ALPHA1, C_D_alpha1) X(C_D_ALPHA2, C_D_alpha2) X(C_D_BETA1, C_D_beta1)         \
  X(C_D_BETA2, C_D_beta2) X(C_D_Q, C_D_q) X(C_D_DELTA_E, C_D_delta_e)                                                 \
  X(C_M_0, C_m_0) X(C_M_ALPHA, C_m_alpha) X(C_M_Q, C_m_q) X(C_M_DELTA_E, C_m_delta_e) X(C_M_FP, C_m_fp)               \
  X(C_Y_0, C_Y_0) X(C_Y_BETA, C_Y_beta) X(C_Y_P, C_Y_p) X(C_Y_R, C_Y_r) X(C_Y_DELTA_A, C_Y_delta_a)                   \
  X(C_Y_DELTA_R, C_Y_delta_r)                                                                                         \
  X(C_L_ROLL_0, C_l_0) X(C_L_ROLL_BETA, C_l_beta) X(C_L_ROLL_P, C_l_p) X(C_L_ROLL_R, C_l_r)                           \
  X(C_L_ROLL_DELTA_A, C_l_delta_a) X(C_L_ROLL_DELTA_R, C_l_delta_r)                                                   \
  X(C_N_0, C_n_0) X(C_N_BETA, C_n_beta) X(C_N_P, C_n_p) X(C_N_R, C_n_r) X(C_N_DELTA_A, C_n_delta_a)                   \
  X(C_N_DELTA_R, C_n_delta_r)                                                                                         \
  X(RHO, rho) X(G, g) X(INV_MASS, inv_mass) X(INV_PI_E_AR, inv_pi_e_ar) X(EXP_2MA0, exp_2Ma0)
static_assert(FW_PAR_N == FW_N_PAR, "FW_N_PAR in fwgym.h must equal the number of fw_par ids");

// Three sources, chosen per kernel:
//   FW_PAR_CONST  the shared value: a constant-bank operand (every instantiation but FwSpecRand);
//   FW_PAR_GLOBAL the per-env row in HBM for randomised parameters (init kernel: two evaluations per aircraft);
//   FW_PAR_SMEM   the attempt kernel reads every parameter 6 times per pass inside a latency-bound dependency chain, so
//                 it copies the adopted aircraft's parameter rows to shared memory ([row][lane]) at adoption and reads
//                 them branch-free: 50 warp-uniform branches per RHS would cut it into basic blocks that cannot
//                 overlap; an unconditional shared-memory read + select keeps it one block.
enum { FW_PAR_CONST = 0, FW_PAR_GLOBAL = 1, FW_PAR_SMEM = 2 };
template <typename T, int MODE> struct FwPar {
  const fw_sim_t& P;
  const double* base;   // GLOBAL: this aircraft's element of parameter row 0
  int64_t stride;
  const T* cache;       // SMEM: this lane's element of cached row 0 (32 lanes per row)
#define FW_PAR_GETTER(ID, F)                                                      \
  __device__ __forceinline__ T F() const {                                        \
    if constexpr (MODE == FW_PAR_GLOBAL) {                                        \
      const int s1 = P.par_slot1[FW_PAR_##ID];                                    \
      if (s1) return (T)base[(int64_t)(s1 - 1) * stride];                         \
    }                                                                             \
    if constexpr (MODE == FW_PAR_SMEM) {                                          \
      const int s1 = P.par_slot1[FW_PAR_##ID];                                    \
      const T v = cache[(s1 > 0 ? s1 - 1 : 0) * 32];                              \
      return s1 > 0 ? v : fw_rd<T>(P, P.F);                                       \
    }                                                                             \
    return fw_rd<T>(P, P.F);                                                      \
  }
  FW_LIVE_PARAMS(FW_PAR_GETTER)
#undef FW_PAR_GETTER
};

// branch-free condition of the variable of rank R: violated constraints set bit R of failmask.  RAW: no condition
// at all (see fw_rhs).
template <typename T, class Spec, int R, bool RAW = false>
__device__ __forceinline__ T fw_cond_r(const fw_sim_t& P, const fw_var_t& v, T x, uint32_t& failmask) {
  if constexpr (RAW) return x;
  if constexpr ((Spec::cons >> R) & 1u) {
    const bool bad = (x < fw_rd<T>(P, v.clo)) | (x > fw_rd<T>(P, v.chi));
    failmask |= bad ? FW_RB(R) : 0u;
  }
  if constexpr ((Spec::clip >> R) & 1u) {
    const T lo = fw_rd<T>(P, v.lo), hi = fw_rd<T>(P, v.hi);
    x = x < lo ? lo : x;     // compares keep NaN, like np.clip
    x = x > hi ? hi : x;
  }
  return x;
}

// d/dt of the 19-state vector.  y is the RAW trial state; PyFly conditions every component (clip / constraint) before
// use except the quaternion, which is used un-normalised (oracle/pyfly_restated.py: _dynamics, _forces).
//
// RAW = the evaluation at t == 0: PyFly._dynamics only writes the trial state into its Variables (and thereby applies
// their conditions) `if t > 0`; f(t0, y0) is computed from the stored values as they are.  Those are already
// conditioned after a step, but NOT after a reset (Variable.reset draws init values without clipping or checking), so
// the first right-hand side of an episode must not clip / check the state variables.  Va, alpha, beta (and the
// elevator / aileron mapping) are conditioned in _forces at every evaluation.
template <typename T, class Spec, bool RAW = false, class PAR>
__device__ __forceinline__ void fw_rhs(const fw_sim_t& P, const PAR& PP, const FwStepIn<T>& in,
                                       const T (&y)[FW_N_ODE], T (&dy)[FW_N_ODE], uint32_t& failmask) {
  typedef FwMath<T> Mt;
  const T e0 = y[0], e1 = y[1], e2 = y[2], e3 = y[3];
  const T p = fw_cond_r<T, Spec, FW_R_P, RAW>(P, P.var[FW_SV_OMEGA_P], y[4], failmask);
  const T q = fw_cond_r<T, Spec, FW_R_Q, RAW>(P, P.var[FW_SV_OMEGA_Q], y[5], failmask);
  const T r = fw_cond_r<T, Spec, FW_R_R, RAW>(P, P.var[FW_SV_OMEGA_R], y[6], failmask);
  // position variables carry no limits (config.py rejects them): their stage states are never formed
  const T u = fw_cond_r<T, Spec, FW_R_U, RAW>(P, P.var[FW_SV_VEL_U], y[10], failmask);
  const T v = fw_cond_r<T, Spec, FW_R_V, RAW>(P, P.var[FW_SV_VEL_V], y[11], failmask);
  const T w = fw_cond_r<T, Spec, FW_R_W, RAW>(P, P.var[FW_SV_VEL_W], y[12], failmask);
  // actuators: value conditions + rate clip (ControlVariable.apply_conditions)
  const T el = fw_cond_r<T, Spec, FW_R_EL, RAW>(P, P.var[FW_SV_ELEVON_L], y[13], failmask);
  const T er = fw_cond_r<T, Spec, FW_R_ER, RAW>(P, P.var[FW_SV_ELEVON_R], y[14], failmask);
  const T th = fw_cond_r<T, Spec, FW_R_TH, RAW>(P, P.var[FW_SV_THROTTLE], y[15], failmask);
  T ad[3] = {y[16], y[17], y[18]};
#pragma unroll
  for (int i = 0; i < 3; ++i)
    if (!RAW && ((Spec::clip >> (FW_R_AD0 + i)) & 1u)) {
      // two selects (compares keep NaN), never a branch: nvcc turned the nested conditional into a BSSY / BRA / BSYNC
      // region per actuator and stage (~40 issue cycles each for a lone warp); identical values for m >= 0
      const T m = P.act_has_dot_max[i] ? fw_rd<T>(P, P.act_dot_max[i]) : (T)CUDART_INF;
      const T nm = -m;
      T x = ad[i];
      x = x < nm ? nm : x;
      x = x > m ? m : x;
      ad[i] = x;
    }
  const T ail = fw_cond_r<T, Spec, FW_R_AIL>(P, P.var[FW_SV_AILERON], (-er + el) * (T)0.5, failmask);
  const T elev = fw_cond_r<T, Spec, FW_R_ELEV>(P, P.var[FW_SV_ELEVATOR], (er + el) * (T)0.5, failmask);
  const T rud = (T)0;

  // ---- airspeed factors (PyFly._calculate_airspeed_factors with the quaternion rotation) ----
  T ur = u, vr = v, wr = w;
  if (Spec::generic && P.wind_enabled) {
    const T wn = in.wind[0], we = in.wind[1], wd = in.wind[2];
    ur -= ((T)-1 + 2 * (e0 * e0 + e1 * e1)) * wn + 2 * (e1 * e2 + e3 * e0) * we + 2 * (e1 * e3 - e2 * e0) * wd;
    vr -= 2 * (e1 * e2 - e3 * e0) * wn + ((T)-1 + 2 * (e0 * e0 + e2 * e2)) * we + 2 * (e2 * e3 + e1 * e0) * wd;
    wr -= 2 * (e1 * e3 + e2 * e0) * wn + 2 * (e2 * e3 - e1 * e0) * we + ((T)-1 + 2 * (e0 * e0 + e3 * e3)) * wd;
  }
  // gusts are zero-filled by the caller when turbulence is off (x - 0 is exact)
  ur -= in.gl[0]; vr -= in.gl[1]; wr -= in.gl[2];
  const T pa = p - in.ga[0], qa = q - in.ga[1], ra = r - in.ga[2];
  // Va = |v_r|, alpha = atan2(w_r, u_r), beta = asin(v_r / Va) = atan2(v_r, hypot(u_r, w_r)): the two atan2 and the
  // two sqrt/rsqrt pairs are independent chains
  const T hxz2 = ur * ur + wr * wr;
  T Va_raw, invVa_raw, hxz, ih;
  Mt::sqrt_rsqrt(hxz2 + vr * vr, &Va_raw, &invVa_raw);
  Mt::sqrt_rsqrt(hxz2, &hxz, &ih);
  T alpha = Mt::atan2_(wr, ur);
  T beta = Mt::atan2_(vr, hxz);
  const T Va = fw_cond_r<T, Spec, FW_R_VA>(P, P.var[FW_SV_VA], Va_raw, failmask);
  T invVa = invVa_raw;
  if (Va != Va_raw) invVa = Mt::rcp_(Va);   // value_min clip engaged (rare)
  alpha = fw_cond_r<T, Spec, FW_R_ALPHA>(P, P.var[FW_SV_ALPHA], alpha, failmask);
  beta = fw_cond_r<T, Spec, FW_R_BETA>(P, P.var[FW_SV_BETA], beta, failmask);

  // ---- forces and moments (PyFly._forces) ----
  const T pre = (T)0.5 * PP.rho() * Va * Va * PP.S_wing();
  const T mg = PP.mass() * PP.g();
  const T fgx = mg * (2 * (e1 * e3 - e2 * e0));
  const T fgy = mg * (2 * (e2 * e3 + e1 * e0));
  const T fgz = mg * (e3 * e3 + e0 * e0 - e1 * e1 - e2 * e2);

  const T CLlin = PP.C_L_0() + PP.C_L_alpha() * alpha;
  // sigma = (1 + e1 + e2) / ((1 + e1)(1 + e2)), e1 = exp(-M(alpha - a0)), e2 = exp(M(alpha + a0)).  e1 * e2 is the
  // constant exp(2 M a0) (host-computed), so fp64 needs ONE exponential: with e2 = C / e1 the quotient becomes
  // (e1 + e1^2 + C) / ((1 + e1)(e1 + C)); |alpha| <= pi keeps e1^2 far inside the fp64 range.
  T sigma;
  if constexpr (sizeof(T) == 8) {
    const T x1 = Mt::exp_(-PP.M() * (alpha - PP.a_0()));
    const T C = PP.exp_2Ma0();
    sigma = Mt::div_(fma(x1, x1, x1) + C, (1 + x1) * (x1 + C));
  } else {
    // fp32: (1+e1)(1+e2) must stay below FLT_MAX, so both exponents are clamped (e1 * e2 is constant)
    const T ex1 = Mt::exp_(fminf(-PP.M() * (alpha - PP.a_0()), 80.0f));
    const T ex2 = Mt::exp_(fminf(PP.M() * (alpha + PP.a_0()), 80.0f));
    sigma = Mt::div_(1 + ex1 + ex2, (1 + ex1) * (1 + ex2));
  }
  // sin/cos of alpha and beta follow algebraically from the airspeed components (beta = asin(v_r / |v_r|) uses the
  // UNclipped airspeed) when neither angle was altered by a clip (the usual configuration); otherwise sincos.
  T sa, ca, sb, cb;
  if (!Spec::generic || (P.var[FW_SV_ALPHA].flags | P.var[FW_SV_BETA].flags) == 0u) {
    const bool nz = hxz > (T)0;
    sa = nz ? wr * ih : (T)0;
    ca = nz ? ur * ih : (T)1;
    sb = vr * invVa_raw;
    cb = hxz * invVa_raw;
  } else {
    Mt::sincos_(alpha, &sa, &ca);
    Mt::sincos_(beta, &sb, &cb);
  }
  const T sgn = alpha > 0 ? (T)1 : (alpha < 0 ? (T)-1 : (T)0);
  const T CL = (1 - sigma) * CLlin + sigma * (2 * sgn * sa * sa * ca);
  const T inv2Va = (T)0.5 * invVa;
  const T c2Va = PP.c() * inv2Va, b2Va = PP.b() * inv2Va;
  const T lift = pre * (CL + PP.C_L_q() * c2Va * qa + PP.C_L_delta_e() * elev);
  T CDa;
  if (!Spec::generic || P.drag_model == 0)
    CDa = PP.C_D_p() + (1 - sigma) * CLlin * CLlin * PP.inv_pi_e_ar() + sigma * (2 * sgn * sa * sa * sa);
  else
    CDa = PP.C_D_0() + PP.C_D_alpha1() * alpha + PP.C_D_alpha2() * alpha * alpha;
  const T CDb = PP.C_D_beta1() * beta + PP.C_D_beta2() * beta * beta;
  const T drag = pre * (CDa + CDb + PP.C_D_q() * c2Va * qa + PP.C_D_delta_e() * elev * elev);
  const T Cm = (1 - sigma) * (PP.C_m_0() + PP.C_m_alpha() * alpha) + sigma * (PP.C_m_fp() * sgn * sa * sa);
  const T mm = pre * PP.c() * (Cm + PP.C_m_q() * b2Va * qa + PP.C_m_delta_e() * elev);
  const T fy = pre * (PP.C_Y_0() + PP.C_Y_beta() * beta + PP.C_Y_p() * b2Va * pa + PP.C_Y_r() * b2Va * ra +
                      PP.C_Y_delta_a() * ail + PP.C_Y_delta_r() * rud);
  const T ll = pre * PP.b() * (PP.C_l_0() + PP.C_l_beta() * beta + PP.C_l_p() * b2Va * pa + PP.C_l_r() * b2Va * ra +
                               PP.C_l_delta_a() * ail + PP.C_l_delta_r() * rud);
  const T nn = pre * PP.b() * (PP.C_n_0() + PP.C_n_beta() * beta + PP.C_n_p() * b2Va * pa + PP.C_n_r() * b2Va * ra +
                               PP.C_n_delta_a() * ail + PP.C_n_delta_r() * rud);
  // f_aero = R(0, alpha, beta) * [-D, Y, -L]
  const T fax = ca * cb * (-drag) + ca * sb * fy + sa * lift;
  const T fay = sb * drag + cb * fy;
  const T faz = sa * cb * (-drag) + sa * sb * fy - ca * lift;
  const T Vd = Va + th * (PP.k_motor() - Va);
  const T fprop = (T)0.5 * PP.rho() * PP.S_prop() * PP.C_prop() * Vd * (Vd - Va);
  const T kot = PP.k_Omega() * th;
  const T tprop = -PP.k_T_P() * kot * kot;
  const T fx = fprop + fgx + fax, fyy = fgy + fay, fz = fgz + faz;
  const T tl = ll + tprop, tm = mm, tn = nn;

  // ---- kinematics / rigid body ----
  dy[0] = (T)0.5 * (-p * e1 - q * e2 - r * e3);
  dy[1] = (T)0.5 * (p * e0 + r * e2 - q * e3);
  dy[2] = (T)0.5 * (q * e0 - r * e1 + p * e3);
  dy[3] = (T)0.5 * (r * e0 + q * e1 - p * e2);
#define FW_G(k) fw_rd<T>(P, P.gammas[k])
  dy[4] = FW_G(1) * p * q - FW_G(2) * q * r + FW_G(3) * tl + FW_G(4) * tn;
  dy[5] = FW_G(5) * p * r - FW_G(6) * (p * p - r * r) + tm * fw_rd<T>(P, P.inv_Jy);
  dy[6] = FW_G(7) * p * q - FW_G(1) * q * r + FW_G(4) * tl + FW_G(8) * tn;
#undef FW_G
  dy[7] = (e1 * e1 + e0 * e0 - e2 * e2 - e3 * e3) * u + 2 * (e1 * e2 - e3 * e0) * v + 2 * (e1 * e3 + e2 * e0) * w;
  dy[8] = 2 * (e1 * e2 + e3 * e0) * u + (e2 * e2 + e0 * e0 - e1 * e1 - e3 * e3) * v + 2 * (e2 * e3 - e1 * e0) * w;
  dy[9] = 2 * (e1 * e3 - e2 * e0) * u + 2 * (e2 * e3 + e1 * e0) * v + (e3 * e3 + e0 * e0 - e1 * e1 - e2 * e2) * w;
  const T im = PP.inv_mass();
  dy[10] = r * v - q * w + fx * im;
  dy[11] = p * w - r * u + fyy * im;
  dy[12] = q * u - p * v + fz * im;
  const T av[3] = {el, er, th};
#pragma unroll
  for (int i = 0; i < 3; ++i) {
#define FW_AC(k) fw_rd<T>(P, P.act_coef[i][k])
    dy[13 + i] = av[i] * FW_AC(0) + in.cmd[i] * FW_AC(2) + ad[i] * FW_AC(1);
    dy[16 + i] = av[i] * FW_AC(3) + in.cmd[i] * FW_AC(5) + ad[i] * FW_AC(4);
#undef FW_AC
  }
}

// Dormand-Prince 5(4) tableau (scipy/integrate/_ivp/rk.py:541-552).  Row 6 of A is B (FSAL).
__constant__ double c_dpA[7][6] = {
    {0, 0, 0, 0, 0, 0},
    {1.0 / 5, 0, 0, 0, 0, 0},
    {3.0 / 40, 9.0 / 40, 0, 0, 0, 0},
    {44.0 / 45, -56.0 / 15, 32.0 / 9, 0, 0, 0},
    {19372.0 / 6561, -25360.0 / 2187, 64448.0 / 6561, -212.0 / 729, 0, 0},
    {9017.0 / 3168, -355.0 / 33, 46732.0 / 5247, 49.0 / 176, -5103.0 / 18656, 0},
    {35.0 / 384, 0, 500.0 / 1113, 125.0 / 192, -2187.0 / 6784, 11.0 / 84}};
__constant__ double c_dpE[7] = {-71.0 / 57600, 0, 71.0 / 16695, -71.0 / 1920, 17253.0 / 339200, -22.0 / 525, 1.0 / 40};
__constant__ float c_dpAf[7][6] = {
    {0, 0, 0, 0, 0, 0},
    {(float)(1.0 / 5), 0, 0, 0, 0, 0},
    {(float)(3.0 / 40), (float)(9.0 / 40), 0, 0, 0, 0},
    {(float)(44.0 / 45), (float)(-56.0 / 15), (float)(32.0 / 9), 0, 0, 0},
    {(float)(19372.0 / 6561), (float)(-25360.0 / 2187), (float)(64448.0 / 6561), (float)(-212.0 / 729), 0, 0},
    {(float)(9017.0 / 3168), (float)(-355.0 / 33), (float)(46732.0 / 5247), (float)(49.0 / 176), (float)(-5103.0 / 18656), 0},
    {(float)(35.0 / 384), 0, (float)(500.0 / 1113), (float)(125.0 / 192), (float)(-2187.0 / 6784), (float)(11.0 / 84)}};
__constant__ float c_dpEf[7] = {(float)(-71.0 / 57600), 0, (float)(71.0 / 16695), (float)(-71.0 / 1920),
                                (float)(17253.0 / 339200), (float)(-22.0 / 525), (float)(1.0 / 40)};
template <typename T> __device__ __forceinline__ T fw_dpA(int s, int j) {
  if constexpr (sizeof(T) == 8) return c_dpA[s][j]; else return c_dpAf[s][j];
}
template <typename T> __device__ __forceinline__ T fw_dpE(int s) {
  if constexpr (sizeof(T) == 8) return c_dpE[s]; else return c_dpEf[s];
}

// The position states (y[7..9]) never feed back into the right-hand side, so their K stages are not stored: their
// contributions to y_new (B row) and to the error estimate (E row) are accumulated in registers as each stage is
// produced.  The other 16 components keep their K stages in shared memory.
#define FW_N_KC 16
__device__ __forceinline__ constexpr int fw_kc_to_ode(int kc) { return kc < 7 ? kc : kc + 3; }

// K-stage storage: shared memory, one lane's values of a (slot, component pair) 16 bytes apart from the next lane's ->
// conflict-free.
template <typename T, int BLOCK> struct FwKStore {
  T* base;
  // components in pairs, [slot][pair][thread][2]: the unrolled stage code reads / writes two components per 16-byte
  // access (LDS.128 / STS.128, 512 B per warp instruction, conflict-free) - half the shared-memory instructions of the
  // [slot][component][thread] layout (round 2: dynamics kernels 143.2 -> 139.2 us)
  __device__ __forceinline__ T& at(int slot, int kc) {
    return base[((slot * (FW_N_KC / 2) + (kc >> 1)) * BLOCK + threadIdx.x) * 2 + (kc & 1)];
  }
};

// Stage state of stage S_ for the 16 stored components: ys = y + h * sum_{j < S_} a_{S_ j} K_j, accumulated exactly as
// the former run-time loop did (ys = fma(h a_sj, K_j, ys), j ascending, zero coefficients included) but with stage and
// term as compile-time numbers: tableau entries become constant-bank operands, K addresses immediates, no loop / remainder
// branches and no copy of y (round 2: that loop was 22 % of the executed instructions and 27 % of a warp's time,
// profiles/r2y_attempt_kernel_ncu_full.csv joined with the SASS; DESIGN.md 4.2).
template <typename T, int BLOCK, int S_, class KS>
__device__ __forceinline__ void fw_stage_state(const T (&y)[FW_N_ODE], T h, KS K, T (&ys)[FW_N_ODE]) {
#pragma unroll
  for (int j = 0; j < S_; ++j) {
    const T ha = h * fw_dpA<T>(S_, j);
#pragma unroll
    for (int kc = 0; kc < FW_N_KC; ++kc) {
      const int c = fw_kc_to_ode(kc);
      ys[c] = fma(ha, K.at(j, kc), j == 0 ? y[c] : ys[c]);
    }
  }
}

// 1/x to ~1 ulp without the division slow path (x is a tolerance scale >= atol > 0, always a normal number)
__device__ __forceinline__ double fw_rcp(double x) {
  double r;
  asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(x));
  r = fma(fma(-x, r, 1.0), r, r);
  r = fma(fma(-x, r, 1.0), r, r);
  return r;
}
__device__ __forceinline__ float fw_rcp(float x) { return FwMath<float>::rcp_(x); }

// ---- resumable scipy-RK45 state of ONE solve_ivp(fun, (0, dt), y0) call ---------------------------------------------
// Everything an aircraft carries from one dopri5 step attempt to the next.  K0 = f(t, y) (FSAL) lives in slot 0 of the
// lane's K store; its position components in k0pos.  Between the INIT kernel and the ATTEMPT kernel (csrc/fwgym.cu)
// the state is parked in HBM, so any lane can pick any aircraft up at an attempt boundary.
template <typename T> struct FwIvp {
  T y[FW_N_ODE];
  T k0pos[3];
  T t, h_abs;
  int status;        // FW_STATUS_*
  int rejected;      // step_rejected of the attempt loop in progress (rk.py:122)
  int attempts, accepted;
  int fail;          // != 0: ConstraintException raised by an RHS evaluation (FW_TERM_FAIL_BASE + sv)
};

template <typename T>
__device__ __forceinline__ int fw_fail_code(uint32_t failmask) {
  // the first violated variable in PyFly's evaluation order names the ConstraintException
  return FW_TERM_FAIL_BASE + c_rank_sv[__ffs((int)failmask) - 1];
}

// RK45.__init__: f0 = f(t0, y0) and select_initial_step (scipy/integrate/_ivp/common.py:68-134, rk.py:85-109).
// Two right-hand-side evaluations.  Returns the failure code (0 = ok); on success f0 holds f(t0, y0) and h_abs the
// initial step size (clamped to the interval; the min_step clamp of the first _step_impl call is applied by
// fw_ivp_attempt like for every other entry).
template <typename T, class Spec, class PAR>
__device__ __forceinline__ int fw_ivp_init(const fw_sim_t& P, const PAR& PP, const FwStepIn<T>& in,
                                           const T (&y)[FW_N_ODE], T (&f0)[FW_N_ODE], T& h_abs) {
  typedef FwMath<T> Mt;
  const T rtol = fw_rd<T>(P, P.rtol), atol = fw_rd<T>(P, P.atol), tb = fw_rd<T>(P, P.dt);
  const T inv_sqrtn = (T)(1.0 / 4.358898943540674);   // 1 / 19 ** 0.5
  uint32_t failmask = 0u;
  fw_rhs<T, Spec, true>(P, PP, in, y, f0, failmask);   // t == 0: stored state values, unconditioned
  if (failmask) return fw_fail_code<T>(failmask);
  T isc[FW_N_ODE];
  T s0 = 0, s1 = 0;
#pragma unroll
  for (int c = 0; c < FW_N_ODE; ++c) {
    isc[c] = fw_rcp(atol + fabs(y[c]) * rtol);
    const T a = y[c] * isc[c], b = f0[c] * isc[c];
    s0 += a * a;
    s1 += b * b;
  }
  const T d0 = Mt::sqrt_(s0) * inv_sqrtn;
  const T d1 = Mt::sqrt_(s1) * inv_sqrtn;
  T h0 = (d0 < (T)1e-5 || d1 < (T)1e-5) ? (T)1e-6 : Mt::div_((T)0.01 * d0, d1);
  h0 = h0 < tb ? h0 : tb;
  T y1[FW_N_ODE], f1[FW_N_ODE];
#pragma unroll
  for (int c = 0; c < FW_N_ODE; ++c) y1[c] = y[c] + h0 * f0[c];
  fw_rhs<T, Spec>(P, PP, in, y1, f1, failmask);
  if (failmask) return fw_fail_code<T>(failmask);
  T s2 = 0;
#pragma unroll
  for (int c = 0; c < FW_N_ODE; ++c) {
    const T a = (f1[c] - f0[c]) * isc[c];
    s2 += a * a;
  }
  const T d2 = Mt::div_(Mt::sqrt_(s2) * inv_sqrtn, h0);
  T h1;
  if (d1 <= (T)1e-15 && d2 <= (T)1e-15) {
    h1 = h0 * (T)1e-3;
    h1 = h1 > (T)1e-6 ? h1 : (T)1e-6;
  } else {
    h1 = Mt::pow_(Mt::div_((T)0.01, d1 > d2 ? d1 : d2), (T)0.2);
  }
  T ha = 100 * h0;
  ha = ha < h1 ? ha : h1;
  h_abs = ha < tb ? ha : tb;
  return 0;
}

// ONE dopri5 step attempt (the body of the `while not step_accepted` loop of RK45._step_impl, rk.py:111-176) for a
// lane whose S.status is RUNNING; six right-hand-side evaluations through one call site.  Updates S (and K slot 0 on
// acceptance); sets S.status to FINISHED when t reaches t_bound or an RHS evaluation raises, TOO_SMALL when the step
// size underflows.
template <typename T, class Spec, int BLOCK, class PAR>
__device__ __forceinline__ void fw_ivp_attempt(const fw_sim_t& P, const PAR& PP,
                                               const FwStepIn<T>& in, FwIvp<T>& S, FwKStore<T, BLOCK> K) {
  typedef FwMath<T> Mt;
  const T rtol = fw_rd<T>(P, P.rtol), atol = fw_rd<T>(P, P.atol), tb = fw_rd<T>(P, P.dt);
  const T inv_sqrtn = (T)(1.0 / 4.358898943540674);
  // ---- start a step attempt (rk.py:111-147); min_step = 10 * |nextafter(t, inf) - t|
  const T min_step = 10 * fabs(Mt::next_up(S.t) - S.t);
  if (!S.rejected && S.h_abs < min_step) S.h_abs = min_step;      // clamp on entry to _step_impl only
  {
    // A NaN step size never shrinks below min_step: scipy's loop would spin forever.  That, and an env step that
    // exceeds the attempt cap (the opt-in fw_sim_t.max_attempts, else the hang guard), ends the step as a NUMERIC
    // failure.  (`!(a >= b)` is true for NaN.)
    const int cap = P.max_attempts > 0 ? P.max_attempts : FW_MAX_ATTEMPTS;
    if (!(S.h_abs >= min_step) || S.attempts >= cap) {
      if (S.h_abs < min_step) S.status = FW_STATUS_TOO_SMALL;     // scipy: "step size too small"; PyFly carries on
      else { S.fail = FW_TERM_NUMERIC; S.status = FW_STATUS_FINISHED; }
      return;
    }
  }
  T t_new = S.t + S.h_abs;
  if (t_new - tb > 0) t_new = tb;
  const T h = t_new - S.t;
  S.h_abs = fabs(h);
  ++S.attempts;
  T accB[3], accE[3];    // running B-row / E-row sums of the position components (never stored as K stages)
#pragma unroll
  for (int j = 0; j < 3; ++j) { accB[j] = fw_dpA<T>(6, 0) * S.k0pos[j]; accE[j] = fw_dpE<T>(0) * S.k0pos[j]; }
#pragma unroll 1
  for (int s = 1; s <= 6; ++s) {
    T ys[FW_N_ODE], f[FW_N_ODE];
    {
      // y_s = y + h * sum_j a_sj K_j, accumulated as y += (h a_sj) K_j (one fma per term, no separate scaling pass)
      switch (s) {
        case 1: fw_stage_state<T, BLOCK, 1>(S.y, h, K, ys); break;
        case 2: fw_stage_state<T, BLOCK, 2>(S.y, h, K, ys); break;
        case 3: fw_stage_state<T, BLOCK, 3>(S.y, h, K, ys); break;
        case 4: fw_stage_state<T, BLOCK, 4>(S.y, h, K, ys); break;
        case 5: fw_stage_state<T, BLOCK, 5>(S.y, h, K, ys); break;
        default: fw_stage_state<T, BLOCK, 6>(S.y, h, K, ys); break;
      }
      // position stage states are never read by the RHS; y_new[pos] is formed from accB when s == 6
#pragma unroll
      for (int j = 0; j < 3; ++j) ys[7 + j] = S.y[7 + j] + h * accB[j];
    }
    uint32_t failmask = 0u;
    fw_rhs<T, Spec>(P, PP, in, ys, f, failmask);
    if (failmask) {
      S.fail = fw_fail_code<T>(failmask);
      S.status = FW_STATUS_FINISHED;
      return;
    }
    if (s < 6) {
#pragma unroll
      for (int kc = 0; kc < FW_N_KC; ++kc) K.at(s, kc) = f[fw_kc_to_ode(kc)];
      const T b = fw_dpA<T>(6, s), e = fw_dpE<T>(s);
#pragma unroll
      for (int j = 0; j < 3; ++j) { accB[j] += b * f[7 + j]; accE[j] += e * f[7 + j]; }
      continue;
    }
    // s == 6: ys == y_new, f == f_new.  error = (K^T . E) * h ; scale = atol + max(|y|,|y_new|)*rtol (rk.py:150-152)
    T se = 0;
#pragma unroll
    for (int kc = 0; kc < FW_N_KC; ++kc) {
      const int c = fw_kc_to_ode(kc);
      T e = fw_dpE<T>(6) * f[c];
#pragma unroll
      for (int j = 0; j < 6; ++j)
        if (j != 1) e += fw_dpE<T>(j) * K.at(j, kc);
      e *= h;
      const T ay = fabs(S.y[c]), an = fabs(ys[c]);
      const T q = e * fw_rcp(atol + (ay > an ? ay : an) * rtol);
      se += q * q;
    }
#pragma unroll
    for (int j = 0; j < 3; ++j) {
      const T e = (accE[j] + fw_dpE<T>(6) * f[7 + j]) * h;
      const T ay = fabs(S.y[7 + j]), an = fabs(ys[7 + j]);
      const T q = e * fw_rcp(atol + (ay > an ? ay : an) * rtol);
      se += q * q;
    }
    const T err = Mt::sqrt_(se) * inv_sqrtn;
    // 0.9 * err ** -0.2 feeds both outcomes (rk.py:160-172); err == 0 gives a huge value that the min() below turns
    // into MAX_FACTOR, exactly the reference's special case
    const T pw = (T)0.9 * Mt::pow_(err, (T)-0.2);
    if (err < (T)1) {
      T factor = pw < (T)10 ? pw : (T)10;
      if (S.rejected) factor = factor < (T)1 ? factor : (T)1;
      S.h_abs *= factor;
      S.t = t_new;
#pragma unroll
      for (int c = 0; c < FW_N_ODE; ++c) S.y[c] = ys[c];
#pragma unroll
      for (int kc = 0; kc < FW_N_KC; ++kc) K.at(0, kc) = f[fw_kc_to_ode(kc)];
#pragma unroll
      for (int j = 0; j < 3; ++j) S.k0pos[j] = f[7 + j];
      ++S.accepted;
      S.rejected = 0;
      if (S.t - tb >= 0) S.status = FW_STATUS_FINISHED;
    } else {
      // NaN error norms land here too: Python's max(0.2, nan) == 0.2
      S.h_abs *= pw > (T)0.2 ? pw : (T)0.2;
      S.rejected = 1;
    }
  }
}
