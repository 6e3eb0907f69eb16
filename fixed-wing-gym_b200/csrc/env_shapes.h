// Compile-time configuration SHAPES for the env-side kernels.
//
// fw_env_kernel / fw_reset_kernel are config-driven: which observation variables, reward factors, target classes,
// history rings ... exist is data (fw_env_t), so the generic instantiation walks those tables with warp-uniform
// branches, indexed constant loads and local-memory arrays (~7700 executed instructions per env step, most of them
// bookkeeping).  For the SHIPPED configurations the structure is known when the library is built: scripts/
// gen_env_shapes.py compiles each shipped JSON and writes the integer fields of the resulting fw_env_t / fw_sim_t as
// constexpr builders (env_shapes_gen.h).  A kernel instantiated on such a shape reads
//     structure (counts, kinds, windows, flags, row numbers)  from a `__device__ const` copy of the shape -> after
//                                                             full unrolling every such read folds to a literal,
//     numbers   (bounds, scalings, means, gains, coefficients) from the runtime __grid_constant__ configuration,
// so the same source yields one straight-line block per shape and the table-walking code for everything else
// (FwShapeGeneric).  The host picks the instantiation whose shape equals the handle's configuration
// (fw_find_shape); any other configuration runs the generic kernels.  Both are parity-tested.
#pragma once
#include "layout.h"
#include "env_shapes_gen.h"

// `mixed`: the configuration flies each env at its own Dryden intensity (fw_sim_t.turb_mixed).  A compile-time property
// of every shape, so that the per-env level code exists only in the instantiations that need it: the generic kernels
// come in two instantiations, FwShapeGeneric (one intensity for the whole handle) and FwShapeGenericMixed.
//
// `bank`: the handle keeps the scenario-bank rows (fw_env_t.bank_enabled, fw_set_bank).  Also compile-time, so that the
// instantiations without it compile to exactly the code they compiled to before the bank existed: two more generic
// instantiations, FwShapeGenericBank and FwShapeGenericMixedBank.
struct FwShapeGeneric {
  static constexpr bool fixed = false;
  static constexpr bool mixed = false;
  static constexpr bool bank = false;
  static constexpr fw_env_t cenv{};
  static __device__ __forceinline__ const fw_env_t& env(const fw_env_t& E) { return E; }
  static __device__ __forceinline__ const fw_sim_t& sim(const fw_sim_t& P) { return P; }
  static __device__ __forceinline__ const FwLayout& lay(const FwLayout& L) { return L; }
};
struct FwShapeGenericMixed : FwShapeGeneric {
  static constexpr bool mixed = true;
};
struct FwShapeGenericBank : FwShapeGeneric {
  static constexpr bool bank = true;
};
struct FwShapeGenericMixedBank : FwShapeGeneric {
  static constexpr bool mixed = true;
  static constexpr bool bank = true;
};

constexpr FwLayout fw_shape_layout(const fw_env_t& e, const fw_sim_t& s) {
  FwLayout L{};
  fw_layout_build(e, s.scale_actions, 0, L, s.turb_mixed);
  return L;
}

#define FW_DEFINE_SHAPE(NAME)                                                                              \
  __device__ const fw_env_t kShapeEnv_##NAME = fw_shape_env_##NAME();                                      \
  __device__ const fw_sim_t kShapeSim_##NAME = fw_shape_sim_##NAME();                                      \
  __device__ const FwLayout kShapeLay_##NAME = fw_shape_layout(fw_shape_env_##NAME(), fw_shape_sim_##NAME()); \
  struct FwShape_##NAME {                                                                                  \
    static constexpr bool fixed = true;                                                                    \
    static constexpr bool mixed = fw_shape_sim_##NAME().turb_mixed != 0;                                   \
    static constexpr bool bank = fw_shape_env_##NAME().bank_enabled != 0;                                  \
    static constexpr fw_env_t cenv = fw_shape_env_##NAME();   /* for constant expressions (loop trip counts) */ \
    static __device__ __forceinline__ const fw_env_t& env(const fw_env_t&) { return kShapeEnv_##NAME; }    \
    static __device__ __forceinline__ const fw_sim_t& sim(const fw_sim_t&) { return kShapeSim_##NAME; }    \
    static __device__ __forceinline__ const FwLayout& lay(const FwLayout&) { return kShapeLay_##NAME; }    \
  };
FW_SHAPE_LIST(FW_DEFINE_SHAPE)
#undef FW_DEFINE_SHAPE

// Loop over i in [0, n).  Fixed shapes: the body is instantiated per index by template recursion, so everything
// indexed by i (shape tables, local arrays) folds to literals.  (Not `#pragma unroll`: the compiler declines to unroll
// a loop around a body as large as one observation variable, and then nothing indexed by i folds.)
//   fw_loop<SH, N>(n, f)      N = the exact trip count as a constant expression for fixed shapes (FW_CNT below):
//                             exactly N bodies are instantiated;
//   fw_loop_le<SH, MAXN>(n, f) small inner loops whose count is only a literal after inlining (a window size of the
//                             enclosing table entry): MAXN guarded bodies, the dead ones fold away.
template <int I, int N, bool GUARD, class F>
__device__ __forceinline__ void fw_static_for(int n, F& f) {
  if constexpr (I < N) {
    if (!GUARD || I < n) f(I);
    fw_static_for<I + 1, N, GUARD>(n, f);
  }
}
template <class SH, int N, class F>
__device__ __forceinline__ void fw_loop(int n, F&& f) {
  if constexpr (SH::fixed) {
    fw_static_for<0, N, false>(n, f);
  } else {
#pragma unroll 1
    for (int i = 0; i < n; ++i) f(i);
  }
}
template <class SH, int MAXN, class F>
__device__ __forceinline__ void fw_loop_le(int n, F&& f) {
  if constexpr (SH::fixed) {
    if (n <= MAXN) {
      fw_static_for<0, MAXN, true>(n, f);
      return;
    }
  }
#pragma unroll 1
  for (int i = 0; i < n; ++i) f(i);
}
// loop bodies are lambdas; without this the inliner may keep a large body out of line, and then the shape is read
// through a pointer at run time instead of folding
#define FW_LAMBDA_INLINE __attribute__((always_inline))
// trip count of a loop over a table of the env configuration, as a constant expression
#define FW_CNT(FIELD) (SH::fixed ? SH::cenv.FIELD : 0)

// ---- host side: does a runtime configuration have this shape? -------------------------------------------------------
inline bool fw_env_same_shape(const fw_env_t& a, const fw_env_t& b) {
  if (a.integration_window != b.integration_window || a.obs_len != b.obs_len || a.obs_step != b.obs_step ||
      a.obs_nvar != b.obs_nvar || a.obs_shape != b.obs_shape || a.obs_norm != b.obs_norm || a.obs_noise != b.obs_noise ||
      a.has_bounds != b.has_bounds || a.n_targets != b.n_targets || a.resample_every != b.resample_every ||
      a.streak_req != b.streak_req || a.n_factors != b.n_factors ||
      a.potential != b.potential || a.step_fail_timesteps != b.step_fail_timesteps || a.n_terms != b.n_terms ||
      a.metrics_enabled != b.metrics_enabled || a.n_rand != b.n_rand || a.n_par_rows != b.n_par_rows ||
      a.n_scale_rows != b.n_scale_rows || a.bank_enabled != b.bank_enabled)
    return false;
  for (int v = 0; v < a.obs_nvar; ++v) {
    const fw_obs_var_t &x = a.obs[v], &y = b.obs[v];
    if (x.type != y.type || x.ref != y.ref || x.value_kind != y.value_kind || x.window != y.window || x.norm != y.norm)
      return false;
  }
  for (int k = 0; k < a.n_targets; ++k) {
    const fw_target_t &x = a.tgt[k], &y = b.tgt[k];
    if (x.sv != y.sv || x.cls != y.cls || x.wrap != y.wrap || x.has_delta != y.has_delta || x.has_bound != y.has_bound ||
        x.to_radians != y.to_radians)
      return false;
  }
  for (int f = 0; f < a.n_factors; ++f) {
    const fw_factor_t &x = a.fac[f], &y = b.fac[f];
    if (x.cls != y.cls || x.type != y.type || x.fclass != y.fclass || x.ref != y.ref || x.window != y.window ||
        x.shaping != y.shaping || x.has_max != y.has_max || x.value_timesteps != y.value_timesteps ||
        x.scale_slot1 != y.scale_slot1)
      return false;
  }
  for (int t = 0; t < a.n_terms; ++t)
    if (a.term_fclass[t] != b.term_fclass[t]) return false;
  return true;
}
inline bool fw_sim_same_shape(const fw_sim_t& a, const fw_sim_t& b) {
  if (a.drag_model != b.drag_model || a.turbulence != b.turbulence || a.turb_mixed != b.turb_mixed ||
      a.wind_enabled != b.wind_enabled ||
      a.scale_actions != b.scale_actions || a.has_scale_low != b.has_scale_low || a.has_scale_high != b.has_scale_high)
    return false;
  for (int f = 0; f < FW_N_FILT; ++f)
    if (a.filt[f].n != b.filt[f].n || a.filt[f].stream != b.filt[f].stream) return false;
  for (int v = 0; v < FW_N_SV; ++v)
    if (a.var[v].flags != b.var[v].flags) return false;
  for (int i = 0; i < FW_N_ACT; ++i)
    if (a.act_has_dot_max[i] != b.act_has_dot_max[i]) return false;
  return true;
}

// index into FW_SHAPE_LIST of the shape this configuration has, -1: none (generic kernels)
inline int fw_find_shape(const fw_env_t& e, const fw_sim_t& s) {
  int idx = 0;
#define FW_TRY_SHAPE(NAME)                                                                                       \
  {                                                                                                              \
    constexpr fw_env_t se = fw_shape_env_##NAME();                                                               \
    constexpr fw_sim_t ss = fw_shape_sim_##NAME();                                                               \
    if (fw_env_same_shape(e, se) && fw_sim_same_shape(s, ss)) return idx;                                        \
    ++idx;                                                                                                       \
  }
  FW_SHAPE_LIST(FW_TRY_SHAPE)
#undef FW_TRY_SHAPE
  return -1;
}
