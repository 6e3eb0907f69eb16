// Env-side work of FixedWingAircraft.step / reset, one thread per env over coalesced SoA rows.
//
// What it replaces (SURVEY §8a): fixed_wing.py:338-437 (step orchestration), :287-336 (reset), :461-521
// (sample_target), :674-774 (get_reward), :776-846 (get_observation), :890-931 (_get_error, _get_goal_status),
// :933-991 (_get_next_target) and PyFly.reset (oracle/pyfly_restated.py: PyFly.reset) for the auto-reset.
#pragma once
#include <math_constants.h>
#include "layout.h"
#include "philox.cuh"
#include "dynamics.cuh"
#include "env_shapes.h"

// Every function below is templated on a configuration shape SH (env_shapes.h).  Convention inside the bodies:
//   Es / Ps / Ls : STRUCTURE (counts, kinds, flags, windows, row numbers) - literals when SH is a fixed shape;
//   E  / P  / L  : the runtime configuration - numbers only (and L.stride through the row accessor).
#define FW_SHAPE_REFS                          \
  const fw_env_t& Es = SH::env(E);             \
  const fw_sim_t& Ps = SH::sim(P);             \
  const FwLayout& Ls = SH::lay(L);             \
  (void)Es; (void)Ps; (void)Ls

#define FW_TWO_PI 6.283185307179586

struct FwEnvCtx {
  double* __restrict__ d;
  int32_t* __restrict__ i;
  int64_t stride;
  int64_t env;
  __device__ __forceinline__ double& D(int row) const { return d[(int64_t)row * stride + env]; }
  __device__ __forceinline__ int32_t& I(int row) const { return i[(int64_t)row * stride + env]; }
};

// NZ > 0: the first n_zpre (even, <= NZ) normals of this tick were drawn ahead of time (fw_env_kernel, before its chunk
// wait) and sit in zpre - an array MEMBER, so that the unrolled observation loop of a fixed shape indexes registers
template <bool INL, int NZ = 0>
struct FwEnvRngT {
  FwRng g;
  uint32_t n_u, n_n;        // uniform / normal draws consumed in this tick
  double z_cached;
  int n_zpre;
  double zpre[NZ > 0 ? NZ : 1];
  __device__ __forceinline__ double uniform(double lo, double hi) { return fw_uniform<INL>(g, FW_RS_ENV_U, n_u++, lo, hi); }
  __device__ __forceinline__ double uniform01() { return fw_uniform01<INL>(g, FW_RS_ENV_U, n_u++); }
  __device__ __forceinline__ double normal(double mean, double std) {
    double z;
    if ((int)n_n < n_zpre) z = zpre[n_n];
    else if (n_n & 1u) z = z_cached;
    else { double z1; fw_normal2_t<INL>(g, FW_RS_ENV_N, n_n >> 1, z, z1); z_cached = z1; }
    ++n_n;
    return mean + std * z;
  }
};

// current value of a PyFly state variable (`simulator.state[name].value`)
__device__ __forceinline__ double fw_sv_value_inl(const FwEnvCtx& c, int sv) {
  switch (sv) {
    case FW_SV_ROLL: return c.D(D_ROLL);
    case FW_SV_PITCH: return c.D(D_PITCH);
    case FW_SV_YAW: return c.D(D_YAW);
    case FW_SV_OMEGA_P: return c.D(D_OMEGA + 0);
    case FW_SV_OMEGA_Q: return c.D(D_OMEGA + 1);
    case FW_SV_OMEGA_R: return c.D(D_OMEGA + 2);
    case FW_SV_POS_N: return c.D(D_POS + 0);
    case FW_SV_POS_E: return c.D(D_POS + 1);
    case FW_SV_POS_D: return c.D(D_POS + 2);
    case FW_SV_VEL_U: return c.D(D_VEL + 0);
    case FW_SV_VEL_V: return c.D(D_VEL + 1);
    case FW_SV_VEL_W: return c.D(D_VEL + 2);
    case FW_SV_VA: return c.D(D_VA);
    case FW_SV_ALPHA: return c.D(D_ALPHA);
    case FW_SV_BETA: return c.D(D_BETA);
    case FW_SV_ELEVATOR: return c.D(D_ELEV);
    case FW_SV_AILERON: return c.D(D_AIL);
    case FW_SV_RUDDER: return 0.0;
    case FW_SV_THROTTLE: return c.D(D_ACT + 2);
    case FW_SV_ELEVON_L: return c.D(D_ACT + 0);
    case FW_SV_ELEVON_R: return c.D(D_ACT + 1);
  }
  return 0.0;
}
__device__ __noinline__ double fw_sv_value(const FwEnvCtx& c, int sv) { return fw_sv_value_inl(c, sv); }
// sv is a literal in a fixed shape: the switch folds to one row load
template <class SH>
__device__ __forceinline__ double fw_sv(const FwEnvCtx& c, int sv) {
  if constexpr (SH::fixed) return fw_sv_value_inl(c, sv);
  else return fw_sv_value(c, sv);
}

// python float floor-mod x % m for m > 0
__device__ __noinline__ double fw_pymod_slow(double x, double m) {
  double r = fmod(x, m);
  if (r != 0.0 && r < 0.0) r += m;
  return r;
}
// Same value without the fmod loop on the three periods around zero (every operand the env produces: angles and
// targets live in [-pi, pi]): fmod(x, m) is x itself for |x| < m and the exact difference x - m for m <= x < 2m.
__device__ __forceinline__ double fw_pymod(double x, double m) {
  if (x >= 0.0 && x < m) return x;
  if (x < 0.0 && x >= -m) return x + m;
  if (x >= m && x < 2.0 * m) return x - m;
  return fw_pymod_slow(x, m);
}

// fixed_wing.py:890-914
__device__ __forceinline__ double fw_error(int wrap, double target, double value) {
  if (wrap) return fw_pymod(value - target + CUDART_PI, FW_TWO_PI) - CUDART_PI;
  return target - value;
}

__device__ __forceinline__ int fw_tcls(uint32_t flags, int k) { return (flags >> (FWF_TCLS_SHIFT + 2 * k)) & 3u; }

// fixed_wing.py:916-931 : bit k = |err_k| <= bound_k for targets with a bound; bit 31 = all()
template <class SH>
__device__ __forceinline__ uint32_t fw_goal_status(const fw_env_t& E, const FwEnvCtx& c) {
  const fw_env_t& Es = SH::env(E);
  uint32_t bits = 0;
  bool all = true;
  fw_loop<SH, FW_CNT(n_targets)>(Es.n_targets, [&](int k) FW_LAMBDA_INLINE {
    if (!Es.tgt[k].has_bound) return;
    const double err = fw_error(Es.tgt[k].wrap, c.D(D_TARGET + k), fw_sv<SH>(c, Es.tgt[k].sv));
    const bool ok = fabs(err) <= E.tgt[k].bound;
    if (ok) bits |= 1u << k;
    all = all && ok;
  });
  if (all) bits |= 1u << 31;
  return bits;
}

// fixed_wing.py:461-521
template <class SH, class RNG>
__device__ __forceinline__ void fw_sample_target(const fw_env_t& E, const FwEnvCtx& c, RNG& rng, uint32_t& flags,
                                                 int steps_count) {
  const fw_env_t& Es = SH::env(E);
  c.I(I_STEPS_TGT) = 0;
  fw_loop<SH, FW_CNT(n_targets)>(Es.n_targets, [&](int k) FW_LAMBDA_INLINE {
    const fw_target_t& t = E.tgt[k];
    const fw_target_t& ts = Es.tgt[k];
    double low = t.low, high = t.high;
    if (ts.has_delta) {
      const double v = fw_sv<SH>(c, ts.sv);
      low = fmax(low, v - t.delta);
      high = fmax(fmin(high, v + t.delta), low);
    }
    const double initial = rng.uniform(low, high);
    flags = (flags & ~(3u << (FWF_TCLS_SHIFT + 2 * k))) | ((uint32_t)ts.cls << (FWF_TCLS_SHIFT + 2 * k));
    if (ts.cls == 1) {   // linear
      double slope = rng.uniform(t.slope_low, t.slope_high);
      if (rng.uniform01() < 0.5) slope *= -1.0;
      if (ts.to_radians) slope = slope * (CUDART_PI / 180.0);
      c.D(D_TSLOPE + k) = slope;
    } else if (ts.cls == 2) {   // sinusoidal
      double amp = rng.uniform(t.amp_low, t.amp_high);
      if (ts.to_radians) amp = amp * (CUDART_PI / 180.0);
      const double period = rng.uniform(t.period_low, t.period_high);
      const double phase = rng.uniform(0.0, FW_TWO_PI) / (FW_TWO_PI / period);
      c.D(D_TAMP + k) = amp;
      c.D(D_TPERIOD + k) = period;
      c.D(D_TPHASE + k) = phase;
      c.D(D_TBIAS + k) = initial - amp * sin(FW_TWO_PI / period * ((double)steps_count + phase));
    }
    c.D(D_TARGET + k) = initial;
  });
}

// fixed_wing.py:933-991 (all next targets are computed from the CURRENT targets, then assigned).  A target's class is
// its configured one unless reset(target=...) forced it to "constant" (flags), so a fixed shape only carries the
// code of the classes it configures.
template <class SH>
__device__ __forceinline__ void fw_next_targets(const fw_env_t& E, const fw_sim_t& P, const FwEnvCtx& c,
                                                uint32_t flags, int steps_count, int steps_tgt, double (&out)[FW_MAX_TARGETS]) {
  const fw_env_t& Es = SH::env(E);
  int pitch_k = -1;
  fw_loop<SH, FW_CNT(n_targets)>(Es.n_targets, [&](int k) FW_LAMBDA_INLINE { if (Es.tgt[k].sv == FW_SV_PITCH) pitch_k = k; });
  fw_loop<SH, FW_CNT(n_targets)>(Es.n_targets, [&](int k) FW_LAMBDA_INLINE {
    const fw_target_t& ts = Es.tgt[k];
    const int cfg_cls = ts.cls;
    const int cls = fw_tcls(flags, k);
    const double cur = c.D(D_TARGET + k);
    double res = cur;
    if (cfg_cls == 3 && cls == 3 && pitch_k >= 0) {   // compensate (Va)
      const int pc = fw_tcls(flags, pitch_k);
      const double pitch_cur = c.D(D_TARGET + pitch_k);
      const double pitch_tar = (Es.tgt[pitch_k >= 0 ? pitch_k : 0].cls == 2 && pc == 2) ? c.D(D_TBIAS + pitch_k) : pitch_cur;
      if (pitch_tar <= -2.5 * (CUDART_PI / 180.0)) {
        const double va_end = 28.434 - 40.0841 * pitch_tar;
        double slope = 0.0;
        if (cur <= va_end) slope = 7.0 * fmax(0.0, cur < va_end * 0.95 ? 1.0 : 1.0 - cur / (va_end * 1.5));
        res = cur + (slope * (-pitch_cur) - 0.25) * P.dt;
      } else if (pitch_tar >= 5.0 * (CUDART_PI / 180.0)) {
        const double va_end = 26.27 - 41.2529 * pitch_tar;
        if (cur > va_end) res = (steps_tgt < 750) ? cur + (va_end - cur) * 1.0 / 150.0 : va_end;
      }
    } else if (cfg_cls == 1 && cls == 1) {
      res = cur + c.D(D_TSLOPE + k) * P.dt;
    } else if (cfg_cls == 2 && cls == 2) {
      res = c.D(D_TAMP + k) * sin(FW_TWO_PI / c.D(D_TPERIOD + k) * ((double)steps_count + c.D(D_TPHASE + k))) + c.D(D_TBIAS + k);
    }
    if (ts.wrap && fabs(res) > CUDART_PI) {
      const double s = res > 0 ? 1.0 : -1.0;
      res = s * (fmod(fabs(res), CUDART_PI) - CUDART_PI);
    }
    out[k] = res;
  });
}

// ---- history rings.  Entry e (0 = the reset entry) lives in slot e % depth. -------------------------------------
__device__ __forceinline__ double fw_ring_get(const FwEnvCtx& c, int row0, int depth, int ncol, int col, int e) {
  return c.D(row0 + (e % depth) * ncol + col);
}
__device__ __forceinline__ void fw_ring_put(const FwEnvCtx& c, int row0, int depth, int ncol, int col, int e, double v) {
  c.D(row0 + (e % depth) * ncol + col) = v;
}

// fixed_wing.py:776-846.  hist_len = len(history["error"][k]) = len(PyFly Variable.history); steps_count as in the
// reference; `stale` selects the reset-time behaviour where the integrator reads the previous episode's history
// (fixed_wing.py:317 runs before :318).
// Observation sink: float32 rows for the policy, optional float64 copy for parity checks.
struct FwObsWriter {
  float* o32;
  double* o64;
  int64_t base;     // first element of this env's row in o64 (and in o32 unless base32 >= 0)
  int64_t base32;   // >= 0: o32 is a staging tile (fw_env_kernel, zero-copy host results) and this is the row's offset in it
  bool commit = true;   // false: the lanes that only accompany a cooperative reset (fw_env_kernel) write nothing
  __device__ __forceinline__ void operator()(int idx, double v) const {
    if (!commit) return;
    if (o32) o32[(base32 >= 0 ? base32 : base) + idx] = (float)v;
    if (o64) o64[base + idx] = v;
  }
};

// sum_{e = lo+1}^{hi-1} |x_e - x_{e-1}| over one ring column, in increasing e (at most `window` - 1 terms), each ring
// entry loaded once.  ACC = float reproduces np.sum(..., dtype=np.float32) (fixed_wing.py:826,828).
template <class SH, class ACC, int NCOL>
__device__ __forceinline__ void fw_ring_abs_diff(const FwEnvCtx& c, int row0, int depth, int col0, int lo, int hi,
                                                 int window, ACC (&acc)[NCOL]) {
  if (hi - lo < 2) return;
  double prev[NCOL];
#pragma unroll
  for (int j = 0; j < NCOL; ++j) prev[j] = fw_ring_get(c, row0, depth, FW_N_ACT, col0 + j, lo);
  fw_loop_le<SH, 8>(window - 1, [&](int t) FW_LAMBDA_INLINE {
    const int e = lo + 1 + t;
    if (e < hi) {
#pragma unroll
      for (int j = 0; j < NCOL; ++j) {
        const double cur = fw_ring_get(c, row0, depth, FW_N_ACT, col0 + j, e);
        acc[j] += (ACC)fabs(cur - prev[j]);
        prev[j] = cur;
      }
    }
  });
}

// Generic instantiation: one out-of-line copy serves the step, terminal-observation and reset call sites
// (instruction-cache footprint).  Fixed shapes inline it (fw_observation).
template <class SH, class RNG>
__device__ __forceinline__ void fw_observation_body(const fw_env_t& E, const fw_sim_t& P, const FwLayout& L,
                                                    const FwEnvCtx& c, RNG& rng, uint32_t flags, int steps_count,
                                                    int hist_len, bool at_reset, const FwObsWriter& out) {
  FW_SHAPE_REFS;
  const int nv = Es.obs_nvar, len = Es.obs_len, step = Es.obs_step;
  const int W = Es.integration_window;
  fw_loop<SH, FW_CNT(obs_len)>(len, [&](int row) FW_LAMBDA_INLINE {
    int i = 1 + row * step;
    double init_noise = 0.0;
    bool has_init_noise = false;
    if (i > steps_count) {
      i = steps_count + 1;
      if (len > 1) { init_noise = rng.uniform(-1.0, 1.0) * P.dt; has_init_noise = true; }
    }
    // index into PyFly / env histories; clamp for the failure step, where nothing was appended
    const int ih = i < hist_len ? i : hist_len;
    fw_loop<SH, FW_CNT(obs_nvar)>(nv, [&](int v) FW_LAMBDA_INLINE {
      const fw_obs_var_t& ov = E.obs[v];
      const fw_obs_var_t& os = Es.obs[v];
      double val;
      bool is_f32 = false;   // the action-delta value is an np.float32 in the reference (fixed_wing.py:826,828)
      if (os.type == 0) {
        if (Ls.sv_depth <= 1 || ih == 1) val = fw_sv<SH>(c, os.ref);
        else val = fw_ring_get(c, Ls.sv_row, Ls.sv_depth, Ls.n_sv_obs, Ls.sv_slot[v], hist_len - ih);
      } else if (os.type == 1) {
        const int k = os.ref;
        if (os.value_kind == 0) {
          if (i == 1) val = fw_error(Es.tgt[k].wrap, c.D(D_TARGET + k), fw_sv<SH>(c, Es.tgt[k].sv));
          else val = fw_ring_get(c, Ls.err_row, Ls.err_depth, Es.n_targets, k, hist_len - ih);
        } else if (os.value_kind == 1) {
          if (i == 1) val = c.D(D_TARGET + k);
          else val = fw_ring_get(c, Ls.tgt_row, Ls.tgt_depth, Es.n_targets, k, hist_len - ih);
        } else {
          if (at_reset && !(flags & FWF_HIST_VALID)) {
            val = fw_error(Es.tgt[k].wrap, c.D(D_TARGET + k), fw_sv<SH>(c, Es.tgt[k].sv)) * (double)W;
          } else {
            // np.sum(history["error"][k][-W-i:-i]) : entries [max(0, n-W-i), n-i)
            const int n = hist_len;
            int hi = n - i, lo = n - W - i;
            if (lo < 0) lo = 0;
            double s = 0.0;
            for (int e = lo; e < hi; ++e) s += fw_ring_get(c, Ls.err_row, Ls.err_depth, Es.n_targets, k, e);
            val = s;
            if (steps_count - i < W) val += (double)(W - (steps_count - i)) * c.D(D_ERR0 + k);
          }
        }
      } else {
        const int a = os.ref;
        if (steps_count - i < 0) {
          const int sv = a == 0 ? FW_SV_ELEVATOR : (a == 1 ? FW_SV_AILERON : FW_SV_THROTTLE);
          val = fw_sv<SH>(c, sv);
          if (Ps.scale_actions) {
            // linear_action_scaling(direction="backward") applied to a vector that is zero except at a
            const double omin = P.act_to_low[a], omax = P.act_to_high[a];
            val = (P.scale_high - P.scale_low) * (val - omin) / (omax - omin) + P.scale_low;
          }
        } else {
          // sum |diff| over the `window` entries of the action (or command) history ending i-1 steps ago,
          // accumulated in float32 (np.sum(..., dtype=np.float32))
          const int n = steps_count;            // len(history["action"])
          const int hi = n - (i - 1);           // exclusive
          int lo = n - os.window - i + 1;
          if (lo < 0) lo = 0;
          const int row0 = Ps.scale_actions ? Ls.act_row : Ls.cmd_row;
          const int depth = Ps.scale_actions ? Ls.act_depth : Ls.cmd_depth;
          float acc[1] = {0.0f};
          fw_ring_abs_diff<SH, float, 1>(c, row0, depth, a, lo, hi, os.window, acc);
          val = (double)acc[0];
          is_f32 = true;
        }
      }
      if (is_f32) {
        // numpy >= 2 (NEP 50) keeps np.float32 (+,-,/) python-float in float32, so the jitter / normalisation /
        // noise of this variable are float32 operations in the oracle run; mirrored here.
        float v32 = (float)val;
        if (has_init_noise) v32 = v32 + (float)init_noise;
        if (Es.obs_norm && os.norm) { v32 = v32 - (float)ov.mean; v32 = v32 / (float)ov.var; }
        if (Es.obs_noise) v32 = v32 + (float)rng.normal(E.obs_noise_mean, E.obs_noise_std);
        val = (double)v32;
      } else {
        if (has_init_noise) val += init_noise;
        if (Es.obs_norm && os.norm) { val -= ov.mean; val /= ov.var; }
        if (Es.obs_noise) val += rng.normal(E.obs_noise_mean, E.obs_noise_std);
      }
      out(row * nv + v, val);
    });
  });
}
__device__ __noinline__ void fw_observation_generic(const fw_env_t& E, const fw_sim_t& P, const FwLayout& L,
                                                    const FwEnvCtx& c, FwEnvRngT<false>& rng, uint32_t flags,
                                                    int steps_count, int hist_len, bool at_reset,
                                                    const FwObsWriter& out) {
  fw_observation_body<FwShapeGeneric>(E, P, L, c, rng, flags, steps_count, hist_len, at_reset, out);
}
template <class SH, class RNG>
__device__ __forceinline__ void fw_observation(const fw_env_t& E, const fw_sim_t& P, const FwLayout& L,
                                               const FwEnvCtx& c, RNG& rng, uint32_t flags, int steps_count,
                                               int hist_len, bool at_reset, const FwObsWriter& out) {
  if constexpr (SH::fixed) fw_observation_body<SH>(E, P, L, c, rng, flags, steps_count, hist_len, at_reset, out);
  else fw_observation_generic(E, P, L, c, rng, flags, steps_count, hist_len, at_reset, out);
}

// fixed_wing.py:674-774.  a = raw action of this step; steps_count already incremented; error history not yet
// extended with this step's entry (hist_len entries).
template <class SH>
__device__ __forceinline__ double fw_reward(const fw_env_t& E, const fw_sim_t& P, const FwLayout& L, const FwEnvCtx& c,
                                            uint32_t& flags, const double (&a)[FW_N_ACT], bool success,
                                            int steps_count, int hist_len, uint32_t goal_bits) {
  FW_SHAPE_REFS;
  double val_t[FW_N_FCLASS] = {0, 0, 0}, shp_t[FW_N_FCLASS] = {0, 0, 0};
  fw_loop<SH, FW_CNT(n_factors)>(Es.n_factors, [&](int f) FW_LAMBDA_INLINE {
    const fw_factor_t& F = E.fac[f];
    const fw_factor_t& Fs = Es.fac[f];
    double val = 0.0;
    if (Fs.cls == 0) {
      if (Fs.type == 0) {
        val = fabs(a[0]) + fabs(a[1]) + fabs(a[2]);
      } else if (Fs.type == 1) {
        if (steps_count > 1) {
          int lo = steps_count - Fs.window;
          if (lo < 0) lo = 0;
          // sum over (e, j) row-major of |a_e[j] - a_{e-1}[j]|, one running sum, each ring entry loaded once
          if (steps_count - lo >= 2) {
            double prev[FW_N_ACT];
#pragma unroll
            for (int j = 0; j < FW_N_ACT; ++j) prev[j] = fw_ring_get(c, Ls.act_row, Ls.act_depth, FW_N_ACT, j, lo);
            fw_loop_le<SH, 8>(Fs.window - 1, [&](int t) FW_LAMBDA_INLINE {
              const int e = lo + 1 + t;
              if (e < steps_count) {
#pragma unroll
                for (int j = 0; j < FW_N_ACT; ++j) {
                  const double cur = fw_ring_get(c, Ls.act_row, Ls.act_depth, FW_N_ACT, j, e);
                  val += fabs(cur - prev[j]);
                  prev[j] = cur;
                }
              }
            });
          }
        }
      } else {
        double hi = 0.0, lo = 0.0;
#pragma unroll
        for (int j = 0; j < FW_N_ACT; ++j) {
          if (a[j] > E.bounds_max[j]) hi += fabs(a[j] - E.bounds_max[j]);
          if (a[j] < E.bounds_min[j]) lo += fabs(a[j] - E.bounds_min[j]);
        }
        val = hi + lo;
      }
    } else if (Fs.cls == 1) {
      if (Fs.type == 0) {
        val = fw_sv<SH>(c, Fs.ref);
      } else if (Fs.type == 1) {
        val = fw_error(Es.tgt[Fs.ref].wrap, c.D(D_TARGET + Fs.ref), fw_sv<SH>(c, Es.tgt[Fs.ref].sv));
      } else {
        const int W = Es.integration_window;
        int lo = hist_len - W;
        if (lo < 0) lo = 0;
        if (W == 0) lo = 0;   // python: list[-0:] is the whole list
        for (int e = lo; e < hist_len; ++e) val += fw_ring_get(c, Ls.err_row, Ls.err_depth, Es.n_targets, Fs.ref, e);
        if (steps_count < W) val += (double)(W - steps_count) * c.D(D_ERR0 + Fs.ref);
      }
    } else if (Fs.cls == 2) {
      if (success) val = Fs.value_timesteps ? (double)(E.steps_max - steps_count) : F.value;
    } else if (Fs.cls == 3) {
      val = F.value;
    } else {
      if (Fs.type == 0) {
        fw_loop<SH, FW_CNT(n_targets)>(Es.n_targets, [&](int k) FW_LAMBDA_INLINE {
          if (Es.tgt[k].has_bound && ((goal_bits >> k) & 1u)) val += F.value / (double)Es.n_targets;
        });
      } else {
        if (goal_bits >> 31) val += F.value;
      }
    }
    // reward.randomize_scaling: a factor with scaling = [low, high] reads this episode's draw (fw_reset_env)
    const double scaling = Fs.scale_slot1 ? c.D(Ls.rs_row + Fs.scale_slot1 - 1) : F.scaling;
    if (Fs.fclass == 0) {
      val = fabs(val) / scaling;
      if (val < 0.0) val = 0.0;
      if (Fs.has_max && val > F.max) val = F.max;
    } else {
      val = val * val / scaling;
    }
    if (Fs.shaping) shp_t[Fs.fclass] += val * F.sign;
    else val_t[Fs.fclass] += val * F.sign;
  });
  double reward = 0.0;
  fw_loop<SH, FW_CNT(n_terms)>(Es.n_terms, [&](int ti) FW_LAMBDA_INLINE {
    const int fc = Es.term_fclass[ti];
    const bool has_prev = (flags >> (FWF_PREVSHAPE_SHIFT + fc)) & 1u;
    const double prev = c.D(D_PREVSHAPE + fc);
    double val;
    if (fc == 1) {
      if (Es.potential) val = has_prev ? -1.0 + exp(val_t[fc] + (shp_t[fc] - prev)) : -1.0 + exp(val_t[fc]);
      else val = -1.0 + exp(val_t[fc] + shp_t[fc]);
    } else {
      val = val_t[fc];
      if (Es.potential) { if (has_prev) val += shp_t[fc] - prev; }
      else val += shp_t[fc];
    }
    c.D(D_PREVSHAPE + fc) = shp_t[fc];
    flags |= 1u << (FWF_PREVSHAPE_SHIFT + fc);
    reward += E.term_weight[ti] * val;
  });
  return reward;
}

// Euler-angle rotation body<-vehicle times a vector (PyFly._rot_b_v with 3 angles)
__device__ __forceinline__ void fw_rot_euler(double phi, double th, double psi, const double (&w)[3], double (&o)[3]) {
  double sphi, cphi, sth, cth, spsi, cpsi;
  sincos(phi, &sphi, &cphi); sincos(th, &sth, &cth); sincos(psi, &spsi, &cpsi);
  o[0] = cth * cpsi * w[0] + cth * spsi * w[1] - sth * w[2];
  o[1] = (sphi * sth * cpsi - cphi * spsi) * w[0] + (sphi * sth * spsi + cphi * cpsi) * w[1] + sphi * cth * w[2];
  o[2] = (cphi * sth * cpsi + sphi * spsi) * w[0] + (cphi * sth * spsi - sphi * cpsi) * w[1] + cphi * cth * w[2];
}

// Dryden white noise for sim step s of the episode keyed by eptick (4 streams, already scaled)
template <bool INL>
__device__ __forceinline__ void fw_turb_noise_g(const fw_sim_t& P, const FwRng& g, int s, double (&u)[4]) {
  fw_normal2_t<INL>(g, FW_RS_TURB, 2u * (uint32_t)s, u[0], u[1]);
  fw_normal2_t<INL>(g, FW_RS_TURB, 2u * (uint32_t)s + 1u, u[2], u[3]);
#pragma unroll
  for (int j = 0; j < 4; ++j) u[j] *= P.turb_noise_scale;
}
template <bool INL>
__device__ __forceinline__ void fw_turb_noise(const fw_sim_t& P, uint32_t k0, uint32_t k1, uint32_t genv, uint32_t eptick,
                                              int s, double (&u)[4]) {
  FwRng g{k0, k1, genv, eptick};
  fw_turb_noise_g<INL>(P, g, s, u);
}
// ... or the caller's samples (PyFly.reset(turbulence_noise=...), fixed_wing.py:287,308): [4, len, n] unscaled standard
// normals; a step beyond the array wraps around (pyfly: idx % noise.shape[-1])
struct FwTurbInject {
  const double* __restrict__ noise;
  int64_t len, n;
};
// (forceinline, arguments by value: a reference to a member of the kernel's parameter struct handed to an out-of-line
// function makes nvcc copy the whole struct to local memory, after which every pointer loaded from it is GENERIC -
// LD / ST / ATOM instead of LDG / STG / ATOMG throughout the kernel; measured +4 us on the env kernel)
__device__ __forceinline__ void fw_turb_noise_injected(const fw_sim_t& P, const FwTurbInject ti, int64_t env, int s,
                                                       double (&u)[4]) {
  const int64_t col = (int64_t)s % ti.len;
#pragma unroll
  for (int j = 0; j < 4; ++j) u[j] = ti.noise[((int64_t)j * ti.len + col) * ti.n + env] * P.turb_noise_scale;
}

// advance the six shaping filters by one sample (scipy lsim recurrence) and refresh the gust rows.  The host zero-pads
// Ad / Bd0 / Bd1 / C of filters of order < 3 (config.py), so the generic loops are fixed-size and everything stays in
// registers; a fixed shape knows each filter's order and skips the padding (whose states stay exactly zero).
// A mixed shape (SH::mixed) reads the output rows C / D of the episode's level `tlvl` (1..3) instead of the handle's:
// the state recurrence does not depend on the intensity, and the operation order is the same as for filt[f].C / D, so
// an env at level l computes bitwise what a handle of that uniform intensity computes.
template <class SH>
__device__ __forceinline__ void fw_turb_advance(const fw_sim_t& P, const FwEnvCtx& c, const double (&unew)[4],
                                                int tlvl = 0) {
  const fw_sim_t& Ps = SH::sim(P);
#pragma unroll
  for (int f = 0; f < FW_N_FILT; ++f) {
    const fw_filter_t& F = P.filt[f];
    const double* __restrict__ Cf = SH::mixed ? P.turb_C[tlvl][f] : F.C;
    const double Df = SH::mixed ? P.turb_D[tlvl][f] : F.D;
    const int st = Ps.filt[f].stream;
    const int nf = SH::fixed ? Ps.filt[f].n : FW_FILT_MAXN;
    const double up = c.D(D_TU + st);
    const double un = st == 0 ? unew[0] : (st == 1 ? unew[1] : (st == 2 ? unew[2] : unew[3]));
    double x[FW_FILT_MAXN], xn[FW_FILT_MAXN];
#pragma unroll
    for (int a = 0; a < FW_FILT_MAXN; ++a) x[a] = a < nf ? c.D(D_TX + 3 * f + a) : 0.0;
    double yv = Df * un;
#pragma unroll
    for (int b = 0; b < FW_FILT_MAXN; ++b) {
      if (b < nf) {
        double s = up * F.Bd0[b] + un * F.Bd1[b];
#pragma unroll
        for (int a = 0; a < FW_FILT_MAXN; ++a)
          if (a < nf) s += x[a] * F.Ad[a * FW_FILT_MAXN + b];
        xn[b] = s;
        yv += s * Cf[b];
      }
    }
#pragma unroll
    for (int b = 0; b < FW_FILT_MAXN; ++b)
      if (b < nf) c.D(D_TX + 3 * f + b) = xn[b];
    c.D(D_GUST + f) = yv;
  }
#pragma unroll
  for (int j = 0; j < 4; ++j) c.D(D_TU + j) = unew[j];
}


// ---- episode metrics: streaming forms of FixedWingAircraft.get_metric (fixed_wing.py:1095-1162) ---------------------
// The reference recomputes every metric from the full per-episode history lists when an episode ends (it calls
// get_metric from inside step(), :417-419).  Each of them has a forward, O(1)-state form (SURVEY App. A.9):
//   avg_error    |mean(e)/e0|            -> running sum of e, e0                        (nan if |e0| < 0.01)
//   total_error  sum |e|                 -> running sum
//   end_error    |mean(e[-50:])|         -> 50-entry ring
//   overshoot    min / max of e vs e0    -> running min, max
//   rise_time    the reference's backward scan without `break` keeps the EARLIEST index i with |e_i| >= lim and
//                |e_{i+1}| < lim, for lim = low|e0| and high|e0|; rise_time = i_low - i_high (nan if either is missing)
//   success / settling_time              -> first history index whose trailing `streak_req` goal bits have mean >=
//                                           fraction, per bounded target state and for "all" (bit rings + counts)
//   success_time_frac                    -> running count of goal bits / history length
//   control_variation  sum |d command| / (3 dt (n_steps - 1)) over PyFly's constrained command history
// History index 0 is the reset entry; entries are only appended on successful simulator steps, commands on every step.
__device__ __forceinline__ double& fw_md(const FwLayout& L, const FwEnvCtx& c, int r) { return c.D(L.m_drow + r); }
__device__ __forceinline__ int32_t& fw_mi(const FwLayout& L, const FwEnvCtx& c, int r) { return c.I(L.m_irow + r); }

// append goal-history entry `idx` (bits from fw_goal_status; the "all" ring / count are maintained by the caller)
__device__ __forceinline__ void fw_metrics_goal(const fw_env_t& E, const FwLayout& L, const FwEnvCtx& c, uint32_t gb,
                                                int idx) {
  const int req = E.streak_req;
  if (req <= 0) return;
  const int slot = idx % req, wd = slot >> 5, bit = slot & 31;
  for (int k = 0; k < E.n_targets; ++k) {
    if (!E.tgt[k].has_bound) continue;
    const int nb = (gb >> k) & 1u;
    uint32_t word = (uint32_t)fw_mi(L, c, MI_GRING + k * L.goal_words + wd);
    const int ob = (word >> bit) & 1u;
    word = (word & ~(1u << bit)) | ((uint32_t)nb << bit);
    fw_mi(L, c, MI_GRING + k * L.goal_words + wd) = (int32_t)word;
    const int cnt = fw_mi(L, c, MI_GCNT + k) + nb - ob;
    fw_mi(L, c, MI_GCNT + k) = cnt;
    fw_mi(L, c, MI_GSUM + k) += nb;
    if (fw_mi(L, c, MI_SETTLE + k) < 0 && idx + 1 >= req && (double)cnt / (double)req >= E.streak_fraction)
      fw_mi(L, c, MI_SETTLE + k) = idx;
  }
  fw_mi(L, c, MI_GSUM + 3) += (int)(gb >> 31);
  if (fw_mi(L, c, MI_SETTLE + 3) < 0 && idx + 1 >= req &&
      (double)c.I(I_GOALCNT) / (double)req >= E.streak_fraction)
    fw_mi(L, c, MI_SETTLE + 3) = idx;
}

// append error-history entry `idx` of target k
__device__ __forceinline__ void fw_metrics_error(const fw_env_t& E, const FwLayout& L, const FwEnvCtx& c, int k,
                                                 double e, int idx) {
  const double ae = fabs(e);
  if (idx == 0) {
    fw_md(L, c, MD_SUME + k) = e;
    fw_md(L, c, MD_SUMABS + k) = ae;
    fw_md(L, c, MD_MIN + k) = e;
    fw_md(L, c, MD_MAX + k) = e;
    fw_mi(L, c, MI_RISE_LO + k) = -1;
    fw_mi(L, c, MI_RISE_HI + k) = -1;
  } else {
    fw_md(L, c, MD_SUME + k) += e;
    fw_md(L, c, MD_SUMABS + k) += ae;
    if (e < fw_md(L, c, MD_MIN + k)) fw_md(L, c, MD_MIN + k) = e;
    if (e > fw_md(L, c, MD_MAX + k)) fw_md(L, c, MD_MAX + k) = e;
    const double pa = fw_md(L, c, MD_PREVABS + k);     // |e_{idx-1}|
    const double a0 = fabs(c.D(D_ERR0 + k));
    const double lo = fabs(E.rise_low * c.D(D_ERR0 + k)), hi = fabs(E.rise_high * c.D(D_ERR0 + k));
    (void)a0;
    if (fw_mi(L, c, MI_RISE_LO + k) < 0 && pa >= lo && ae < lo) fw_mi(L, c, MI_RISE_LO + k) = idx - 1;
    if (fw_mi(L, c, MI_RISE_HI + k) < 0 && pa >= hi && ae < hi) fw_mi(L, c, MI_RISE_HI + k) = idx - 1;
  }
  fw_md(L, c, MD_PREVABS + k) = ae;
  c.D(L.end_row + (idx % FW_END_WINDOW) * E.n_targets + k) = e;
}

// every simulator step (also a failing one) appends the constrained commands to PyFly's actuator histories
__device__ __forceinline__ void fw_metrics_command(const FwLayout& L, const FwEnvCtx& c, int n_steps) {
  double s = 0.0;
  for (int j = 0; j < 3; ++j) {
    const double cmd = c.D(D_CMD + j);
    if (n_steps > 1) s += fabs(cmd - fw_md(L, c, MD_PREVCMD + j));
    fw_md(L, c, MD_PREVCMD + j) = cmd;
  }
  if (n_steps > 1) fw_md(L, c, MD_CV) += s;
  else fw_md(L, c, MD_CV) = 0.0;
}

// episode end: one row of fw_episode_dim doubles (layout.h EP_*)
__device__ __forceinline__ void fw_metrics_finish(const fw_env_t& E, const fw_sim_t& P, const FwLayout& L,
                                                  const FwEnvCtx& c, int n, int n_steps, double ep_return,
                                                  double* __restrict__ out) {
  const double nan = __longlong_as_double(0x7ff8000000000000ll);
  out[EP_RETURN] = ep_return;
  out[EP_LENGTH] = (double)n_steps;
  out[EP_CV] = fw_md(L, c, MD_CV) / (3.0 * P.dt * (double)(n_steps - 1));   // 0/0 = nan for a 1-step episode
  const bool goal = E.streak_req > 0;
  out[EP_SUCCESS_ALL] = goal ? (fw_mi(L, c, MI_SETTLE + 3) >= 0 ? 1.0 : 0.0) : nan;
  out[EP_SETTLE_ALL] = (goal && fw_mi(L, c, MI_SETTLE + 3) >= 0) ? (double)fw_mi(L, c, MI_SETTLE + 3) : nan;
  out[EP_STF_ALL] = goal ? (double)fw_mi(L, c, MI_GSUM + 3) / (double)n : nan;
  for (int k = 0; k < E.n_targets; ++k) {
    double* o = out + EP_PER_TARGET + k * EPT_N;
    const double e0 = c.D(D_ERR0 + k);
    o[EPT_AVG] = fabs(e0) >= 0.01 ? fabs((fw_md(L, c, MD_SUME + k) / (double)n) / e0) : nan;
    o[EPT_TOTAL] = fw_md(L, c, MD_SUMABS + k);
    const int m = n < FW_END_WINDOW ? n : FW_END_WINDOW;
    double s = 0.0;
    for (int i = n - m; i < n; ++i) s += c.D(L.end_row + (i % FW_END_WINDOW) * E.n_targets + k);
    o[EPT_END] = fabs(s / (double)m);
    const int rl = fw_mi(L, c, MI_RISE_LO + k), rh = fw_mi(L, c, MI_RISE_HI + k);
    o[EPT_RISE] = (rl >= 0 && rh >= 0) ? (double)(rl - rh) : nan;
    const double opp = e0 > 0 ? fw_md(L, c, MD_MIN + k) : fw_md(L, c, MD_MAX + k);
    const int so = (opp > 0) - (opp < 0), s0 = (e0 > 0) - (e0 < 0);
    o[EPT_OVERSHOOT] = so == s0 ? nan : fabs(opp / e0);
    const bool gk = goal && E.tgt[k].has_bound;
    o[EPT_SUCCESS] = gk ? (fw_mi(L, c, MI_SETTLE + k) >= 0 ? 1.0 : 0.0) : nan;
    o[EPT_SETTLE] = (gk && fw_mi(L, c, MI_SETTLE + k) >= 0) ? (double)fw_mi(L, c, MI_SETTLE + k) : nan;
    o[EPT_STF] = gk ? (double)fw_mi(L, c, MI_GSUM + k) / (double)n : nan;
  }
}

// histories restart at reset: entry 0
__device__ __forceinline__ void fw_metrics_reset(const fw_env_t& E, const FwLayout& L, const FwEnvCtx& c, uint32_t gb) {
  for (int r = 0; r < MI_GRING + 3 * L.goal_words; ++r) fw_mi(L, c, r) = 0;
  for (int k = 0; k < 4; ++k) fw_mi(L, c, MI_SETTLE + k) = -1;
  fw_md(L, c, MD_CV) = 0.0;
  for (int k = 0; k < E.n_targets; ++k) fw_metrics_error(E, L, c, k, c.D(D_ERR0 + k), 0);
  fw_metrics_goal(E, L, c, gb, 0);
}

// PyFly.reset + FixedWingAircraft.reset for one env.  init_state rows: FW_N_SV + 3 (wind n,e,d); NaN = sample.
// SH-templated and out of line: episode ends are rare, so the step path of every instantiation keeps this code out
// of its straight-line block; inside, a fixed shape still folds (the shape is taken from SH, not from arguments).
// COOP (fw_env_kernel's auto-resets): the WHOLE WARP runs this function for one env - identical inputs, identical control
// flow, every lane writes the same values to the same state rows (one of the writes lands; CUDA defines that) and only
// the lane that owns the env writes observations (out.commit).  What it buys: the reset's ~30 Philox blocks are computed
// once, two per lane, and broadcast by shuffles (philox.cuh, FwRng::coop) instead of one lane computing them in series
// while 31 wait.
template <class SH, bool COOP = false>
__device__ __forceinline__ void fw_reset_env_body(const fw_env_t& E, const fw_sim_t& P, const FwLayout& L, const FwEnvCtx& c,
                                                  uint32_t k0, uint32_t k1, uint32_t genv,
                                                  const double* __restrict__ init_state,
                                                  const double* __restrict__ init_target, int64_t in_stride,
                                                  const FwTurbInject ti, const FwObsWriter& out) {
  FW_SHAPE_REFS;
  const uint32_t tick = (uint32_t)c.I(I_TICK);
  if constexpr (COOP) __syncwarp();     // every lane has read the counter before any lane overwrites it
  c.I(I_TICK) = (int32_t)(tick + 1u);
  c.I(I_EPTICK) = (int32_t)tick;
  FwRng g{k0, k1, genv, tick};
  if constexpr (COOP) fw_rng_fill_bank(g);
  int dummy = 0;
  auto given = [&](int r, double& v) -> bool {
    if (!init_state) return false;
    v = init_state[(int64_t)r * in_stride + c.env];
    return !isnan(v);
  };
  auto init_var = [&](int sv) -> double {
    double v;
    if (given(sv, v)) return fw_cond_wrap<double>(P.var[sv], sv, v, dummy);
    // (fixed shapes inline Philox: the ~15 independent draws of a reset interleave instead of running as serial calls -
    // a reset is ONE lane of a warp working while 31 wait, and half of the env blocks of a step contain one)
    return fw_uniform<SH::fixed>(g, FW_RS_INIT, (uint32_t)sv, P.var[sv].init_min, P.var[sv].init_max);
  };
  // ---- PyFly.reset ----
  const double roll = init_var(FW_SV_ROLL), pitch = init_var(FW_SV_PITCH), yaw = init_var(FW_SV_YAW);
  c.D(D_ROLL) = roll; c.D(D_PITCH) = pitch; c.D(D_YAW) = yaw;
  for (int j = 0; j < 3; ++j) c.D(D_OMEGA + j) = init_var(FW_SV_OMEGA_P + j);
  for (int j = 0; j < 3; ++j) c.D(D_POS + j) = init_var(FW_SV_POS_N + j);
  double vel[3];
  for (int j = 0; j < 3; ++j) { vel[j] = init_var(FW_SV_VEL_U + j); c.D(D_VEL + j) = vel[j]; }
  const int act_sv[3] = {FW_SV_ELEVON_L, FW_SV_ELEVON_R, FW_SV_THROTTLE};
  double act[3];
  for (int j = 0; j < 3; ++j) { act[j] = init_var(act_sv[j]); c.D(D_ACT + j) = act[j]; c.D(D_ACTDOT + j) = 0.0; }
  c.D(D_ELEV) = fw_cond<double>(P.var[FW_SV_ELEVATOR], FW_SV_ELEVATOR, (act[1] + act[0]) / 2, dummy);
  c.D(D_AIL) = fw_cond<double>(P.var[FW_SV_AILERON], FW_SV_AILERON, (-act[1] + act[0]) / 2, dummy);
  for (int j = 0; j < 3; ++j) c.D(D_CMD + j) = 0.0;
  double wind[3] = {0, 0, 0};
  {
    double wv[3];
    const bool have = given(FW_N_SV + 0, wv[0]) & given(FW_N_SV + 1, wv[1]) & given(FW_N_SV + 2, wv[2]);
    if (have) { wind[0] = wv[0]; wind[1] = wv[1]; wind[2] = wv[2]; }
    else {
      // counter-based draws: with a zero magnitude range all three are exactly 0 whatever the random words, so the
      // Philox blocks can be skipped without moving any other draw
      if (P.wind_mag_min != 0.0 || P.wind_mag_max != 0.0) {
        const double mag = fw_uniform<SH::fixed>(g, FW_RS_WIND, 0, P.wind_mag_min, P.wind_mag_max);
        wind[0] = fw_uniform<SH::fixed>(g, FW_RS_WIND, 1, -mag, mag);
        const double we_max = sqrt(mag * mag - wind[0] * wind[0]);
        wind[1] = fw_uniform<SH::fixed>(g, FW_RS_WIND, 2, -we_max, we_max);
        wind[2] = sqrt(mag * mag - wind[0] * wind[0] - wind[1] * wind[1]);
      }
    }
  }
  for (int j = 0; j < 3; ++j) c.D(D_WIND + j) = wind[j];
  // Dryden: x = 0, first sample drawn, gust = D*u0
  for (int j = 0; j < 18; ++j) c.D(D_TX + j) = 0.0;
  double gl[3] = {0, 0, 0};
  // mixed handle: the episode's intensity, the requested level or one draw of its own stream (no other draw moves);
  // level 0 (none) then takes exactly the path of a handle without turbulence
  int tlvl = 0;
  if constexpr (SH::mixed) {
    const int req = c.I(Ls.tl_row);
    if (req >= 0) {
      tlvl = req;
    } else {
      const double u = fw_uniform01<SH::fixed>(g, FW_RS_TURBLVL, 0);
      tlvl = (u >= P.turb_cdf[0]) + (u >= P.turb_cdf[1]) + (u >= P.turb_cdf[2]);   // first l with u < cdf[l]
    }
    c.I(Ls.tl_row + 1) = tlvl;
  }
  // (the condition is spelled out at both of its uses, not kept in a variable: a handle without per-env levels then
  // compiles to exactly the code it compiled to before they existed)
  if (SH::mixed ? tlvl != 0 : Ps.turbulence != 0) {
    double u0[4];
    if (ti.noise) fw_turb_noise_injected(P, ti, c.env, 0, u0);
    else fw_turb_noise_g<SH::fixed>(P, g, 0, u0);
    for (int j = 0; j < 4; ++j) c.D(D_TU + j) = u0[j];
#pragma unroll
    for (int f = 0; f < FW_N_FILT; ++f) {
      const int st = Ps.filt[f].stream;
      const double Df = SH::mixed ? P.turb_D[tlvl][f] : P.filt[f].D;
      const double gv = Df * (st == 0 ? u0[0] : (st == 1 ? u0[1] : (st == 2 ? u0[2] : u0[3])));
      c.D(D_GUST + f) = gv;
      if (f < 3) gl[f] = gv;
    }
  } else {
    for (int j = 0; j < 4; ++j) c.D(D_TU + j) = 0.0;
    for (int j = 0; j < 6; ++j) c.D(D_GUST + j) = 0.0;
  }
  // Va, alpha, beta from the Euler-angle rotation of the steady wind + gust
  double wb[3] = {0.0, 0.0, 0.0};
  if (wind[0] != 0.0 || wind[1] != 0.0 || wind[2] != 0.0) fw_rot_euler(roll, pitch, yaw, wind, wb);   // (R * 0 = 0)
  const double ur = vel[0] - (wb[0] + gl[0]), vr = vel[1] - (wb[1] + gl[1]), wr = vel[2] - (wb[2] + gl[2]);
  // branch-free fwmath routines as in the step path (fw_commit_step): asin(vr / Va) = atan2(vr, hypot(ur, wr))
  const double hxz2 = ur * ur + wr * wr;
  const double Va = fwm_sqrt(hxz2 + vr * vr);
  c.D(D_VA) = fw_cond<double>(P.var[FW_SV_VA], FW_SV_VA, Va, dummy);
  c.D(D_ALPHA) = fw_cond<double>(P.var[FW_SV_ALPHA], FW_SV_ALPHA, fwm_atan2(wr, ur), dummy);
  c.D(D_BETA) = fw_cond<double>(P.var[FW_SV_BETA], FW_SV_BETA, fwm_atan2(vr, fwm_sqrt(hxz2)), dummy);
  {
    double sphi, cphi, sth, cth, spsi, cpsi;
    // sin / cos of the half angles through sincospi (straight-line; the libdevice sincos slow path is ~3x the code)
    const double inv2pi = 0.15915494309189535;   // 1 / (2 pi)
    fwm_sincospi(roll * inv2pi, &sphi, &cphi); fwm_sincospi(pitch * inv2pi, &sth, &cth); fwm_sincospi(yaw * inv2pi, &spsi, &cpsi);
    c.D(D_Q + 0) = cpsi * cth * cphi + spsi * sth * sphi;
    c.D(D_Q + 1) = cpsi * cth * sphi - spsi * sth * cphi;
    c.D(D_Q + 2) = cpsi * sth * cphi + spsi * cth * sphi;
    c.D(D_Q + 3) = spsi * cth * cphi - cpsi * sth * sphi;
  }
  // ---- FixedWingAircraft.reset ----
  uint32_t flags = (uint32_t)c.I(I_FLAGS);
  const int old_hist_len = c.I(I_HISTLEN);
  c.I(I_STEPS) = 0;
  FwEnvRngT<SH::fixed> rng{g, 0u, 0u, 0.0};
  // sample_simulator_parameters (fixed_wing.py:523-570) runs between simulator.reset and sample_target (:308-310) and
  // draws from the env's generator in table order.  Fixed shapes have no table (n_rand == 0).
  if (Es.n_rand > 0) {
    for (int j = 0; j < E.n_rand; ++j) {
      const fw_rand_t& r = E.rand[j];
      double v;
      if (r.dist == 0) {
        v = rng.normal(r.orig, r.var);
        if (r.has_clip) { v = fmax(v, r.orig - r.clip); v = fmin(v, r.orig + r.clip); }   // np.clip order
      } else if (r.dist == 1) {
        v = rng.uniform(r.orig - r.var, r.orig + r.var);
      } else {
        v = rng.uniform(r.orig, r.var);
      }
      if (r.slot1) c.D(Ls.par_row + r.slot1 - 1) = v;
    }
    // derived rows: what the right-hand side multiplies by instead of dividing / exponentiating at every evaluation
    auto par = [&](int id, double shared) -> double {
      const int s1 = P.par_slot1[id];
      return s1 ? c.D(Ls.par_row + s1 - 1) : shared;
    };
    if (P.par_slot1[FW_PAR_INV_MASS]) c.D(Ls.par_row + P.par_slot1[FW_PAR_INV_MASS] - 1) = 1.0 / par(FW_PAR_MASS, P.mass);
    if (P.par_slot1[FW_PAR_INV_PI_E_AR])
      c.D(Ls.par_row + P.par_slot1[FW_PAR_INV_PI_E_AR] - 1) = 1.0 / (CUDART_PI * par(FW_PAR_E, P.e) * par(FW_PAR_AR, P.ar));
    if (P.par_slot1[FW_PAR_EXP_2MA0])
      c.D(Ls.par_row + P.par_slot1[FW_PAR_EXP_2MA0] - 1) = exp(2.0 * par(FW_PAR_M, P.M) * par(FW_PAR_A_0, P.a_0));
  }
  fw_sample_target<SH>(E, c, rng, flags, 0);
  if (init_target) {
    for (int k = 0; k < Es.n_targets; ++k) {
      const double v = init_target[(int64_t)k * in_stride + c.env];
      if (isnan(v)) continue;
      const int cls = fw_tcls(flags, k);
      if (cls != 0 && cls != 3) flags &= ~(3u << (FWF_TCLS_SHIFT + 2 * k));
      c.D(D_TARGET + k) = v;
    }
  }
  // observation BEFORE the histories are rebuilt (fixed_wing.py:317 vs :318): the PyFly state histories are new
  // (hist_len 1) but the integrator still reads the previous episode's error history.
  fw_observation<SH>(E, P, L, c, rng, flags, 0, (flags & FWF_HIST_VALID) ? old_hist_len : 1, true, out);
  // rebuild histories
  c.I(I_HISTLEN) = 1;
  fw_loop<SH, FW_CNT(n_targets)>(Es.n_targets, [&](int k) FW_LAMBDA_INLINE {
    const double err = fw_error(Es.tgt[k].wrap, c.D(D_TARGET + k), fw_sv<SH>(c, Es.tgt[k].sv));
    c.D(D_ERR0 + k) = err;
    if (Ls.err_depth > 0) fw_ring_put(c, Ls.err_row, Ls.err_depth, Es.n_targets, k, 0, err);
    if (Ls.tgt_depth > 0) fw_ring_put(c, Ls.tgt_row, Ls.tgt_depth, Es.n_targets, k, 0, c.D(D_TARGET + k));
  });
  if (Ls.sv_depth > 1)
    fw_loop<SH, FW_CNT(obs_nvar)>(Es.obs_nvar, [&](int v) FW_LAMBDA_INLINE {
      if (Es.obs[v].type == 0)
        fw_ring_put(c, Ls.sv_row, Ls.sv_depth, Ls.n_sv_obs, Ls.sv_slot[v], 0, fw_sv<SH>(c, Es.obs[v].ref));
    });
  uint32_t gb0 = 0u;
  if (Es.streak_req > 0) {
    for (int wd = 0; wd < Ls.goal_words; ++wd) c.I(I_GOALRING + wd) = 0;
    const uint32_t gb = fw_goal_status<SH>(E, c);
    gb0 = gb;
    const int all = (int)(gb >> 31);
    if (all) c.I(I_GOALRING) = 1;
    c.I(I_GOALCNT) = all;
  }
  flags |= FWF_HIST_VALID;
  flags &= ~(7u << FWF_PREVSHAPE_SHIFT);
  flags &= ~(FWF_EP_SUCCESS | FWF_TURB_INJ);
  if (ti.noise && (SH::mixed ? tlvl != 0 : Ps.turbulence != 0)) flags |= FWF_TURB_INJ;
  // reward.randomize_scaling (fixed_wing.py:330-334): after the observation and the history rebuild, one uniform draw
  // per factor configured with scaling = [low, high], in factor order
  if (Es.n_scale_rows > 0)
    for (int f = 0; f < Es.n_factors; ++f)
      if (Es.fac[f].scale_slot1)
        c.D(Ls.rs_row + Es.fac[f].scale_slot1 - 1) = rng.uniform(E.fac[f].scale_low, E.fac[f].scale_high);
  c.I(I_FLAGS) = (int32_t)flags;
  c.I(I_STATUS) = 0;
  c.I(I_LASTK) = 0;
  c.D(D_EPRET) = 0.0;
  if (Ls.met) fw_metrics_reset(E, L, c, gb0);
}
// out of line: the explicit-reset kernel (one thread per env)
template <class SH>
__device__ __noinline__ void fw_reset_env(const fw_env_t& E, const fw_sim_t& P, const FwLayout& L, const FwEnvCtx& c,
                                          uint32_t k0, uint32_t k1, uint32_t genv, const double* __restrict__ init_state,
                                          const double* __restrict__ init_target, int64_t in_stride,
                                          const FwTurbInject ti, const FwObsWriter& out) {
  fw_reset_env_body<SH, false>(E, P, L, c, k0, k1, genv, init_state, init_target, in_stride, ti, out);
}
