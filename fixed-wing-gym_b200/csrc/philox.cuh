// Counter-based per-env RNG: Philox4x32-10 (Salmon et al., SC'11).  The reference draws from numpy MT19937
// (fixed_wing.py:57,220; PyFly per-variable RandomState); this framework replaces that with a keyed counter so any
// sharding of envs over GPUs produces identical per-env streams (SURVEY §8e).  oracle/philox.py is the numpy twin.
//
// counter = (global env id, tick, stream, index), key = 64-bit seed.
//   tick   : per-env count of reset()/step() calls since seeding; each call uses its own tick.
//   stream : FW_RS_* below.
//   index  : draw index inside (tick, stream).
#pragma once
#include <stdint.h>
#include "fwmath.cuh"

#define FW_RS_INIT 0    // PyFly Variable.reset uniform draws, index = fw_sv id
#define FW_RS_WIND 1    // steady wind magnitude / components
#define FW_RS_TURB 2    // Dryden white noise; tick = episode tick, index = 2*sim_step + {0,1}
#define FW_RS_ENV_U 3   // env-side uniform draws in call order (target sampling, init noise)
#define FW_RS_ENV_N 4   // env-side normal draws in call order (observation noise), two per block
#define FW_RS_TURBLVL 5 // Dryden intensity of a mixed handle's episode (one uniform at the reset's tick, index 0)

// Two forms of every generator.  INL = false (generic, table-walking env kernels): out of line on purpose, ~100
// instructions x ~25 call sites would otherwise dominate that kernel's code size.  INL = true (shape-specialised
// kernels, env_shapes.h): inlined, so the independent draws of one env step (7 noise pairs + 2 gust pairs)
// interleave instead of running as serial calls.
__device__ __forceinline__ void fw_philox4x32_10_inl(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3,
                                                     uint32_t k0, uint32_t k1, uint32_t out[4]) {
  const uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u, W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    uint64_t p0 = (uint64_t)M0 * c0, p1 = (uint64_t)M1 * c2;
    uint32_t hi0 = (uint32_t)(p0 >> 32), lo0 = (uint32_t)p0, hi1 = (uint32_t)(p1 >> 32), lo1 = (uint32_t)p1;
    uint32_t n0 = hi1 ^ c1 ^ k0, n2 = hi0 ^ c3 ^ k1;
    c0 = n0; c1 = lo1; c2 = n2; c3 = lo0;
    k0 += W0; k1 += W1;
  }
  out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}

__device__ __noinline__ void fw_philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3,
                                              uint32_t k0, uint32_t k1, uint32_t out[4]) {
  fw_philox4x32_10_inl(c0, c1, c2, c3, k0, k1, out);
}

// coop (fw_env_kernel's warp-cooperative auto-reset): ALL 32 lanes of the warp run the reset of ONE env together, so
// they draw the same (stream, idx) at the same instruction.  The Philox blocks of that (env, tick) are then computed ONCE,
// two per lane (bank: slots `lane` and `32 + lane` of fw_pc_slot's numbering), and a draw is four shuffles instead of a
// 90-instruction block: a reset is ~30 draws and was ~60 % Philox.  Same counters, same words, same values.
struct FwRng {
  uint32_t k0, k1, env, tick;
  bool coop = false;
  uint32_t bank[8] = {0u, 0u, 0u, 0u, 0u, 0u, 0u, 0u};
  double zbank[4] = {0.0, 0.0, 0.0, 0.0};   // Box-Muller pairs of this lane's two blocks (used for the TURB / ENV_N slots)
};
#define FW_PC_SLOTS 64
// (stream, idx) <-> slot: INIT idx = fw_sv id 0..20 | WIND 0..2 | TURB 0..1 | ENV_U 0..13 | ENV_N 0..23; -1: not banked
__device__ __forceinline__ int fw_pc_slot(uint32_t stream, uint32_t idx) {
  // branch-free for run-time arguments: first slot and slot count of the stream, one byte each
  const uint32_t first = (uint32_t)(0x281a181500ull >> (8u * stream)) & 0xffu;    // 0, 21, 24, 26, 40
  const uint32_t count = (uint32_t)(0x180e020315ull >> (8u * stream)) & 0xffu;    // 21, 3, 2, 14, 24
  return (stream < 5u && idx < count) ? (int)(first + idx) : -1;
}
__device__ __forceinline__ void fw_pc_unslot(int slot, uint32_t& stream, uint32_t& idx) {
  if (slot < 21) { stream = 0u; idx = (uint32_t)slot; }
  else if (slot < 24) { stream = 1u; idx = (uint32_t)(slot - 21); }
  else if (slot < 26) { stream = 2u; idx = (uint32_t)(slot - 24); }
  else if (slot < 40) { stream = 3u; idx = (uint32_t)(slot - 26); }
  else { stream = 4u; idx = (uint32_t)(slot - 40); }
}
// one Philox block of the generator: from the warp's bank when it holds it (cooperative mode), else computed
template <bool INL>
__device__ __forceinline__ void fw_block(const FwRng& g, uint32_t stream, uint32_t idx, uint32_t (&w)[4]) {
  if (g.coop) {
    const int s = fw_pc_slot(stream, idx);
    if (s >= 0) {                       // warp-uniform (all lanes draw the same block)
      const int src = s & 31;
      const bool hi = s >= 32;
#pragma unroll
      for (int k = 0; k < 4; ++k)       // `hi` is warp-uniform: every lane selects its own word first, then one shuffle
        w[k] = __shfl_sync(0xffffffffu, hi ? g.bank[4 + k] : g.bank[k], src);
      return;
    }
  }
  if constexpr (INL) fw_philox4x32_10_inl(g.env, g.tick, stream, idx, g.k0, g.k1, w);
  else fw_philox4x32_10(g.env, g.tick, stream, idx, g.k0, g.k1, w);
}

// 53-bit uniform in [0,1) from two words (same construction as numpy's random_sample: (a>>5, b>>6))
__device__ __forceinline__ double fw_u53(uint32_t a, uint32_t b) {
  return ((double)(a >> 5) * 67108864.0 + (double)(b >> 6)) * (1.0 / 9007199254740992.0);
}

template <bool INL = false>
__device__ __forceinline__ double fw_uniform01(const FwRng& g, uint32_t stream, uint32_t idx) {
  uint32_t w[4];
  fw_block<INL>(g, stream, idx, w);
  return fw_u53(w[0], w[1]);
}

template <bool INL = false>
__device__ __forceinline__ double fw_uniform(const FwRng& g, uint32_t stream, uint32_t idx, double lo, double hi) {
  return lo + (hi - lo) * fw_uniform01<INL>(g, stream, idx);   // numpy: low + (high-low)*random_sample()
}

// two standard normals per Philox block (Box-Muller); u1 in (0,1] so the log is finite
__device__ __forceinline__ void fw_box_muller(const uint32_t (&w)[4], double& z0, double& z1);
__device__ __forceinline__ void fw_normal2_inl(const FwRng& g, uint32_t stream, uint32_t idx, double& z0, double& z1) {
  if (g.coop) {                         // cooperative reset: the pair was computed by the lane that holds the block
    const int s = fw_pc_slot(stream, idx);
    if (s >= 0) {
      const int src = s & 31;
      const bool hi = s >= 32;
      z0 = __shfl_sync(0xffffffffu, hi ? g.zbank[2] : g.zbank[0], src);
      z1 = __shfl_sync(0xffffffffu, hi ? g.zbank[3] : g.zbank[1], src);
      return;
    }
  }
  uint32_t w[4];
  fw_block<true>(g, stream, idx, w);
  fw_box_muller(w, z0, z1);
}
__device__ __forceinline__ void fw_box_muller(const uint32_t (&w)[4], double& z0, double& z1) {
  double u1 = 1.0 - fw_u53(w[0], w[1]);
  double u2 = fw_u53(w[2], w[3]);
  // branch-free fwmath routines (csrc/fwmath.cuh): 14 observation-noise draws + 4 gust draws per env step make
  // this the env kernel's largest block of arithmetic
  double r = fwm_sqrt(-2.0 * fwm_log(u1));
  double s, c;
  fwm_sincospi(2.0 * u2, &s, &c);
  z0 = r * c;
  z1 = r * s;
}
// fill the bank of a cooperative generator (every lane of the warp must call)
__device__ __forceinline__ void fw_rng_fill_bank(FwRng& g) {
  const int lane = threadIdx.x & 31;
#pragma unroll
  for (int r = 0; r < 2; ++r) {
    uint32_t stream, idx, w[4];
    fw_pc_unslot(r * 32 + lane, stream, idx);
    fw_philox4x32_10_inl(g.env, g.tick, stream, idx, g.k0, g.k1, w);
#pragma unroll
    for (int k = 0; k < 4; ++k) g.bank[4 * r + k] = w[k];
    // the normal pair of the block, whatever its stream (one uniform evaluation per round for the whole warp; only the
    // TURB slots of round 0 and the ENV_N slots of round 1 are ever asked for)
    fw_box_muller(w, g.zbank[2 * r], g.zbank[2 * r + 1]);
  }
  g.coop = true;
}

__device__ __noinline__ void fw_normal2(const FwRng& g, uint32_t stream, uint32_t idx, double& z0, double& z1) {
  fw_normal2_inl(g, stream, idx, z0, z1);
}
template <bool INL>
__device__ __forceinline__ void fw_normal2_t(const FwRng& g, uint32_t stream, uint32_t idx, double& z0, double& z1) {
  if constexpr (INL) fw_normal2_inl(g, stream, idx, z0, z1);
  else fw_normal2(g, stream, idx, z0, z1);
}
