// root_noise.cuh — EXTENSION (not in the reference, mcts.rs:204-207 is a TODO): Dirichlet noise on the root priors,
// drawn on the device (DESIGN.md §4.6).
//
// eta ~ Dir(alpha) over the n children of a root is drawn by one warp, lane i owning children i, i + 32, ... :
//   * gamma_i ~ Gamma(alpha) by Marsaglia–Tsang for shape a = alpha (alpha >= 1) or a = alpha + 1 with the boost
//     gamma = gamma_{a} * U^(1/alpha) (alpha < 1); carried as log gamma so that a small alpha cannot underflow;
//   * every uniform / normal (Box–Muller) comes from splitmix64 counters keyed by (root key, child, attempt, draw);
//   * at most NOISE_ATTEMPTS proposals per child; if all are rejected (probability < 0.05^32) log gamma = log d;
//   * eta_i = exp(lg_i - max) / sum, the sum in a fixed order (lane order within a round, rounds ascending, then an
//     xor butterfly whose partial sums are the same on every lane), so the result is deterministic.
// The key is a pure function of (seed, global game id, root ply, n): a domain constant keeps the stream apart from the
// temperature sampler's, which is keyed by the same kind of (seed, game id, ply) triple.
#pragma once
#include "games.cuh"

namespace spb {

constexpr uint64_t NOISE_DOMAIN = 0xD1E1C41E7B00A5EDull;
constexpr int NOISE_ATTEMPTS = 32;

__host__ __device__ __forceinline__ uint64_t noise_key(uint64_t seed, uint64_t game_id, uint32_t ply, uint32_t n) {
  return splitmix64(seed ^ splitmix64(NOISE_DOMAIN ^ splitmix64(game_id ^ splitmix64(((uint64_t)ply << 16) | n))));
}

// uniform in (0, 1]: never 0, so its logarithm is finite
__device__ __forceinline__ float noise_uniform(uint64_t key, uint32_t child, uint32_t attempt, uint32_t draw) {
  const uint64_t h = splitmix64(key ^ splitmix64(((uint64_t)child << 16) | ((uint64_t)attempt << 2) | draw));
  return (float)((h >> 40) + 1ull) * (1.0f / 16777216.0f);
}

// log of one Gamma(alpha) variate for child `child` of the root with key `key`
__device__ __forceinline__ float noise_log_gamma(uint64_t key, uint32_t child, float alpha) {
  const bool boost = alpha < 1.0f;
  const float a = boost ? alpha + 1.0f : alpha;
  const float d = a - 1.0f / 3.0f;
  const float c = 1.0f / sqrtf(9.0f * d);
  float lg = logf(d);                                                    // fallback: every proposal rejected
  for (uint32_t k = 0; k < (uint32_t)NOISE_ATTEMPTS; ++k) {
    const float u1 = noise_uniform(key, child, k, 0), u2 = noise_uniform(key, child, k, 1);
    const float x = sqrtf(-2.0f * logf(u1)) * cospif(2.0f * u2);
    const float t = 1.0f + c * x;
    if (t <= 0.0f) continue;
    const float v = t * t * t;
    const float u = noise_uniform(key, child, k, 2);
    if (logf(u) < 0.5f * x * x + d - d * v + d * logf(v)) { lg = logf(d) + logf(v); break; }
  }
  if (boost) lg += logf(noise_uniform(key, child, NOISE_ATTEMPTS, 3)) / alpha;
  return lg;
}

// eta of one root by the whole warp: out[0..n) (child order) and zeros in out[n..cap).  ROUNDS * 32 >= n.
template <int ROUNDS>
__device__ __forceinline__ void warp_dirichlet(uint64_t key, uint32_t n, float alpha, int lane, float* out, uint32_t cap) {
  float lg[ROUNDS];
  float mx = -INFINITY;
#pragma unroll
  for (int r = 0; r < ROUNDS; ++r) {
    const uint32_t i = (uint32_t)r * 32u + (uint32_t)lane;
    lg[r] = i < n ? noise_log_gamma(key, i, alpha) : -INFINITY;
    mx = fmaxf(mx, lg[r]);
  }
#pragma unroll
  for (int o = 16; o >= 1; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
  float s = 0.0f;
#pragma unroll
  for (int r = 0; r < ROUNDS; ++r) {
    const uint32_t i = (uint32_t)r * 32u + (uint32_t)lane;
    lg[r] = i < n ? expf(lg[r] - mx) : 0.0f;
    s += lg[r];
  }
#pragma unroll
  for (int o = 16; o >= 1; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
#pragma unroll
  for (int r = 0; r < ROUNDS; ++r) {
    const uint32_t i = (uint32_t)r * 32u + (uint32_t)lane;
    if (i < n) out[i] = lg[r] / s;
  }
  for (uint32_t i = n + (uint32_t)lane; i < cap; i += 32u) out[i] = 0.0f;
}

}  // namespace spb
