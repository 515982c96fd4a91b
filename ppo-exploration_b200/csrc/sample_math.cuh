// Per-element math of the policy's action sampling (models.py:30-50 / 75-99), shared by ppx_policy_sample (sample.cu) and
// ppx_policy_act_record (collect.cu): both kernels draw from the same Philox stream with the same arithmetic, so a
// seed / draw number gives the same actions and log-probabilities whichever of the two ran.
#pragma once
#include <stdint.h>

#include "philox.cuh"

namespace ppx {

constexpr float kProbEps = 1.1920928955078125e-07f;      // torch.finfo(float32).eps (clamp_probs)
constexpr float kHalfLog2Pi = 0.91893853320467274178f;   // log(sqrt(2*pi))

// Box: the two N(0,1) of the element pair that starts at the even flat index i = n*A + a, counter (i, draw)
__device__ __forceinline__ void box_pair_normals(int64_t i, uint64_t seed, uint64_t draw, float (&z)[2]) {
  uint32_t c[4] = {(uint32_t)i, (uint32_t)(i >> 32), (uint32_t)draw, (uint32_t)(draw >> 32)};
  philox4x32(c, seed);
  box_muller(c[0], c[1], z[0], z[1]);
}

// Box: Normal(tanh(*pre), exp(*ls)) -- the sample for the standard normal z and its log-probability
__device__ __forceinline__ void box_sample(const float* pre, const float* ls, float z, float& act, float& logp) {
  const float mu = tanhf(*pre);
  const float sigma = expf(*ls);
  act = mu + sigma * z;                                           // Normal.sample: mean + std * eps
  const float d = act - mu;
  logp = -(d * d) / (2.f * sigma * sigma) - logf(sigma) - kHalfLog2Pi;   // Normal.log_prob
}

// Discrete: Categorical(probs=softmax(l[0..A))) -- probabilities renormalised as torch.distributions does, inverse-CDF
// draw for env n (counter (n, draw)); returns the action id and its clamped log-probability in `logp`
__device__ __forceinline__ int discrete_sample(const float* l, int A, int64_t n, uint64_t seed, uint64_t draw, float& logp) {
  float mx = l[0];
  for (int j = 1; j < A; ++j) mx = fmaxf(mx, l[j]);
  float se = 0.f;
  for (int j = 0; j < A; ++j) se += expf(l[j] - mx);
  float sq = 0.f;                                                 // Categorical(probs=softmax): probs / probs.sum()
  for (int j = 0; j < A; ++j) sq += expf(l[j] - mx) / se;
  uint32_t c[4] = {(uint32_t)n, (uint32_t)(n >> 32), (uint32_t)draw, (uint32_t)(draw >> 32)};
  philox4x32(c, seed);
  const float u = (float)c[0] * 2.3283064365386963e-10f;           // [0,1)
  float acc = 0.f;
  int pick = A - 1;
  for (int j = 0; j < A; ++j) {
    acc += (expf(l[j] - mx) / se) / sq;
    if (u < acc) { pick = j; break; }
  }
  const float q = (expf(l[pick] - mx) / se) / sq;
  logp = logf(fminf(fmaxf(q, kProbEps), 1.f - kProbEps));
  return pick;
}

}  // namespace ppx
