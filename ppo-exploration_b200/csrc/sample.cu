// Rollout-side action sampling on the device (SURVEY §8f.1): the tail of Policy.act (models.py:30-50 / 75-99) --
// build the action distribution from the actor output, draw one action per env, evaluate its log-probability -- in
// ONE launch instead of the ~10 torch.distributions kernels, writing the f64 actions / f32 log-probs in the layout the
// rollout buffer stores (buffer.py:154, :159).
//   Box       Normal(tanh(actor_out), exp(log_std)), per-dimension sample and log_prob (models.py:160-170)
//   Discrete  Categorical(softmax(logits)) (models.py:62): probabilities renormalised and clamped to [eps, 1-eps] exactly
//             as torch.distributions does (and as ppo_loss.cu evaluates them in train()), inverse-CDF draw
// Randomness: Philox4x32-10 keyed by `seed`, counter = (env, draw number) -- a counter-based stream of ppx's own
// (torch's generator state is not reproducible from a kernel); the log-probability of the drawn action is exact.
#include "common.cuh"
#include "sample_math.cuh"

namespace ppx {
namespace {

__global__ void __launch_bounds__(256)
sample_box_kernel(const float* __restrict__ actor_out, const float* __restrict__ log_std, int64_t N, int A, uint64_t seed, uint64_t draw,
                  double* __restrict__ actions, float* __restrict__ logp) {
  const int64_t total = N * A;
  for (int64_t i = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) * 2; i < total; i += (int64_t)gridDim.x * blockDim.x * 2) {
    float z[2];
    box_pair_normals(i, seed, draw, z);
#pragma unroll
    for (int e = 0; e < 2; ++e) {
      if (i + e >= total) break;
      const int a = (int)((i + e) % A);
      float act, lp;
      box_sample(actor_out + i + e, log_std + a, z[e], act, lp);
      actions[i + e] = (double)act;
      logp[i + e] = lp;
    }
  }
}

__global__ void __launch_bounds__(256)
sample_discrete_kernel(const float* __restrict__ logits, int64_t N, int A, uint64_t seed, uint64_t draw, double* __restrict__ actions,
                       float* __restrict__ logp) {
  for (int64_t n = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; n < N; n += (int64_t)gridDim.x * blockDim.x) {
    float lp;
    const int pick = discrete_sample(logits + n * A, A, n, seed, draw, lp);
    actions[n] = (double)pick;
    logp[n] = lp;
  }
}

}  // namespace
}  // namespace ppx

using namespace ppx;

extern "C" int ppx_policy_sample(const float* actor_out, const float* log_std, int64_t N, int A, int discrete, uint64_t seed,
                                 uint64_t draw, double* actions_out, float* logp_out, void* stream) {
  PPX_REQUIRE(actor_out && actions_out && logp_out && N >= 0 && A >= 1 && (discrete || log_std), "policy_sample: bad arguments");
  if (N == 0) return PPX_OK;
  cudaStream_t st = (cudaStream_t)stream;
  if (discrete) {
    const unsigned grid = (unsigned)std::min<int64_t>(ceil_div(N, 256), (int64_t)sm_count() * 8);
    sample_discrete_kernel<<<grid, 256, 0, st>>>(actor_out, N, A, seed, draw, actions_out, logp_out);
  } else {
    const unsigned grid = (unsigned)std::min<int64_t>(ceil_div(ceil_div(N * A, 2), 256), (int64_t)sm_count() * 8);
    sample_box_kernel<<<grid, 256, 0, st>>>(actor_out, log_std, N, A, seed, draw, actions_out, logp_out);
  }
  return after_launch("policy_sample");
}
