// Policy evaluation on an environment that lives on the GPU (ppx.evaluate_policy / Policy.predict, DESIGN.md §3.17): a
// step is the policy forward, one launch forming the env-facing actions, the user's env.step and one launch recording the
// finished episodes, with no host round trip.
//   ppx_policy_act_eval    the actions alone (no rollout rows, log-probs or values): deterministic -- Box tanh(mean), the
//                          sampled action at z = 0; Discrete the argmax of the logits -- or one draw with the arithmetic of
//                          ppx_policy_sample (sample_math.cuh), counter keyed by the GLOBAL row row_offset + n
//   ppx_eval_episode_step  after env.step: SB3 evaluate_policy's episode targets -- global env g keeps its first
//                          (n_eval_episodes + g) // total_envs finished episodes (return, length, end step) -- and a device
//                          count of the episodes still missing
#include "common.cuh"
#include "sample_math.cuh"

namespace ppx {
namespace {

__global__ void __launch_bounds__(256)
act_eval_kernel(const float* __restrict__ actor_out, const float* __restrict__ log_std, int64_t N, int A, int discrete,
                int deterministic, uint64_t seed, uint64_t draw, int64_t row_offset, void* __restrict__ env_actions) {
  const int64_t tid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  if (discrete) {
    int64_t* ids = static_cast<int64_t*>(env_actions);
    for (int64_t n = tid; n < N; n += stride) {
      const float* l = actor_out + n * A;
      int pick = 0;
      if (deterministic) {
        // argmax of the logits, lowest index on ties (np.argmax).  softmax is monotone, so this is the most probable
        // action, except where two different logits round to the same f32 probability: the logits decide those.
        float best = l[0];
        for (int j = 1; j < A; ++j)
          if (l[j] > best) { best = l[j]; pick = j; }
      } else {
        float lp;
        pick = discrete_sample(l, A, row_offset + n, seed, draw, lp);
      }
      ids[n] = pick;
    }
    return;
  }
  double* act = static_cast<double*>(env_actions);
  if (deterministic) {
    for (int64_t i = tid; i < N * A; i += stride) act[i] = (double)tanhf(actor_out[i]);   // box_sample's mean
    return;
  }
  // the Philox pairs are those of one launch over all rows: element pair p (even global flat index) feeds elements p, p+1
  const int64_t lo = row_offset * A, hi = lo + N * A;
  for (int64_t p = (lo & ~(int64_t)1) + tid * 2; p < hi; p += stride * 2) {
    float z[2];
    box_pair_normals(p, seed, draw, z);
#pragma unroll
    for (int e = 0; e < 2; ++e) {
      const int64_t g = p + e;
      if (g < lo || g >= hi) continue;
      const int a = (int)(g % A);
      float v, lp;
      box_sample(actor_out + (g - lo), log_std + a, z[e], v, lp);
      act[g - lo] = (double)v;
    }
  }
}

// state[0]: running sum of the blocks' counts, state[1]: ticket word of the last-block detection, state[2]: episodes still
// missing on this rank after this step (written by the last block, which re-arms state[0] and the ticket)
__global__ void __launch_bounds__(256)
eval_episode_step_kernel(const uint8_t* __restrict__ dones, const double* __restrict__ ep_returns,
                         const int64_t* __restrict__ ep_lengths, int64_t N, int64_t n_eval, int64_t env_offset, int64_t total,
                         int64_t step, int64_t* __restrict__ counts, double* __restrict__ out_ret, int64_t* __restrict__ out_len,
                         int64_t* __restrict__ out_end, int64_t kmax, unsigned long long* state) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  unsigned int missing = 0;
  for (int64_t n = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; n < N; n += stride) {
    const int64_t target = (n_eval + env_offset + n) / total;
    int64_t c = counts[n];
    if (c < target && dones[n]) {
      out_ret[n * kmax + c] = ep_returns[n];
      out_len[n * kmax + c] = ep_lengths[n];
      out_end[n * kmax + c] = step;
      counts[n] = ++c;
    }
    missing += (unsigned int)(target - c);
  }
  missing = __reduce_add_sync(0xffffffffu, missing);            // one atomic per warp
  if ((threadIdx.x & 31) == 0 && missing) atomicAdd(state, (unsigned long long)missing);
  if (last_block_done(reinterpret_cast<unsigned int*>(state + 1)) && threadIdx.x == 0) state[2] = atomicExch(state, 0ull);
}

unsigned grid_for(int64_t work) {
  return (unsigned)std::max<int64_t>(1, std::min<int64_t>(ceil_div(work, 256), (int64_t)sm_count() * 8));
}

}  // namespace
}  // namespace ppx

using namespace ppx;

extern "C" int ppx_policy_act_eval(const float* actor_out, const float* log_std, int64_t N, int A, int discrete, int deterministic,
                                   uint64_t seed, uint64_t draw, int64_t row_offset, void* env_actions, void* stream) {
  PPX_REQUIRE(actor_out && env_actions && N >= 0 && A >= 1 && row_offset >= 0 && (discrete || log_std),
              "policy_act_eval: bad arguments");
  PPX_REQUIRE(deterministic || (draw >> 63), "policy_act_eval: evaluation draw numbers have bit 63 set (got %llu)",
              (unsigned long long)draw);
  if (N == 0) return PPX_OK;
  const int64_t work = discrete ? N : (deterministic ? N * A : ceil_div(N * A, 2) + 1);
  act_eval_kernel<<<grid_for(work), 256, 0, (cudaStream_t)stream>>>(actor_out, log_std, N, A, discrete, deterministic, seed, draw,
                                                                    row_offset, env_actions);
  return after_launch("policy_act_eval");
}

extern "C" int ppx_eval_episode_step(const uint8_t* dones, const double* ep_returns, const int64_t* ep_lengths, int64_t N,
                                     int64_t n_eval_episodes, int64_t env_offset, int64_t total_envs, int64_t step, int64_t* counts,
                                     double* out_ret, int64_t* out_len, int64_t* out_end, int64_t kmax, int64_t* state,
                                     void* stream) {
  PPX_REQUIRE(dones && ep_returns && ep_lengths && counts && out_ret && out_len && out_end && state && N >= 1 &&
              n_eval_episodes >= 1 && env_offset >= 0 && total_envs >= env_offset + N && step >= 0 &&
              kmax >= ceil_div(n_eval_episodes, total_envs) && n_eval_episodes < (1ll << 31),
              "eval_episode_step: bad arguments");
  eval_episode_step_kernel<<<grid_for(N), 256, 0, (cudaStream_t)stream>>>(dones, ep_returns, ep_lengths, N, n_eval_episodes,
                                                                         env_offset, total_envs, step, counts, out_ret, out_len,
                                                                         out_end, kmax, reinterpret_cast<unsigned long long*>(state));
  return after_launch("eval_episode_step");
}
