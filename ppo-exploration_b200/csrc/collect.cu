// Rollout collection from an environment that lives on the GPU (collect_samples' device path, INTEGRATION.md §4): the
// rollout row of one env step is written by two launches around the user's env.step, with no host round trip.
//   ppx_policy_act_record    after the policy forward: the tail of Policy.act (models.py:30-50 / 75-99) plus the rows of
//                            RolloutStorage.add that are known before the step -- observation, f64 action, log-prob,
//                            value(s) at rollout step `pos` -- and a separate env-facing copy of the actions
//   ppx_rollout_record_step  after env.step: rewards, masks (dones) and RND's intrinsic rewards at `pos`
//                            (buffer.py:165-186, :305-318), plus a device episode counter
// The sampling math is sample_math.cuh, shared with ppx_policy_sample: the same seed / draw number gives the same actions.
#include "common.cuh"
#include "sample_math.cuh"

namespace ppx {
namespace {

__global__ void __launch_bounds__(256)
act_record_kernel(const float* __restrict__ actor_out, const float* __restrict__ value, const float* __restrict__ int_value,
                  const float* __restrict__ log_std, const float* __restrict__ obs, int64_t N, int A, int D, int discrete,
                  int vec4, uint64_t seed, uint64_t draw, float* __restrict__ obs_row, double* __restrict__ act_row,
                  float* __restrict__ logp_row, float* __restrict__ value_row, float* __restrict__ int_value_row,
                  void* __restrict__ env_actions) {
  const int64_t tid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  if (vec4) {                                                     // D % 4 == 0, both rows 16-byte aligned
    const int64_t n4 = N * D / 4;
    for (int64_t i = tid; i < n4; i += stride)
      reinterpret_cast<float4*>(obs_row)[i] = ld_stream4(reinterpret_cast<const float4*>(obs) + i);
  } else {
    for (int64_t i = tid; i < N * D; i += stride) obs_row[i] = ld_stream(obs + i);
  }
  for (int64_t n = tid; n < N; n += stride) {
    value_row[n] = value[n];
    if (int_value_row) int_value_row[n] = int_value[n];
  }
  if (discrete) {
    int64_t* env_ids = static_cast<int64_t*>(env_actions);
    for (int64_t n = tid; n < N; n += stride) {
      float lp;
      const int pick = discrete_sample(actor_out + n * A, A, n, seed, draw, lp);
      act_row[n] = (double)pick;
      logp_row[n] = lp;
      env_ids[n] = pick;
    }
  } else {
    double* env_act = static_cast<double*>(env_actions);
    const int64_t total = N * A;
    for (int64_t i = tid * 2; i < total; i += stride * 2) {
      float z[2];
      box_pair_normals(i, seed, draw, z);
#pragma unroll
      for (int e = 0; e < 2; ++e) {
        if (i + e >= total) break;
        const int a = (int)((i + e) % A);
        float act, lp;
        box_sample(actor_out + i + e, log_std + a, z[e], act, lp);
        act_row[i + e] = (double)act;
        env_act[i + e] = (double)act;
        logp_row[i + e] = lp;
      }
    }
  }
}

__global__ void __launch_bounds__(256)
record_step_kernel(const void* __restrict__ rewards, int rewards_f64, const uint8_t* __restrict__ dones,
                   const float* __restrict__ int_rewards, int64_t N, float* __restrict__ rew_row, double* __restrict__ rew_f64_row,
                   uint8_t* __restrict__ mask_row, float* __restrict__ int_rew_row, unsigned long long* __restrict__ episodes) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  unsigned int ended = 0;
  for (int64_t n = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; n < N; n += stride) {
    if (rewards_f64) {
      const double r = static_cast<const double*>(rewards)[n];
      if (rew_f64_row) rew_f64_row[n] = r;                        // SimHash adds its bonus in f64 before the one rounding
      else rew_row[n] = __double2float_rn(r);
    } else {
      rew_row[n] = static_cast<const float*>(rewards)[n];
    }
    const uint8_t d = dones[n];
    mask_row[n] = d;
    ended += d != 0;
    if (int_rew_row) int_rew_row[n] = int_rewards ? int_rewards[n] : 0.f;
  }
  ended = __reduce_add_sync(0xffffffffu, ended);                  // one atomic per warp
  if ((threadIdx.x & 31) == 0 && ended) atomicAdd(episodes, (unsigned long long)ended);
}

unsigned grid_for(int64_t work) {
  return (unsigned)std::max<int64_t>(1, std::min<int64_t>(ceil_div(work, 256), (int64_t)sm_count() * 8));
}

}  // namespace
}  // namespace ppx

using namespace ppx;

extern "C" int ppx_policy_act_record(const float* actor_out, const float* value, const float* int_value, const float* log_std,
                                     const float* obs, int64_t N, int A, int D, int discrete, uint64_t seed, uint64_t draw,
                                     float* obs_row, double* actions_row, float* logp_row, float* value_row, float* int_value_row,
                                     void* env_actions, void* stream) {
  PPX_REQUIRE(actor_out && value && obs && obs_row && actions_row && logp_row && value_row && env_actions && N >= 0 && A >= 1 &&
              D >= 1 && (discrete || log_std) && (!int_value_row || int_value), "policy_act_record: bad arguments");
  if (N == 0) return PPX_OK;
  const int vec4 = D % 4 == 0 && ((uintptr_t)obs % 16) == 0 && ((uintptr_t)obs_row % 16) == 0;
  const int64_t work = std::max<int64_t>(vec4 ? N * D / 4 : N * D, discrete ? N : ceil_div(N * A, 2));
  act_record_kernel<<<grid_for(work), 256, 0, (cudaStream_t)stream>>>(actor_out, value, int_value, log_std, obs, N, A, D, discrete,
                                                                      vec4, seed, draw, obs_row, actions_row, logp_row, value_row,
                                                                      int_value_row, env_actions);
  return after_launch("policy_act_record");
}

extern "C" int ppx_rollout_record_step(const void* rewards, int rewards_f64, const uint8_t* dones, const float* int_rewards, int64_t N,
                                       float* rewards_row, double* rewards_f64_row, uint8_t* masks_row, float* int_rewards_row,
                                       int64_t* episodes, void* stream) {
  PPX_REQUIRE(rewards && dones && masks_row && episodes && N >= 0 && (rewards_row || (rewards_f64 && rewards_f64_row)),
              "rollout_record_step: bad arguments");
  if (N == 0) return PPX_OK;
  record_step_kernel<<<grid_for(N), 256, 0, (cudaStream_t)stream>>>(rewards, rewards_f64, dones, int_rewards, N, rewards_row,
                                                                    rewards_f64 ? rewards_f64_row : nullptr, masks_row,
                                                                    int_rewards_row, (unsigned long long*)episodes);
  return after_launch("rollout_record_step");
}
