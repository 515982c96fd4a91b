// ES episode evaluation on an environment that lives on the GPU (EvolutionStrategy.evaluate, INTEGRATION.md §4): env i runs
// population member i for one episode, and a step is two launches around the user's env.step, with no host round trip.
//   ppx_es_act           the population forward of the members still running (evaluate / get_action, evolution_strategies.py
//                        :75-95, 153-170): f32 observations read straight from the env, weights theta + sigma*eps_p formed on
//                        the fly (es_walk.cuh, the walk of ppx_es_forward: bit-identical logits), actions written into the
//                        env-facing buffer -- Box tanh(logits) f64, Discrete one categorical draw int64 with numpy's
//                        RandomState.choice arithmetic.  A finished member reads no noise and gets action 0.
//   ppx_es_act_rows      the brains of EvolutionStrategy.run: env row m acts with its own parameter vector thetas[m] at
//                        sigma = 0, through the same walk (bit-identical to ppx_es_act with theta = thetas[m]).
//   ppx_es_episode_step  after env.step: fitness += reward (f64) and length += 1 while the member runs, its behaviour row
//                        latched at its terminating step, alive &= !done, and a device count of the members still running.
#include "common.cuh"
#include "es_walk.cuh"
#include "philox.cuh"

namespace ppx {
namespace {

struct EsActP {
  const double* theta; const float* noise; const int64_t* offsets; float sigma; int P, D, n_layers;
  int sizes[kFwdMaxLayers + 1];
  int vec[kFwdMaxLayers];
  const float* obs; const uint8_t* alive; void* actions; int discrete;
  uint64_t seed; const int64_t* draw; int64_t step, member_lo; const double* uniforms;
};

__device__ __forceinline__ double exp_logit(const float* lg, int j) { return exp((double)lg[j]); }

// np.sum(np.exp(l)) in numpy's order (pairwise_sum of the add reduction: sequential below 8 elements, eight accumulators up
// to 128, halves split at a multiple of 8 above).  Widths <= kFwdMaxWidth = 256 need at most two splits.
template <int SPLITS>
__device__ __forceinline__ double np_sum_exp(const float* lg, int lo, int n) {
  if (n < 8) {
    double r = -0.0;
    for (int i = 0; i < n; ++i) r += exp_logit(lg, lo + i);
    return r;
  }
  if constexpr (SPLITS > 0) {
    if (n > 128) {
      int n2 = n / 2;
      n2 -= n2 % 8;
      return np_sum_exp<SPLITS - 1>(lg, lo, n2) + np_sum_exp<SPLITS - 1>(lg, lo + n2, n - n2);
    }
  }
  double r[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) r[j] = exp_logit(lg, lo + j);
  int i = 8;
  for (; i < n - (n % 8); i += 8) {
#pragma unroll
    for (int j = 0; j < 8; ++j) r[j] += exp_logit(lg, lo + i + j);
  }
  double res = ((r[0] + r[1]) + (r[2] + r[3])) + ((r[4] + r[5]) + (r[6] + r[7]));
  for (; i < n; ++i) res += exp_logit(lg, lo + i);
  return res;
}

// discrete_action (:81-82) as numpy computes it: p = exp(l) / sum(exp(l)) in f64, cdf = cumsum(p), cdf /= cdf[-1],
// index = searchsorted(cdf, u, side="right") = the number of cdf entries <= u
__device__ __forceinline__ int np_choice(const float* lg, int A, double u) {
  const double s = np_sum_exp<2>(lg, 0, A);
  double c = 0.0;
  for (int j = 0; j < A; ++j) c += exp_logit(lg, j) / s;
  const double last = c;
  int idx = 0;
  c = 0.0;
  for (int j = 0; j < A; ++j) {
    c += exp_logit(lg, j) / s;
    idx += (c / last) <= u;
  }
  return idx;
}

__global__ void __launch_bounds__(256) es_act_kernel(EsActP p) {
  extern __shared__ float sm_f[];
  float* th = sm_f;                                         // [D]
  float* act = th + ((p.D + 3) & ~3);                       // [8 warps][3][kFwdMaxWidth]: two activation buffers + the logits
  for (int i = threadIdx.x; i < p.D; i += blockDim.x) th[i] = (float)__ldg(p.theta + i);
  __syncthreads();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  float* a0 = act + (size_t)warp * 3 * kFwdMaxWidth;
  float* a1 = a0 + kFwdMaxWidth;
  float* lg = a1 + kFwdMaxWidth;
  const int A = p.sizes[p.n_layers];
  for (int m = blockIdx.x * 8 + warp; m < p.P; m += gridDim.x * 8) {
    if (p.alive && !p.alive[m]) {                           // finished: action 0, no noise and no observation read
      if (p.discrete) {
        if (lane == 0) static_cast<int64_t*>(p.actions)[m] = 0;
      } else {
        for (int j = lane; j < A; j += 32) static_cast<double*>(p.actions)[(size_t)m * A + j] = 0.0;
      }
      continue;
    }
    const float* eps = p.noise + (p.offsets ? __ldg(p.offsets + m) : (int64_t)m * p.D);
    for (int i = lane; i < p.sizes[0]; i += 32) a0[i] = __ldg(p.obs + (size_t)m * p.sizes[0] + i);
    __syncwarp();
    es_member_walk(p, eps, th, a0, a1, lane, [&](int j, int no, float v) {
      if (p.discrete) lg[j] = v;
      else static_cast<double*>(p.actions)[(size_t)m * no + j] = (double)tanhf(v);
    });
    if (p.discrete) {                                       // the walk ended in __syncwarp: the logits are in lg
      if (lane == 0) {
        double u;
        if (p.uniforms) {
          u = p.uniforms[m];
        } else {                                            // 53-bit uniform in [0, 1), as numpy's random_sample forms it
          const uint64_t gen = p.draw ? (uint64_t)*p.draw : 0;
          const uint64_t member = (uint64_t)(p.member_lo + m);
          uint32_t c[4] = {(uint32_t)member, (uint32_t)p.step, (uint32_t)gen, (uint32_t)(gen >> 32)};
          philox4x32(c, p.seed);
          u = ((double)(c[0] >> 5) * 67108864.0 + (double)(c[1] >> 6)) * (1.0 / 9007199254740992.0);
        }
        static_cast<int64_t*>(p.actions)[m] = np_choice(lg, A, u);
      }
      __syncwarp();
    }
  }
}

// The brains of EvolutionStrategy.run (§3.15): CTA m stages thetas[m] and its warp 0 runs env row m with it at sigma = 0 --
// the member walk of es_act_kernel on table offset 0 (fmaf(0, eps, t) = t), so a row's logits and action are bit for bit
// those of es_act_kernel for theta = thetas[m], sigma = 0 and the same Philox key.  M is a handful of rows: one CTA each.
__global__ void __launch_bounds__(128) es_act_rows_kernel(EsActP p) {
  extern __shared__ float sm_f[];
  const int m = blockIdx.x;
  const int A = p.sizes[p.n_layers];
  if (p.alive && !p.alive[m]) {
    if (p.discrete) {
      if (threadIdx.x == 0) static_cast<int64_t*>(p.actions)[m] = 0;
    } else {
      for (int j = threadIdx.x; j < A; j += blockDim.x) static_cast<double*>(p.actions)[(size_t)m * A + j] = 0.0;
    }
    return;
  }
  float* th = sm_f;                                         // [D]
  float* a0 = th + ((p.D + 3) & ~3);                        // [3][kFwdMaxWidth]: two activation buffers + the logits
  float* a1 = a0 + kFwdMaxWidth;
  float* lg = a1 + kFwdMaxWidth;
  const double* theta = p.theta + (size_t)m * p.D;
  for (int i = threadIdx.x; i < p.D; i += blockDim.x) th[i] = (float)__ldg(theta + i);
  __syncthreads();
  if (threadIdx.x >= 32) return;
  const int lane = threadIdx.x;
  for (int i = lane; i < p.sizes[0]; i += 32) a0[i] = __ldg(p.obs + (size_t)m * p.sizes[0] + i);
  __syncwarp();
  es_member_walk(p, p.noise, th, a0, a1, lane, [&](int j, int no, float v) {
    if (p.discrete) lg[j] = v;
    else static_cast<double*>(p.actions)[(size_t)m * no + j] = (double)tanhf(v);
  });
  if (p.discrete && lane == 0) {
    const uint64_t gen = p.draw ? (uint64_t)*p.draw : 0;
    uint32_t c[4] = {(uint32_t)m, (uint32_t)p.step, (uint32_t)gen, (uint32_t)(gen >> 32)};
    philox4x32(c, p.seed);
    const double u = ((double)(c[0] >> 5) * 67108864.0 + (double)(c[1] >> 6)) * (1.0 / 9007199254740992.0);
    static_cast<int64_t*>(p.actions)[m] = np_choice(lg, A, u);
  }
}

// state[0]: running sum of the blocks' counts, state[1]: ticket word of the last-block detection, state[2]: members still
// running after this step (written by the last block, which re-arms state[0] and the ticket)
__global__ void __launch_bounds__(256)
es_episode_step_kernel(const void* __restrict__ rewards, int rewards_f64, const uint8_t* __restrict__ dones,
                       const double* __restrict__ behavior, int k, int64_t N, int last_step, uint8_t* __restrict__ alive,
                       double* __restrict__ fitness, int64_t* __restrict__ lengths, double* __restrict__ behavior_out,
                       unsigned long long* state) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  unsigned int running = 0;
  for (int64_t n = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; n < N; n += stride) {
    if (!alive[n]) continue;
    const double r = rewards_f64 ? static_cast<const double*>(rewards)[n] : (double)static_cast<const float*>(rewards)[n];
    fitness[n] += r;
    lengths[n] += 1;
    const bool end = dones[n] != 0 || last_step;
    if (end) {
      if (behavior)
        for (int c = 0; c < k; ++c) behavior_out[n * k + c] = behavior[n * k + c];
      alive[n] = 0;
    } else {
      ++running;
    }
  }
  running = __reduce_add_sync(0xffffffffu, running);           // one atomic per warp
  if ((threadIdx.x & 31) == 0 && running) atomicAdd(state, (unsigned long long)running);
  if (last_block_done(reinterpret_cast<unsigned int*>(state + 1)) && threadIdx.x == 0) state[2] = atomicExch(state, 0ull);
}

}  // namespace
}  // namespace ppx

using namespace ppx;

extern "C" int ppx_es_act(const double* theta, const float* noise, const int64_t* offsets, double sigma, int N, const int* layer_sizes,
                          int n_layers, const float* obs, const uint8_t* alive, int discrete, uint64_t seed, const int64_t* draw_dev,
                          int64_t step, int64_t member_lo, const double* uniforms, void* actions, void* stream) {
  PPX_REQUIRE(theta && noise && layer_sizes && obs && actions && N >= 1 && step >= 0 && member_lo >= 0, "es_act: bad arguments");
  EsActP p{};
  p.theta = theta; p.noise = noise; p.offsets = offsets; p.sigma = (float)sigma; p.P = N;
  p.obs = obs; p.alive = alive; p.actions = actions; p.discrete = discrete;
  p.seed = seed; p.draw = draw_dev; p.step = step; p.member_lo = member_lo; p.uniforms = uniforms;
  int rc = es_plan(p, noise, offsets, layer_sizes, n_layers, "es_act");
  if (rc) return rc;
  const size_t smem = sizeof(float) * ((size_t)((p.D + 3) & ~3) + 8 * 3 * kFwdMaxWidth);
  PPX_REQUIRE(smem <= 227 * 1024, "es_act: %d parameters do not fit in shared memory", p.D);
  static size_t configured = 0;
  if (smem > configured) {
    PPX_CUDA(cudaFuncSetAttribute(es_act_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    configured = smem;
  }
  // persistent grid with a whole number of members per warp, as ppx_es_forward's
  static int per_sm = 0;
  if (!per_sm) {
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, es_act_kernel, 256, smem) != cudaSuccess || per_sm < 1) per_sm = 1;
  }
  const int64_t resident = (int64_t)sm_count() * per_sm;
  const int64_t k = std::max<int64_t>(1, ceil_div(N, 8 * resident));
  const unsigned grid = (unsigned)ceil_div(N, 8 * k);
  es_act_kernel<<<grid, 256, smem, (cudaStream_t)stream>>>(p);
  return after_launch("es_act");
}

extern "C" int ppx_es_act_rows(const double* thetas, const float* noise, int M, const int* layer_sizes, int n_layers, const float* obs,
                               const uint8_t* alive, int discrete, uint64_t seed, const int64_t* draw_dev, int64_t step, void* actions,
                               void* stream) {
  PPX_REQUIRE(thetas && noise && layer_sizes && obs && actions && M >= 1 && step >= 0, "es_act_rows: bad arguments");
  EsActP p{};
  p.theta = thetas; p.noise = noise; p.sigma = 0.f; p.P = M;
  p.obs = obs; p.alive = alive; p.actions = actions; p.discrete = discrete;
  p.seed = seed; p.draw = draw_dev; p.step = step;
  static const int64_t table_offset = 0;                    // every row reads the table at offset 0: the layer plan of a table member
  int rc = es_plan(p, noise, &table_offset, layer_sizes, n_layers, "es_act_rows");
  if (rc) return rc;
  const size_t smem = sizeof(float) * ((size_t)((p.D + 3) & ~3) + 3 * kFwdMaxWidth);
  PPX_REQUIRE(smem <= 227 * 1024, "es_act_rows: %d parameters do not fit in shared memory", p.D);
  static size_t configured = 0;
  if (smem > configured) {
    PPX_CUDA(cudaFuncSetAttribute(es_act_rows_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    configured = smem;
  }
  es_act_rows_kernel<<<M, 128, smem, (cudaStream_t)stream>>>(p);
  return after_launch("es_act_rows");
}

extern "C" int ppx_es_episode_step(const void* rewards, int rewards_f64, const uint8_t* dones, const double* behavior, int k, int64_t N,
                                   int last_step, uint8_t* alive, double* fitness, int64_t* lengths, double* behavior_out,
                                   int64_t* state, void* stream) {
  PPX_REQUIRE(rewards && dones && alive && fitness && lengths && state && N >= 1 && (!behavior || (k >= 1 && behavior_out)),
              "es_episode_step: bad arguments");
  const unsigned grid = (unsigned)std::max<int64_t>(1, std::min<int64_t>(ceil_div(N, 256), (int64_t)sm_count() * 8));
  es_episode_step_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(rewards, rewards_f64, dones, behavior, k, N, last_step, alive, fitness,
                                                                 lengths, behavior_out, reinterpret_cast<unsigned long long*>(state));
  return after_launch("es_episode_step");
}
