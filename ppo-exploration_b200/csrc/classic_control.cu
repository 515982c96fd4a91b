// Gym 0.17 classic-control environments stepped on the GPU, and the device-side episode statistics (DESIGN.md §3.13).
//   ppx_classic_step          one launch per env step, one thread per env: action -> f64 dynamics -> termination and time
//                             limit -> observation / reward / done (+ the pre-reset state for ES behaviours) -> episode
//                             monitor -> in-place auto-reset of the finished envs
//   ppx_classic_reset         a new episode in every env
//   ppx_episode_monitor_step  the same monitor for any env on the GPU (returns / lengths of the episodes that just ended)
//   ppx_episode_log_record    learner side, per step: the finished envs' monitor values into row t of a [T, N] log
//   ppx_episode_log_tail      learner side, per rollout: the last K finished episodes of the log, newest first
// This file is compiled with -fmad=false (Makefile): every + - * / of the dynamics rounds once, as numpy's does, so the
// only differences from the numpy restatement (oracle/classic_control.py) are CUDA's sin / cos.  fmod is exact in both.
#include "common.cuh"
#include "philox.cuh"

namespace ppx {
namespace {

enum Kind { CARTPOLE = 0, MOUNTAIN_CAR = 1, MOUNTAIN_CAR_CONT = 2, PENDULUM = 3 };

template <int K> struct Spec;
template <> struct Spec<CARTPOLE> { static constexpr int S = 4, D = 4, LIMIT = 500, DRAWS = 4; };
template <> struct Spec<MOUNTAIN_CAR> { static constexpr int S = 2, D = 2, LIMIT = 200, DRAWS = 1; };
template <> struct Spec<MOUNTAIN_CAR_CONT> { static constexpr int S = 2, D = 2, LIMIT = 999, DRAWS = 1; };
template <> struct Spec<PENDULUM> { static constexpr int S = 2, D = 3, LIMIT = 200, DRAWS = 2; };

constexpr double kPi = 3.141592653589793;

// numpy's random_double: 53 random bits -> [0, 1)
__device__ __forceinline__ double u53(uint32_t a, uint32_t b) {
  return ((double)(a >> 5) * 67108864.0 + (double)(b >> 6)) * (1.0 / 9007199254740992.0);
}

// Reset draws of (global env g, episode e): Philox4x32-10 under `seed` at counter (g lo, g hi, e, block).  They depend on
// neither the number of envs nor the rank, so rank r's slice of a W*N env equals an env of N at offset r*N.
template <int K>
__device__ __forceinline__ void reset_state(double (&s)[Spec<K>::S], uint64_t seed, int64_t g, int64_t e) {
  double u[4];
#pragma unroll
  for (int blk = 0; blk < (Spec<K>::DRAWS + 1) / 2; ++blk) {
    uint32_t c[4] = {(uint32_t)g, (uint32_t)((uint64_t)g >> 32), (uint32_t)e, (uint32_t)blk};
    philox4x32(c, seed);
    u[2 * blk] = u53(c[0], c[1]);
    u[2 * blk + 1] = u53(c[2], c[3]);
  }
  // np_random.uniform(low, high) = low + (high - low) * u
  if constexpr (K == CARTPOLE) {
#pragma unroll
    for (int k = 0; k < 4; ++k) s[k] = -0.05 + (0.05 - -0.05) * u[k];
  } else if constexpr (K == PENDULUM) {
    s[0] = -kPi + (kPi - -kPi) * u[0];
    s[1] = -1.0 + (1.0 - -1.0) * u[1];
  } else {
    s[0] = -0.6 + (-0.4 - -0.6) * u[0];
    s[1] = 0.0;
  }
}

__device__ __forceinline__ double clip(double x, double lo, double hi) { return fmin(fmax(x, lo), hi); }

// One step of gym 0.17's dynamics in its own evaluation order.  Returns the f64 reward; sets `term`.
template <int K>
__device__ __forceinline__ double dynamics(double (&s)[Spec<K>::S], const void* actions, int64_t n, bool& term) {
  if constexpr (K == CARTPOLE) {
    const double gravity = 9.8, masscart = 1.0, masspole = 0.1, total_mass = masspole + masscart, length = 0.5;
    const double polemass_length = masspole * length, force_mag = 10.0, tau = 0.02;
    const double theta_threshold = 12 * 2 * kPi / 360, x_threshold = 2.4;
    const int64_t a = static_cast<const int64_t*>(actions)[n];
    const double x = s[0], x_dot = s[1], theta = s[2], theta_dot = s[3];
    const double force = a == 1 ? force_mag : -force_mag;
    const double costheta = cos(theta), sintheta = sin(theta);
    const double temp = (force + polemass_length * (theta_dot * theta_dot) * sintheta) / total_mass;
    const double thetaacc = (gravity * sintheta - costheta * temp) /
                            (length * (4.0 / 3.0 - masspole * (costheta * costheta) / total_mass));
    const double xacc = temp - polemass_length * thetaacc * costheta / total_mass;
    s[0] = x + tau * x_dot;
    s[1] = x_dot + tau * xacc;
    s[2] = theta + tau * theta_dot;
    s[3] = theta_dot + tau * thetaacc;
    term = s[0] < -x_threshold || s[0] > x_threshold || s[2] < -theta_threshold || s[2] > theta_threshold;
    return 1.0;
  } else if constexpr (K == MOUNTAIN_CAR) {
    const int64_t a = static_cast<const int64_t*>(actions)[n];
    double p = s[0], v = s[1];
    v = v + ((double)(a - 1) * 0.001 + cos(3 * p) * (-0.0025));
    v = clip(v, -0.07, 0.07);
    p = p + v;
    p = clip(p, -1.2, 0.6);
    if (p == -1.2 && v < 0) v = 0.0;
    term = p >= 0.5 && v >= 0.0;
    s[0] = p; s[1] = v;
    return -1.0;
  } else if constexpr (K == MOUNTAIN_CAR_CONT) {
    const double a = static_cast<const double*>(actions)[n];
    double p = s[0], v = s[1];
    const double force = fmin(fmax(a, -1.0), 1.0);
    v = v + (force * 0.0015 - 0.0025 * cos(3 * p));
    if (v > 0.07) v = 0.07;
    if (v < -0.07) v = -0.07;
    p = p + v;
    if (p > 0.6) p = 0.6;
    if (p < -1.2) p = -1.2;
    if (p == -1.2 && v < 0) v = 0.0;
    term = p >= 0.45 && v >= 0.0;
    s[0] = p; s[1] = v;
    return (term ? 100.0 : 0.0) - a * a * 0.1;                   // the unclipped action, as gym
  } else {
    const double a = static_cast<const double*>(actions)[n];
    const double th = s[0], thdot = s[1];
    const double u = clip(a, -2.0, 2.0);
    double an = fmod(th + kPi, 2 * kPi);                            // numpy's floor-mod: the sign of the divisor
    if (an != 0.0) { if (an < 0.0) an = an + 2 * kPi; } else { an = 0.0; }
    an = an - kPi;
    const double costs = an * an + 0.1 * (thdot * thdot) + 0.001 * (u * u);
    const double newthdot = thdot + (-3 * 10.0 / (2 * 1.0) * sin(th + kPi) + 3.0 / (1.0 * 1.0) * u) * 0.05;
    s[0] = th + newthdot * 0.05;                                    // the unclipped velocity, as gym
    s[1] = clip(newthdot, -8.0, 8.0);
    term = false;
    return -costs;
  }
}

template <int K>
__device__ __forceinline__ void write_obs(const double (&s)[Spec<K>::S], float* o) {
  if constexpr (K == PENDULUM) {
    o[0] = (float)cos(s[0]); o[1] = (float)sin(s[0]); o[2] = (float)s[1];
  } else {
#pragma unroll
    for (int k = 0; k < Spec<K>::S; ++k) o[k] = (float)s[k];
  }
}

template <int K>
__global__ void __launch_bounds__(256)
classic_step_kernel(int64_t N, int64_t env_offset, uint64_t seed, const void* __restrict__ actions, double* __restrict__ state,
                    int64_t* __restrict__ elapsed, int64_t* __restrict__ episode, double* __restrict__ mon_ret,
                    int64_t* __restrict__ mon_len, double* __restrict__ ep_ret, int64_t* __restrict__ ep_len,
                    float* __restrict__ obs, void* __restrict__ reward, int reward_f64, uint8_t* __restrict__ done,
                    double* __restrict__ behavior) {
  constexpr int S = Spec<K>::S;
  const int64_t n = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= N) return;
  double s[S];
#pragma unroll
  for (int k = 0; k < S; ++k) s[k] = state[k * N + n];             // [S, N]: coalesced
  bool term;
  const double r = dynamics<K>(s, actions, n, term);
  int64_t el = elapsed[n] + 1;
  const bool d = term || el >= Spec<K>::LIMIT;                     // TimeLimit: an ordinary done (4-tuple API)
  double ret = mon_ret[n] + r;
  int64_t len = mon_len[n] + 1;
  if (behavior) {
#pragma unroll
    for (int k = 0; k < S; ++k) behavior[n * S + k] = s[k];
  }
  if (reward_f64) static_cast<double*>(reward)[n] = r;
  else static_cast<float*>(reward)[n] = __double2float_rn(r);
  if (d) {
    ep_ret[n] = ret;
    ep_len[n] = len;
    ret = 0.0;
    len = 0;
    el = 0;
    const int64_t e = episode[n] + 1;
    episode[n] = e;
    reset_state<K>(s, seed, env_offset + n, e);
  }
  mon_ret[n] = ret;
  mon_len[n] = len;
  elapsed[n] = el;
#pragma unroll
  for (int k = 0; k < S; ++k) state[k * N + n] = s[k];
  write_obs<K>(s, obs + n * Spec<K>::D);
  done[n] = d;
}

template <int K>
__global__ void __launch_bounds__(256)
classic_reset_kernel(int64_t N, int64_t env_offset, uint64_t seed, double* __restrict__ state, int64_t* __restrict__ elapsed,
                     int64_t* __restrict__ episode, double* __restrict__ mon_ret, int64_t* __restrict__ mon_len,
                     float* __restrict__ obs) {
  constexpr int S = Spec<K>::S;
  const int64_t n = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= N) return;
  const int64_t e = episode[n] + 1;
  episode[n] = e;
  double s[S];
  reset_state<K>(s, seed, env_offset + n, e);
#pragma unroll
  for (int k = 0; k < S; ++k) state[k * N + n] = s[k];
  elapsed[n] = 0;
  mon_ret[n] = 0.0;
  mon_len[n] = 0;
  write_obs<K>(s, obs + n * Spec<K>::D);
}

__global__ void __launch_bounds__(256)
episode_monitor_kernel(const void* __restrict__ rewards, int rewards_f64, const uint8_t* __restrict__ dones, int64_t N,
                       double* __restrict__ acc_ret, int64_t* __restrict__ acc_len, double* __restrict__ ep_ret,
                       int64_t* __restrict__ ep_len) {
  const int64_t n = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= N) return;
  const double r = rewards_f64 ? static_cast<const double*>(rewards)[n] : (double)static_cast<const float*>(rewards)[n];
  double ret = acc_ret[n] + r;
  int64_t len = acc_len[n] + 1;
  if (dones[n]) {
    ep_ret[n] = ret;
    ep_len[n] = len;
    ret = 0.0;
    len = 0;
  }
  acc_ret[n] = ret;
  acc_len[n] = len;
}

__global__ void __launch_bounds__(256)
episode_log_record_kernel(const uint8_t* __restrict__ dones, const double* __restrict__ ep_ret, const int64_t* __restrict__ ep_len,
                          int64_t N, double* __restrict__ log_ret, int64_t* __restrict__ log_len) {
  const int64_t n = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (n < N && dones[n]) {
    log_ret[n] = ep_ret[n];
    log_len[n] = ep_len[n];
  }
}

constexpr int kTailThreads = 1024, kTailPer = 16;

// One block walks the flat [T*N] done flags backwards in chunks of 16K; each thread owns 16 consecutive flags.  A block
// scan gives every thread the number of dones after its range, so the reverse rank of each done is known and the newest
// K are written to out[rank].  Stops after the chunk in which the K-th newest was found.
__global__ void __launch_bounds__(kTailThreads)
episode_log_tail_kernel(const uint8_t* __restrict__ dones, const double* __restrict__ log_ret, const int64_t* __restrict__ log_len,
                        int64_t total, int64_t K, double* __restrict__ out_ret, int64_t* __restrict__ out_len,
                        int64_t* __restrict__ out_count) {
  __shared__ int warp_sums[kTailThreads / 32];
  const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
  constexpr int nw = kTailThreads / 32;
  constexpr int64_t chunk = (int64_t)kTailThreads * kTailPer;
  int64_t found = 0;
  for (int64_t end = total; end > 0 && found < K; end -= chunk) {
    const int64_t base = end - chunk + (int64_t)tid * kTailPer;
    uint32_t bits = 0;
#pragma unroll
    for (int j = 0; j < kTailPer; ++j) {
      const int64_t i = base + j;
      if (i >= 0 && i < end && dones[i]) bits |= 1u << j;
    }
    int x = __popc(bits);
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int y = __shfl_up_sync(0xffffffffu, x, o);
      if (lane >= o) x += y;
    }
    if (lane == 31) warp_sums[w] = x;
    __syncthreads();
    if (w == 0) {
      int v = warp_sums[lane];
#pragma unroll
      for (int o = 1; o < nw; o <<= 1) {
        const int y = __shfl_up_sync(0xffffffffu, v, o);
        if (lane >= o) v += y;
      }
      warp_sums[lane] = v;
    }
    __syncthreads();
    const int incl = x + (w > 0 ? warp_sums[w - 1] : 0);
    const int chunk_total = warp_sums[nw - 1];
    int64_t rank = found + (chunk_total - incl);                    // dones after this thread's range
    for (int j = kTailPer - 1; j >= 0 && rank < K; --j) {
      if (bits >> j & 1u) {
        out_ret[rank] = log_ret[base + j];
        out_len[rank] = log_len[base + j];
        ++rank;
      }
    }
    found += chunk_total;
    __syncthreads();                                              // warp_sums is rewritten by the next chunk
  }
  if (tid == 0) *out_count = found < K ? found : K;
}

unsigned blocks_for(int64_t N) { return (unsigned)ceil_div(N, 256); }

template <int K>
void launch_step(int64_t N, int64_t off, uint64_t seed, const void* actions, double* state, int64_t* elapsed, int64_t* episode,
                 double* mon_ret, int64_t* mon_len, double* ep_ret, int64_t* ep_len, float* obs, void* reward, int reward_f64,
                 uint8_t* done, double* behavior, cudaStream_t st) {
  classic_step_kernel<K><<<blocks_for(N), 256, 0, st>>>(N, off, seed, actions, state, elapsed, episode, mon_ret, mon_len, ep_ret,
                                                        ep_len, obs, reward, reward_f64, done, behavior);
}

template <int K>
void launch_reset(int64_t N, int64_t off, uint64_t seed, double* state, int64_t* elapsed, int64_t* episode, double* mon_ret,
                  int64_t* mon_len, float* obs, cudaStream_t st) {
  classic_reset_kernel<K><<<blocks_for(N), 256, 0, st>>>(N, off, seed, state, elapsed, episode, mon_ret, mon_len, obs);
}

}  // namespace
}  // namespace ppx

using namespace ppx;

extern "C" int ppx_classic_step(int env, int64_t N, int64_t env_offset, uint64_t seed, const void* actions, double* state,
                                int64_t* elapsed, int64_t* episode, double* mon_ret, int64_t* mon_len, double* ep_ret,
                                int64_t* ep_len, float* obs, void* reward, int reward_f64, uint8_t* done, double* behavior,
                                void* stream) {
  PPX_REQUIRE(env >= 0 && env <= 3 && N >= 0 && env_offset >= 0 && actions && state && elapsed && episode && mon_ret && mon_len &&
              ep_ret && ep_len && obs && reward && done, "classic_step: bad arguments");
  if (N == 0) return PPX_OK;
  cudaStream_t st = (cudaStream_t)stream;
#define PPX_STEP(KIND) launch_step<KIND>(N, env_offset, seed, actions, state, elapsed, episode, mon_ret, mon_len, ep_ret, ep_len, \
                                         obs, reward, reward_f64, done, behavior, st)
  switch (env) {
    case CARTPOLE: PPX_STEP(CARTPOLE); break;
    case MOUNTAIN_CAR: PPX_STEP(MOUNTAIN_CAR); break;
    case MOUNTAIN_CAR_CONT: PPX_STEP(MOUNTAIN_CAR_CONT); break;
    default: PPX_STEP(PENDULUM); break;
  }
#undef PPX_STEP
  return after_launch("classic_step");
}

extern "C" int ppx_classic_reset(int env, int64_t N, int64_t env_offset, uint64_t seed, double* state, int64_t* elapsed,
                                 int64_t* episode, double* mon_ret, int64_t* mon_len, float* obs, void* stream) {
  PPX_REQUIRE(env >= 0 && env <= 3 && N >= 0 && env_offset >= 0 && state && elapsed && episode && mon_ret && mon_len && obs,
              "classic_reset: bad arguments");
  if (N == 0) return PPX_OK;
  cudaStream_t st = (cudaStream_t)stream;
  switch (env) {
    case CARTPOLE: launch_reset<CARTPOLE>(N, env_offset, seed, state, elapsed, episode, mon_ret, mon_len, obs, st); break;
    case MOUNTAIN_CAR: launch_reset<MOUNTAIN_CAR>(N, env_offset, seed, state, elapsed, episode, mon_ret, mon_len, obs, st); break;
    case MOUNTAIN_CAR_CONT:
      launch_reset<MOUNTAIN_CAR_CONT>(N, env_offset, seed, state, elapsed, episode, mon_ret, mon_len, obs, st);
      break;
    default: launch_reset<PENDULUM>(N, env_offset, seed, state, elapsed, episode, mon_ret, mon_len, obs, st); break;
  }
  return after_launch("classic_reset");
}

extern "C" int ppx_episode_monitor_step(const void* rewards, int rewards_f64, const uint8_t* dones, int64_t N, double* acc_ret,
                                        int64_t* acc_len, double* ep_ret, int64_t* ep_len, void* stream) {
  PPX_REQUIRE(rewards && dones && acc_ret && acc_len && ep_ret && ep_len && N >= 0, "episode_monitor_step: bad arguments");
  if (N == 0) return PPX_OK;
  episode_monitor_kernel<<<blocks_for(N), 256, 0, (cudaStream_t)stream>>>(rewards, rewards_f64, dones, N, acc_ret, acc_len, ep_ret,
                                                                          ep_len);
  return after_launch("episode_monitor_step");
}

extern "C" int ppx_episode_log_record(const uint8_t* dones, const double* ep_ret, const int64_t* ep_len, int64_t N,
                                      double* log_ret_row, int64_t* log_len_row, void* stream) {
  PPX_REQUIRE(dones && ep_ret && ep_len && log_ret_row && log_len_row && N >= 0, "episode_log_record: bad arguments");
  if (N == 0) return PPX_OK;
  episode_log_record_kernel<<<blocks_for(N), 256, 0, (cudaStream_t)stream>>>(dones, ep_ret, ep_len, N, log_ret_row, log_len_row);
  return after_launch("episode_log_record");
}

extern "C" int ppx_episode_log_tail(const uint8_t* dones, const double* log_ret, const int64_t* log_len, int64_t total, int64_t K,
                                    double* out_ret, int64_t* out_len, int64_t* out_count, void* stream) {
  PPX_REQUIRE(dones && log_ret && log_len && out_ret && out_len && out_count && total >= 0 && K >= 1,
              "episode_log_tail: bad arguments");
  episode_log_tail_kernel<<<1, kTailThreads, 0, (cudaStream_t)stream>>>(dones, log_ret, log_len, total, K, out_ret, out_len,
                                                                         out_count);
  return after_launch("episode_log_tail");
}
