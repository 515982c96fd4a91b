// Epilogue kernels of the RND / ICM bonus paths and the running-moment normalisers.
//
// The dense layers of the bonus nets run through linear.cu; this file holds what surrounds them:
//   RunningMeanStd.update                      util.py:20-44           -> rms_update
//   BaseAlgorithm.normalize_obs                algorithms.py:111-118   -> normalize_obs
//   RndNetwork.int_reward tail                 models.py:265           -> rnd_sqerr
//   int_rew_rms.update + divide, per env step  algorithms.py:396-398   -> rnd_normalize_rollout
//   ICM int_reward tail + reward blend         models.py:319-320, algorithms.py:630 -> icm_bonus_tail
//   ICM action_encoder (nn.Embedding)          models.py:294           -> embedding fwd/bwd
// Moments are float64 like the reference; batch mean/var are accumulated in f64 (the reference lets
// numpy accumulate float32 inputs in float32 -- same value to ~1e-7 relative).
#include "common.cuh"

namespace ppx {
namespace {

template <typename T>
__device__ __forceinline__ double ldd(const void* x, int64_t i) { return (double)((const T*)x)[i]; }

// util.py:30-44 for one scalar stream
__device__ __forceinline__ void merge_moments(double bm, double bv, double bc, double& mean, double& var, double count) {
  const double delta = bm - mean;
  const double tot = count + bc;
  const double new_mean = mean + delta * bc / tot;
  const double m2 = var * count + bv * bc + delta * delta * count * bc / (count + bc);
  mean = new_mean;
  var = m2 / (count + bc);
}

// 32 columns x 8 row phases per CTA; two passes (mean, centred second moment)
template <typename T>
__global__ void __launch_bounds__(256)
rms_cols_kernel(const T* __restrict__ x, int64_t n, int dim, double* __restrict__ mean, double* __restrict__ var,
                const double* __restrict__ count) {
  __shared__ double s[8][33];
  const int c = threadIdx.x & 31, ph = threadIdx.x >> 5;
  const int col = blockIdx.x * 32 + c;
  double a = 0.0;
  if (col < dim)
    for (int64_t r = ph; r < n; r += 8) a += (double)x[r * dim + col];
  s[ph][c] = a;
  __syncthreads();
  double bm = 0.0;
  for (int q = 0; q < 8; ++q) bm += s[q][c];
  bm /= (double)n;
  __syncthreads();
  a = 0.0;
  if (col < dim)
    for (int64_t r = ph; r < n; r += 8) {
      const double d = (double)x[r * dim + col] - bm;
      a += d * d;
    }
  s[ph][c] = a;
  __syncthreads();
  if (ph == 0 && col < dim) {
    double bv = 0.0;
    for (int q = 0; q < 8; ++q) bv += s[q][c];
    bv /= (double)n;
    double m = mean[col], v = var[col];
    merge_moments(bm, bv, (double)n, m, v, *count);
    mean[col] = m;
    var[col] = v;
  }
}

template <typename T>
__global__ void __launch_bounds__(1024)
rms_scalar_kernel(const T* __restrict__ x, int64_t n, double* mean, double* var, double* count) {
  __shared__ double s_red[32];
  double a = 0.0;
  for (int64_t i = threadIdx.x; i < n; i += blockDim.x) a += (double)x[i];
  const double bm = block_sum(a, s_red) / (double)n;
  a = 0.0;
  for (int64_t i = threadIdx.x; i < n; i += blockDim.x) {
    const double d = (double)x[i] - bm;
    a += d * d;
  }
  const double bv = block_sum(a, s_red) / (double)n;
  if (threadIdx.x == 0) {
    double m = *mean, v = *var;
    merge_moments(bm, bv, (double)n, m, v, *count);
    *mean = m; *var = v; *count += (double)n;
  }
}

__global__ void bump_count_kernel(double* count, double n) { *count += n; }

// istd[d] = 1 / sqrt(var[d] + 1e-10)  (f64; algorithms.py:114-116).  The normalisation itself is then
// clip((x - mean) * istd, +-5) in f64 -> f32: one rounding away from the reference's division, identical after the f32
// cast except in double-rounding ties; the same formula runs inside the tcgen05 A-split stage (tc_gemm.cu).
__global__ void __launch_bounds__(256) obs_istd_kernel(const double* __restrict__ var, int dim, double* __restrict__ istd) {
  const int d = blockIdx.x * blockDim.x + threadIdx.x;
  if (d < dim) istd[d] = 1.0 / sqrt(var[d] + 1e-10);
}

// grid (column blocks of 1024, row slices): a thread owns 4 consecutive columns (constants in registers) and walks rows
__global__ void __launch_bounds__(256)
normalize_obs_kernel(const float* __restrict__ obs, int64_t n, int dim, const double* __restrict__ mean,
                     const double* __restrict__ istd, float* __restrict__ out) {
  const int c0 = (blockIdx.x * 256 + threadIdx.x) * 4;
  if (c0 >= dim) return;
  const bool vec = (dim % 4 == 0) && ((((uintptr_t)obs | (uintptr_t)out) & 15) == 0);
  double m[4], s[4];
#pragma unroll
  for (int j = 0; j < 4; ++j) { m[j] = c0 + j < dim ? mean[c0 + j] : 0.0; s[j] = c0 + j < dim ? istd[c0 + j] : 0.0; }
  for (int64_t r = blockIdx.y; r < n; r += gridDim.y) {
    const int64_t base = r * dim + c0;
    float x[4];
    if (vec) { const float4 v = ld_stream4(reinterpret_cast<const float4*>(obs + base)); x[0] = v.x; x[1] = v.y; x[2] = v.z; x[3] = v.w; }
    else {
#pragma unroll
      for (int j = 0; j < 4; ++j) x[j] = c0 + j < dim ? obs[base + j] : 0.f;
    }
    float z[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) z[j] = fminf(fmaxf((float)(((double)x[j] - m[j]) * s[j]), -5.f), 5.f);
    if (vec) *reinterpret_cast<float4*>(out + base) = make_float4(z[0], z[1], z[2], z[3]);
    else {
#pragma unroll
      for (int j = 0; j < 4; ++j) if (c0 + j < dim) out[base + j] = z[j];
    }
  }
}

__global__ void sqerr_kernel(const float* __restrict__ p, const float* __restrict__ t, int64_t n, float* __restrict__ r) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) { const float d = p[i] - t[i]; r[i] = d * d; }
}

// per-row batch moments of r[T,N]
__global__ void __launch_bounds__(256) row_moments_kernel(const float* __restrict__ r, int N, double* __restrict__ mom /*[T][2]*/) {
  __shared__ double s_red[32];
  const float* row = r + (int64_t)blockIdx.x * N;
  double a = 0.0;
  for (int i = threadIdx.x; i < N; i += blockDim.x) a += (double)row[i];
  const double bm = block_sum(a, s_red) / (double)N;
  a = 0.0;
  for (int i = threadIdx.x; i < N; i += blockDim.x) { const double d = (double)row[i] - bm; a += d * d; }
  const double bv = block_sum(a, s_red) / (double)N;
  if (threadIdx.x == 0) { mom[2 * blockIdx.x] = bm; mom[2 * blockIdx.x + 1] = bv; }
}
// sequential merge over t (tiny), producing the divisor of every step   algorithms.py:396-398
__global__ void merge_rows_kernel(double* mom, int T, int N, double* mean, double* var, double* count) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  double m = *mean, v = *var, c = *count;
  for (int t = 0; t < T; ++t) {
    merge_moments(mom[2 * t], mom[2 * t + 1], (double)N, m, v, c);
    c += (double)N;
    mom[2 * t] = sqrt(v) + 1e-08;
  }
  *mean = m; *var = v; *count = c;
}
__global__ void scale_rows_kernel(float* __restrict__ r, int N, int64_t total, const double* __restrict__ mom) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < total) r[i] = (float)((double)r[i] / mom[2 * (i / N)]);
}

// one warp per row
__global__ void __launch_bounds__(256)
icm_tail_kernel(const float* __restrict__ pred, const float* __restrict__ feat, int64_t n, int F, float w_ext, float w_int,
                float* rewards, float* ri_out) {
  const int64_t row = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= n) return;
  const int lane = threadIdx.x & 31;
  float s = 0.f;
  for (int j = lane; j < F; j += 32) { const float d = pred[row * F + j] - feat[row * F + j]; s += d * d; }
  s = warp_sum(s);
  if (lane == 0) {
    const float ri = fminf(fmaxf(s / (float)F, -5.f), 5.f);
    if (ri_out) ri_out[row] = ri;
    if (rewards) rewards[row] = w_ext * rewards[row] + w_int * ri;
  }
}

template <typename IdT>
__global__ void embedding_fwd_kernel(const float* __restrict__ table, int C, const IdT* __restrict__ ids, int id_stride, int64_t B,
                                     float* __restrict__ out, int ldo) {
  const int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= B * C) return;
  const int64_t b = g / C; const int j = (int)(g - b * C);
  const int id = (int)ids[b * id_stride];
  out[b * ldo + j] = table[(int64_t)id * C + j];
}
// deterministic: thread (c, j) walks the batch in order
template <typename IdT>
__global__ void embedding_bwd_kernel(const float* __restrict__ d_out, int ldo, const IdT* __restrict__ ids, int id_stride, int64_t B,
                                     int C, float* __restrict__ d_table) {
  const int g = blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= C * C) return;
  const int c = g / C, j = g - c * C;
  float s = 0.f;
  for (int64_t b = 0; b < B; ++b)
    if ((int)ids[b * id_stride] == c) s += d_out[b * ldo + j];
  d_table[g] = s;
}

}  // namespace
}  // namespace ppx

using namespace ppx;

extern "C" int ppx_rms_update(const void* x, int x_is_f64, int64_t n, int dim, double* mean, double* var, double* count,
                              void* /*workspace*/, void* stream) {
  PPX_REQUIRE(x && mean && var && count && n >= 1 && dim >= 1, "rms_update: bad arguments");
  cudaStream_t st = (cudaStream_t)stream;
  if (dim == 1) {
    if (x_is_f64) rms_scalar_kernel<double><<<1, 1024, 0, st>>>((const double*)x, n, mean, var, count);
    else rms_scalar_kernel<float><<<1, 1024, 0, st>>>((const float*)x, n, mean, var, count);
    return after_launch("rms_update(scalar)");
  }
  const unsigned grid = (unsigned)ceil_div(dim, 32);
  if (x_is_f64) rms_cols_kernel<double><<<grid, 256, 0, st>>>((const double*)x, n, dim, mean, var, count);
  else rms_cols_kernel<float><<<grid, 256, 0, st>>>((const float*)x, n, dim, mean, var, count);
  int rc = after_launch("rms_update");
  if (rc) return rc;
  bump_count_kernel<<<1, 1, 0, st>>>(count, (double)n);
  return after_launch("rms_update(count)");
}

extern "C" int ppx_obs_istd(const double* var, int dim, double* istd, void* stream) {
  PPX_REQUIRE(var && istd && dim >= 1, "obs_istd: bad arguments");
  obs_istd_kernel<<<(unsigned)ceil_div(dim, 256), 256, 0, (cudaStream_t)stream>>>(var, dim, istd);
  return after_launch("obs_istd");
}

extern "C" int ppx_normalize_obs(const float* obs, int64_t n, int dim, const double* mean, const double* var, float* out, void* stream) {
  PPX_REQUIRE(obs && mean && var && out && n >= 0 && dim >= 1, "normalize_obs: bad arguments");
  if (n == 0) return PPX_OK;
  static GrowOnlyScratch scratch;                               // stream-ordered, one learner thread
  int rc = grow_scratch(scratch, (size_t)dim * sizeof(double));
  if (rc) return rc;
  double* istd = (double*)scratch.p;
  obs_istd_kernel<<<(unsigned)ceil_div(dim, 256), 256, 0, (cudaStream_t)stream>>>(var, dim, istd);
  rc = after_launch("normalize_obs(istd)");
  if (rc) return rc;
  const unsigned gx = (unsigned)ceil_div(dim, 1024);
  const unsigned gy = (unsigned)std::max<int64_t>(1, std::min<int64_t>(n, ceil_div((int64_t)sm_count() * 16, gx)));
  normalize_obs_kernel<<<dim3(gx, gy), 256, 0, (cudaStream_t)stream>>>(obs, n, dim, mean, istd, out);
  return after_launch("normalize_obs");
}

extern "C" int ppx_rnd_sqerr(const float* pred, const float* target, int64_t n, float* r, void* stream) {
  PPX_REQUIRE(pred && target && r && n >= 0, "rnd_sqerr: bad arguments");
  if (n == 0) return PPX_OK;
  sqerr_kernel<<<(unsigned)ceil_div(n, 256), 256, 0, (cudaStream_t)stream>>>(pred, target, n, r);
  return after_launch("rnd_sqerr");
}

extern "C" int ppx_rnd_normalize_rollout(float* r, int T, int N, double* mean, double* var, double* count, void* stream) {
  PPX_REQUIRE(r && mean && var && count && T >= 1 && N >= 1, "rnd_normalize_rollout: bad arguments");
  cudaStream_t st = (cudaStream_t)stream;
  static GrowOnlyScratch scratch;
  int rc = grow_scratch(scratch, (size_t)T * 2 * sizeof(double));
  if (rc) return rc;
  double* mom = (double*)scratch.p;
  row_moments_kernel<<<T, 256, 0, st>>>(r, N, mom);
  rc = after_launch("rnd_normalize_rollout(moments)");
  if (rc) return rc;
  merge_rows_kernel<<<1, 32, 0, st>>>(mom, T, N, mean, var, count);
  rc = after_launch("rnd_normalize_rollout(merge)");
  if (rc) return rc;
  const int64_t total = (int64_t)T * N;
  scale_rows_kernel<<<(unsigned)ceil_div(total, 256), 256, 0, st>>>(r, N, total, mom);
  return after_launch("rnd_normalize_rollout(scale)");
}

extern "C" int ppx_icm_bonus_tail(const float* pred_feat, const float* next_feat, int64_t n, int F, double eta,
                                  float* rewards_inout, float* ri_out, void* stream) {
  PPX_REQUIRE(pred_feat && next_feat && n >= 0 && F >= 1, "icm_bonus_tail: bad arguments");
  if (n == 0) return PPX_OK;
  icm_tail_kernel<<<(unsigned)ceil_div(n, 8), 256, 0, (cudaStream_t)stream>>>(pred_feat, next_feat, n, F, (float)(1.0 - eta),
                                                                               (float)eta, rewards_inout, ri_out);
  return after_launch("icm_bonus_tail");
}

extern "C" int ppx_embedding_fwd(const float* table, int C, const void* ids, int ids_are_f64, int id_stride, int64_t B,
                                 float* out, int ldo, void* stream) {
  PPX_REQUIRE(table && ids && out && C >= 1 && B >= 0 && ldo >= C, "embedding_fwd: bad arguments");
  if (B == 0) return PPX_OK;
  const unsigned grid = (unsigned)ceil_div(B * C, 256);
  if (ids_are_f64) embedding_fwd_kernel<double><<<grid, 256, 0, (cudaStream_t)stream>>>(table, C, (const double*)ids, id_stride, B, out, ldo);
  else embedding_fwd_kernel<int64_t><<<grid, 256, 0, (cudaStream_t)stream>>>(table, C, (const int64_t*)ids, id_stride, B, out, ldo);
  return after_launch("embedding_fwd");
}

extern "C" int ppx_embedding_bwd(const float* d_out, int ldo, const void* ids, int ids_are_f64, int id_stride, int64_t B, int C,
                                 float* d_table, void* stream) {
  PPX_REQUIRE(d_out && ids && d_table && C >= 1 && B >= 0, "embedding_bwd: bad arguments");
  const unsigned grid = (unsigned)ceil_div(C * C, 128);
  if (ids_are_f64) embedding_bwd_kernel<double><<<grid, 128, 0, (cudaStream_t)stream>>>(d_out, ldo, (const double*)ids, id_stride, B, C, d_table);
  else embedding_bwd_kernel<int64_t><<<grid, 128, 0, (cudaStream_t)stream>>>(d_out, ldo, (const int64_t*)ids, id_stride, B, C, d_table);
  return after_launch("embedding_bwd");
}

// ---------------------------------------------------------------------------------------------------------------
// VecNormalize on the device (SURVEY §8f.3; the reference wraps its envs in stable_baselines3's VecNormalize with
// norm_reward=True, env.py:11): running observation statistics + normalisation, discounted-return statistics + reward
// normalisation, the per-env return accumulator reset on `done`.  The running moments are the RunningMeanStd state of
// ppx_rms_update (util.py:9-44 has the same update rule as stable_baselines3's).
namespace ppx {
namespace {

__global__ void __launch_bounds__(256)
vecnorm_obs_kernel(const float* __restrict__ obs, int64_t n, int dim, const double* __restrict__ mean, const double* __restrict__ var,
                   double eps, float clip, float* __restrict__ out) {
  const int64_t total = n * dim;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int d = (int)(i % dim);
    const double z = ((double)obs[i] - mean[d]) / sqrt(var[d] + eps);
    out[i] = fminf(fmaxf((float)z, -clip), clip);
  }
}

// one CTA.  While training (update): ret = ret * gamma + r; ret_rms.update(ret).  Then r_out = clip(r / sqrt(ret_var + eps),
// +-clip) and ret[done] = 0.  As in stable_baselines3's step_wait, the returns do not accumulate when not training.
__global__ void __launch_bounds__(1024)
vecnorm_reward_kernel(const float* __restrict__ r, const uint8_t* __restrict__ done, double* __restrict__ ret, int n, double gamma,
                      double* mean, double* var, double* count, double eps, float clip, int update, float* __restrict__ out) {
  __shared__ double s_red[32];
  __shared__ double s_var;
  if (update) {
    double a = 0.0;
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
      const double v = ret[i] * gamma + (double)r[i];
      ret[i] = v;
      a += v;
    }
    const double bm = block_sum(a, s_red) / (double)n;
    a = 0.0;
    for (int i = threadIdx.x; i < n; i += blockDim.x) { const double d = ret[i] - bm; a += d * d; }
    const double bv = block_sum(a, s_red) / (double)n;
    if (threadIdx.x == 0) {
      double m = *mean, v = *var;
      merge_moments(bm, bv, (double)n, m, v, *count);
      *mean = m; *var = v; *count += (double)n;
      s_var = v;
    }
  } else if (threadIdx.x == 0) {
    s_var = *var;
  }
  __syncthreads();
  const double inv = 1.0 / sqrt(s_var + eps);
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    out[i] = fminf(fmaxf((float)((double)r[i] * inv), -clip), clip);
    if (done[i]) ret[i] = 0.0;
  }
}

}  // namespace
}  // namespace ppx

extern "C" int ppx_vecnorm_obs(const float* obs, int64_t n, int dim, const double* mean, const double* var, double eps, double clip,
                               float* out, void* stream) {
  PPX_REQUIRE(obs && mean && var && out && n >= 0 && dim >= 1 && clip > 0.0, "vecnorm_obs: bad arguments");
  if (n == 0) return PPX_OK;
  const unsigned grid = (unsigned)std::min<int64_t>(ceil_div(n * dim, 256), (int64_t)sm_count() * 16);
  ppx::vecnorm_obs_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(obs, n, dim, mean, var, eps, (float)clip, out);
  return after_launch("vecnorm_obs");
}

extern "C" int ppx_vecnorm_reward(const float* rewards, const uint8_t* dones, double* returns_inout, int n, double gamma,
                                  double* ret_mean, double* ret_var, double* ret_count, double eps, double clip, int update_stats,
                                  float* rewards_out, void* stream) {
  PPX_REQUIRE(rewards && dones && returns_inout && ret_mean && ret_var && ret_count && rewards_out && n >= 1 && clip > 0.0,
              "vecnorm_reward: bad arguments");
  ppx::vecnorm_reward_kernel<<<1, 1024, 0, (cudaStream_t)stream>>>(rewards, dones, returns_inout, n, gamma, ret_mean, ret_var, ret_count,
                                                                   eps, (float)clip, update_stats, rewards_out);
  return after_launch("vecnorm_reward");
}
