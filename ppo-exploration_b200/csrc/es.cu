// ES-NSRA step: shared noise table, population perturbation, fitness-shaped parameter update,
// centred ranks and novelty k-NN over the behaviour archive.
//
// Replaces EvolutionStrategy._get_population/_get_weights_try (evolution_strategies.py:137-145,
// 172-182), _update_weights (:217-239) and get_kNN + the novelty lines (:264-281, :318-325).
//
// The reference draws fresh randn per member and stacks a [P,in,out] f64 tensor per layer each
// iteration.  Here a population member is an int64 offset into one resident f32 noise table
// (ppx_noise_fill), theta is one flat f64 vector over all layers, and both hot kernels stream the
// noise exactly once:
//   perturb  out[p,:] = theta + sigma*eps_p            8*D  B/perturbation  (f32 out)
//   update   theta   += f * sum_p c_p eps_p            4*D  B/perturbation  (GEMV, f64 accumulate,
//                                                      split over members, fixed-order reduction)
// Parity mode passes a dense [P,D] eps (offsets == NULL) holding the very values given to the
// reference.  All state (theta, lr) stays on device; the std==0 early-out of :225-226 is a device flag.
#include "es_walk.cuh"
#include "p2p.cuh"
#include "philox.cuh"

namespace ppx {
namespace {

__global__ void __launch_bounds__(256) noise_kernel(float* __restrict__ table, int64_t n, uint64_t seed) {
  const int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;      // quad index
  if (q * 4 >= n) return;
  uint32_t c[4] = {(uint32_t)q, (uint32_t)(q >> 32), 0u, 0u};
  philox4x32(c, seed);
  float z[4];
  box_muller(c[0], c[1], z[0], z[1]);
  box_muller(c[2], c[3], z[2], z[3]);
#pragma unroll
  for (int e = 0; e < 4; ++e)
    if (q * 4 + e < n) table[q * 4 + e] = z[e];
}

// population = P offsets into the noise table, drawn on the device: Philox4x32-10 keyed by the seed, counter =
// (member, draw number); the draw number lives on the device and is bumped here, so the launch replays from a CUDA
// graph and every rank (same seed, same number) draws the identical population.  Offsets are multiples of 4 (16-byte
// aligned noise rows).  draw[0] = the draw number, draw[1] = ticket word of the last-block detection (zero).
__global__ void __launch_bounds__(256) es_offsets_kernel(uint64_t seed, int64_t* draw, int P, int64_t hi, int64_t* __restrict__ out) {
  const uint64_t n = (uint64_t)draw[0];                     // every block reads the draw number before the LAST block bumps it
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p < P) {
    uint32_t c[4] = {(uint32_t)p, (uint32_t)n, (uint32_t)(n >> 32), 0x6f666673u};
    philox4x32(c, seed);
    const uint64_t u = ((uint64_t)c[1] << 32) | c[0];
    out[p] = (int64_t)(u % (uint64_t)hi) * 4;
  }
  if (last_block_done(reinterpret_cast<unsigned int*>(draw + 1)) && threadIdx.x == 0) draw[0] = (int64_t)(n + 1);
}

// ---------------- perturb ----------------
template <typename OutT>
__global__ void __launch_bounds__(256)
perturb_kernel(const double* __restrict__ theta, const float* __restrict__ noise, const int64_t* __restrict__ offsets,
               double sigma, int P, int D, OutT* __restrict__ out) {
  const int p = blockIdx.y;
  const float* eps = noise + (offsets ? offsets[p] : (int64_t)p * D);
  OutT* o = out + (int64_t)p * D;
  for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < D; j += gridDim.x * blockDim.x) {
    // w + SIGMA * eps with separate rounding of product and sum, like numpy (evolution_strategies.py:143-144)
    o[j] = (OutT)__dadd_rn(theta[j], __dmul_rn(sigma, (double)ld_stream(eps + j)));
  }
}

// Same arithmetic over the flat [P, D/4] index space with 16-byte noise loads (D % 4 == 0, every member's noise
// row 16-byte aligned): a persistent grid-stride loop, two independent quads in flight per thread.
template <typename OutT>
__global__ void __launch_bounds__(256)
perturb_vec_kernel(const double* __restrict__ theta, const float* __restrict__ noise, const int64_t* __restrict__ offsets,
                   double sigma, int P, int D4, OutT* __restrict__ out) {
  const int64_t total = (int64_t)P * D4, stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += stride) {
    const int p = (int)(i / D4), j = (int)(i - (int64_t)p * D4) * 4;
    const float* eps = noise + (offsets ? __ldg(offsets + p) : (int64_t)p * D4 * 4) + j;
    const float4 e = ld_stream4(reinterpret_cast<const float4*>(eps));
    const double2 t0 = __ldg(reinterpret_cast<const double2*>(theta + j));
    const double2 t1 = __ldg(reinterpret_cast<const double2*>(theta + j + 2));
    const double r0 = __dadd_rn(t0.x, __dmul_rn(sigma, (double)e.x)), r1 = __dadd_rn(t0.y, __dmul_rn(sigma, (double)e.y));
    const double r2 = __dadd_rn(t1.x, __dmul_rn(sigma, (double)e.z)), r3 = __dadd_rn(t1.y, __dmul_rn(sigma, (double)e.w));
    OutT* o = out + (int64_t)p * D4 * 4 + j;
    if (sizeof(OutT) == 4) {
      *reinterpret_cast<float4*>(o) = make_float4((float)r0, (float)r1, (float)r2, (float)r3);
    } else {
      *reinterpret_cast<double2*>(o) = make_double2(r0, r1);
      *reinterpret_cast<double2*>(o + 2) = make_double2(r2, r3);
    }
  }
}

// ---------------- population forward (FeedForwardNetwork.predict, evolution_strategies.py:48-61) ----------------
// Every member p acts on its own observation with weights theta + sigma*eps_p formed on the fly from the noise table --
// the perturbed weights are never materialised (ppx_es_perturb writes 8 D bytes per member for the same purpose).
// The per-member layer walk is es_walk.cuh (shared with ppx_es_act).
// fp32 arithmetic (the reference is f64; the B200's FP64 pipe made an f64 version 6x slower than this one -- 250 us vs
// 40 us at C5 -- and the path's bound is 1e-5 relative): hidden layers arctan (:57), last layer linear, then tanh for
// Box action spaces (continuous_action :84-89).
struct EsFwdP {
  const double* theta; const float* noise; const int64_t* offsets; float sigma; int P, D, n_layers;
  int sizes[kFwdMaxLayers + 1];
  int vec[kFwdMaxLayers];                                   // 4: 16-byte slot path, 1: scalar slot path (narrow layer), 0: generic (host-checked)
  const double* obs; double* out; int squash;
};

__global__ void __launch_bounds__(256) es_forward_kernel(EsFwdP p) {
  extern __shared__ float sm_f[];
  float* th = sm_f;                                         // [D]
  float* act = th + ((p.D + 3) & ~3);                       // [8 warps][2][kFwdMaxWidth]
  for (int i = threadIdx.x; i < p.D; i += blockDim.x) th[i] = (float)__ldg(p.theta + i);
  __syncthreads();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  float* a0 = act + (size_t)warp * 2 * kFwdMaxWidth;
  float* a1 = a0 + kFwdMaxWidth;
  for (int m = blockIdx.x * 8 + warp; m < p.P; m += gridDim.x * 8) {
    const float* eps = p.noise + (p.offsets ? __ldg(p.offsets + m) : (int64_t)m * p.D);
    for (int i = lane; i < p.sizes[0]; i += 32) a0[i] = (float)__ldg(p.obs + (size_t)m * p.sizes[0] + i);
    __syncwarp();
    es_member_walk(p, eps, th, a0, a1, lane,
                   [&](int j, int no, float v) { p.out[(size_t)m * no + j] = (double)(p.squash ? tanhf(v) : v); });
  }
}

// ---------------- update ----------------
// stats[0]=mean, stats[1]=std(ddof 0), stats[2]=skip flag
__global__ void __launch_bounds__(1024) es_stats_kernel(const double* __restrict__ r, int P, int rank_mode, double* stats, int* status) {
  __shared__ double s_red[32];
  double a = 0.0;
  for (int i = threadIdx.x; i < P; i += blockDim.x) a += r[i];
  const double mean = block_sum(a, s_red) / (double)P;
  a = 0.0;
  for (int i = threadIdx.x; i < P; i += blockDim.x) { const double d = r[i] - mean; a += d * d; }
  const double var = block_sum(a, s_red) / (double)P;
  if (threadIdx.x == 0) {
    const double sd = sqrt(var);
    const bool skip = !rank_mode && (sd == 0.0);
    stats[0] = mean; stats[1] = sd; stats[2] = skip ? 1.0 : 0.0;
    if (status) *status = skip ? 1 : 0;
  }
}

__global__ void __launch_bounds__(256)
rank_kernel(const double* __restrict__ r, int P, int64_t* __restrict__ rank_out, double* __restrict__ centred_out) {
  __shared__ double s_r[256];
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  const double mine = p < P ? r[p] : 0.0;
  int64_t cnt = 0;
  for (int base = 0; base < P; base += 256) {
    const int q = base + threadIdx.x;
    s_r[threadIdx.x] = q < P ? r[q] : 0.0;
    __syncthreads();
    const int lim = min(256, P - base);
    for (int t = 0; t < lim; ++t) {
      const double o = s_r[t];
      cnt += (o < mine) || (o == mine && (base + t) < p);
    }
    __syncthreads();
  }
  if (p < P) {
    if (rank_out) rank_out[p] = cnt;
    if (centred_out) centred_out[p] = (double)cnt / (double)(P - 1) - 0.5;
  }
}

// coef[p] = f * shaped fitness (0 everywhere when the update is skipped)
__global__ void __launch_bounds__(256)
es_coef_kernel(const double* __restrict__ r, const double* __restrict__ centred, int P, const double* __restrict__ stats,
               const double* __restrict__ lr, double sigma, double nw, double novelty, const double* __restrict__ novelty_dev,
               int use_novelty, int rank_mode, double* __restrict__ coef) {
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= P) return;
  if (stats[2] != 0.0) { coef[p] = 0.0; return; }
  if (novelty_dev) novelty = *novelty_dev;
  const double f = *lr / ((double)P * sigma);                          // update_factor, :230
  double z = rank_mode ? centred[p] : (r[p] - stats[0]) / stats[1];   // :227
  if (use_novelty) z = ((1.0 - nw) * z + nw * novelty) / 2.0;          // :235
  coef[p] = f * z;
}

// z-score path in ONE launch: mean / std (ddof 0) / skip flag, then the coefficients of all P members
__global__ void __launch_bounds__(1024)
es_stats_coef_kernel(const double* __restrict__ r, int P, double* stats, int* status, const double* __restrict__ lr, double sigma,
                     double nw, double novelty, const double* __restrict__ novelty_dev, int use_novelty, double* __restrict__ coef) {
  __shared__ double s_red[32];
  double a = 0.0;
  for (int i = threadIdx.x; i < P; i += blockDim.x) a += r[i];
  const double mean = block_sum(a, s_red) / (double)P;
  a = 0.0;
  for (int i = threadIdx.x; i < P; i += blockDim.x) { const double d = r[i] - mean; a += d * d; }
  const double sd = sqrt(block_sum(a, s_red) / (double)P);
  const bool skip = (sd == 0.0);
  if (threadIdx.x == 0) {
    stats[0] = mean; stats[1] = sd; stats[2] = skip ? 1.0 : 0.0;
    if (status) *status = skip ? 1 : 0;
  }
  if (novelty_dev) novelty = *novelty_dev;
  const double f = *lr / ((double)P * sigma);
  for (int p = threadIdx.x; p < P; p += blockDim.x) {
    double z = (r[p] - mean) / sd;
    if (use_novelty) z = ((1.0 - nw) * z + nw * novelty) / 2.0;
    coef[p] = skip ? 0.0 : f * z;
  }
}

template <bool VEC>
__global__ void __launch_bounds__(128)
es_gemv_kernel(const float* __restrict__ noise, const int64_t* __restrict__ offsets, const double* __restrict__ coef, int P, int D,
               int p_chunk, double* __restrict__ partial) {
  const int j = (blockIdx.x * 128 + threadIdx.x) * 4;
  const int p0 = min(P, (int)blockIdx.y * p_chunk), p1 = min(P, p0 + p_chunk);
  double a0 = 0.0, a1 = 0.0, a2 = 0.0, a3 = 0.0;
  if (j < D) {
#pragma unroll 8
    for (int p = p0; p < p1; ++p) {
      const float* eps = noise + (offsets ? __ldg(offsets + p) : (int64_t)p * D) + j;
      const double c = __ldg(coef + p);
      float4 e;
      if (VEC) e = ld_stream4(reinterpret_cast<const float4*>(eps));
      else {
        e.x = ld_stream(eps);
        e.y = j + 1 < D ? ld_stream(eps + 1) : 0.f;
        e.z = j + 2 < D ? ld_stream(eps + 2) : 0.f;
        e.w = j + 3 < D ? ld_stream(eps + 3) : 0.f;
      }
      a0 = fma(c, (double)e.x, a0); a1 = fma(c, (double)e.y, a1);
      a2 = fma(c, (double)e.z, a2); a3 = fma(c, (double)e.w, a3);
    }
    double* out = partial + (int64_t)blockIdx.y * D + j;
    out[0] = a0;
    if (j + 1 < D) out[1] = a1;
    if (j + 2 < D) out[2] = a2;
    if (j + 3 < D) out[3] = a3;
  }
}

// column sums of the per-split partials in a fixed order: block = 32 columns x 8 slices of the split list (slice q takes
// splits q, q+8, ...), slices combined 0..7.  Single GPU: theta += sum (unless the std == 0 early-out) and lr *= decay;
// sharded: this rank's partial update over ITS members -> the peer-visible buffer (es_apply_p2p_kernel sums the ranks).
__global__ void __launch_bounds__(256)
es_colsum_kernel(const double* __restrict__ partial, int splits, int D, const double* __restrict__ stats, double* __restrict__ theta,
                 double* __restrict__ dtheta, double decay, double* lr) {
  __shared__ double sl[8][33];
  const int c = threadIdx.x & 31, q = threadIdx.x >> 5, j = blockIdx.x * 32 + c;
  double a = 0.0;
  if (j < D)
    for (int k = q; k < splits; k += 8) a += partial[(int64_t)k * D + j];
  sl[q][c] = a;
  __syncthreads();
  if (q != 0 || j >= D) return;
  const bool skip = stats[2] != 0.0;
  double sum = 0.0;
#pragma unroll
  for (int k = 0; k < 8; ++k) sum += sl[k][c];
  if (dtheta) dtheta[j] = skip ? 0.0 : sum;
  else if (!skip) theta[j] += sum;
  if (!dtheta && j == 0 && !skip) *lr *= decay;                        // :239 (not reached on the early return)
}

// sharded update, last step: theta += sum over ranks (rank order: identical on every replica) of the peers' partial updates
__global__ void __launch_bounds__(1024)
es_apply_p2p_kernel(p2p::Peers P, double* __restrict__ theta, int D, const double* __restrict__ stats, double decay, double* lr) {
  if (threadIdx.x < 32) p2p::barrier_all(P);
  __syncthreads();
  const bool skip = stats[2] != 0.0;
  if (skip) return;
  for (int j = threadIdx.x; j < D; j += blockDim.x) {
    double s = 0.0;
    for (int r = 0; r < P.W; ++r) s += p2p::ld_peer_f64((const double*)P.data[r] + j);
    theta[j] += s;
  }
  if (threadIdx.x == 0) *lr *= decay;
}

__global__ void __launch_bounds__(256)
es_apply_kernel(double* __restrict__ theta, const double* __restrict__ partial, int splits, int D, const double* __restrict__ stats,
                double decay, double* lr) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  const bool skip = stats[2] != 0.0;
  if (j < D && !skip) {
    double s = 0.0;
    for (int k = 0; k < splits; ++k) s += partial[(int64_t)k * D + j];
    theta[j] += s;
  }
  if (j == 0 && !skip) *lr *= decay;                                   // :239 (not reached on the early return)
}

// ---------------- novelty k-NN ----------------
// Exact k-NN distance sums.  Stage 1: grid (splits, Q), one WARP per (query, archive slice): every lane keeps a
// sorted top-K of the distances it saw, a K-round warp merge pops the slice's K smallest in ascending order into
// cand[q][split][K].  Stage 2: one warp per query merges the splits*K candidates the same way and sums the S
// smallest in ascending order (the order the reference's sorted kneighbors() output is summed in).  Few queries
// (the reference asks for 2 per iteration) still spread over the whole machine through the archive split.
// Distances use explicit __dmul_rn/__dadd_rn (no FMA contraction) -> bit-equal to the direct CPU distance.
template <int KMAX>
__device__ __forceinline__ void warp_pop_sorted(double (&best)[KMAX], int rounds, int lane, double* out /*[rounds] or null*/, double* sum) {
  double acc = 0.0;
  for (int round = 0; round < rounds; ++round) {
    double mn = best[0];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) mn = fmin(mn, __shfl_xor_sync(0xffffffffu, mn, o));
    const unsigned who = __ballot_sync(0xffffffffu, best[0] == mn);
    acc = __dadd_rn(acc, mn);
    if (out && lane == 0) out[round] = mn;
    if (lane == __ffs(who) - 1) {
#pragma unroll
      for (int i = 0; i + 1 < KMAX; ++i) best[i] = best[i + 1];
      best[KMAX - 1] = INFINITY;
    }
  }
  if (sum) *sum = acc;
}

template <int KMAX>
__device__ __forceinline__ void sorted_insert(double (&best)[KMAX], double v) {
  if (v < best[KMAX - 1]) {
#pragma unroll
    for (int i = 0; i < KMAX; ++i) {
      if (v < best[i]) { const double t = best[i]; best[i] = v; v = t; }
    }
  }
}

template <int KMAX>
__global__ void __launch_bounds__(32)
knn_slice_kernel(const double* __restrict__ archive, int64_t M, const double* __restrict__ queries, int dim, int K,
                 int splits, double* __restrict__ cand) {
  const int q = blockIdx.y, sp = blockIdx.x, lane = threadIdx.x;
  const int64_t per = (M + splits - 1) / splits, m0 = sp * per, m1 = min(M, m0 + per);
  const double* qv = queries + (int64_t)q * dim;
  double best[KMAX];
#pragma unroll
  for (int i = 0; i < KMAX; ++i) best[i] = INFINITY;
  for (int64_t m = m0 + lane; m < m1; m += 32) {
    const double* a = archive + m * dim;
    double d2 = 0.0;
    for (int d = 0; d < dim; ++d) {
      const double diff = __dsub_rn(a[d], qv[d]);
      d2 = __dadd_rn(d2, __dmul_rn(diff, diff));                      // no FMA contraction: match the CPU distance
    }
    sorted_insert<KMAX>(best, __dsqrt_rn(d2));
  }
  warp_pop_sorted<KMAX>(best, K, lane, cand + ((int64_t)q * splits + sp) * K, nullptr);   // INF-padded when the slice is short
}

template <int KMAX>
__global__ void __launch_bounds__(32)
knn_merge_kernel(const double* __restrict__ cand, int n_cand, int64_t M, int K, double* __restrict__ sum_out,
                 double* __restrict__ nov_out) {
  const int q = blockIdx.x, lane = threadIdx.x;
  double best[KMAX];
#pragma unroll
  for (int i = 0; i < KMAX; ++i) best[i] = INFINITY;
  for (int c = lane; c < n_cand; c += 32) sorted_insert<KMAX>(best, cand[(int64_t)q * n_cand + c]);
  const int S = (int)min((int64_t)K, M);
  double sum;
  warp_pop_sorted<KMAX>(best, S, lane, nullptr, &sum);
  if (lane == 0) {
    if (sum_out) sum_out[q] = sum;
    if (nov_out) {
      double nu = sum / (double)S;
      if (nu <= 1e-3) nu = 5e-3;                                       // :323-324
      nov_out[q] = nu;
    }
  }
}

// ---------------- novelty k-NN for a population of queries ----------------
// ppx_knn_novelty_many: one THREAD per query, so any Q runs in one launch with no scratch.  Archive rows pass through shared
// memory in tiles of kKnnTile rows; every thread of the CTA reads the same row (a shared-memory broadcast).  Each thread keeps
// a sorted top-K of SQUARED distances in registers and takes square roots only of its S = min(K, M) winners at the end.
// Why this equals ppx_knn_novelty bit for bit: d2 is formed by the same sequence of __dsub_rn / __dmul_rn / __dadd_rn, and a
// correctly rounded square root is monotone (x <= y -> sqrt(x) <= sqrt(y)).  Sorting the d2 ascending and applying
// __dsqrt_rn keeps the list sorted, so the first S entries are a valid choice of the S smallest distances -- and the multiset
// of the S smallest values of a list is unique.  Summing them ascending from 0.0 with __dadd_rn is then the very sum
// knn_merge_kernel pops (equal values in either order add identically).  A row whose d2 is not below the current K-th best
// cannot change that multiset and is rejected with one compare.
constexpr int kKnnTile = 256, kKnnManyMaxDim = 8, kKnnManyThreads = 64;

template <int KMAX>
__global__ void __launch_bounds__(kKnnManyThreads)
knn_many_kernel(const double* __restrict__ archive, int64_t M, const double* __restrict__ queries, int Q, int dim, int K,
                double* __restrict__ sum_out, double* __restrict__ nov_out) {
  __shared__ double tile[kKnnTile * kKnnManyMaxDim];
  const int q = blockIdx.x * kKnnManyThreads + threadIdx.x;
  const bool live = q < Q;
  double qv[kKnnManyMaxDim];
#pragma unroll
  for (int d = 0; d < kKnnManyMaxDim; ++d) qv[d] = (live && d < dim) ? queries[(int64_t)q * dim + d] : 0.0;
  // the top K sit right-aligned in best[KMAX - K .. KMAX): -inf below them keeps the array sorted, so sorted_insert works
  // unchanged and the K-th best is always best[KMAX - 1], a fixed register
  double best[KMAX];
#pragma unroll
  for (int i = 0; i < KMAX; ++i) best[i] = i < KMAX - K ? -INFINITY : INFINITY;
  for (int64_t base = 0; base < M; base += kKnnTile) {
    const int rows = (int)min((int64_t)kKnnTile, M - base);
    __syncthreads();
    for (int i = threadIdx.x; i < rows * dim; i += kKnnManyThreads) tile[i] = archive[base * dim + i];
    __syncthreads();
    if (!live) continue;
    for (int r = 0; r < rows; ++r) {
      const double* a = tile + r * dim;
      double d2 = 0.0;
#pragma unroll
      for (int d = 0; d < kKnnManyMaxDim; ++d) {
        if (d < dim) {
          const double diff = __dsub_rn(a[d], qv[d]);
          d2 = __dadd_rn(d2, __dmul_rn(diff, diff));                   // no FMA contraction: the existing kernel's distance
        }
      }
      if (d2 < best[KMAX - 1]) sorted_insert<KMAX>(best, d2);
    }
  }
  if (!live) return;
  const int S = (int)min((int64_t)K, M);
  double sum = 0.0;
#pragma unroll
  for (int i = 0; i < KMAX; ++i)
    if (i >= KMAX - K && i < KMAX - K + S) sum = __dadd_rn(sum, __dsqrt_rn(best[i]));
  if (sum_out) sum_out[q] = sum;
  if (nov_out) {
    double nu = sum / (double)S;
    if (nu <= 1e-3) nu = 5e-3;                                         // :323-324
    nov_out[q] = nu;
  }
}

// ---------------- update with a novelty per member (NSRA-ES, Conti et al. 2018, Alg. 3) ----------------
// mean and ddof-0 variance of v[0..P) by the block reduction of es_stats_coef_kernel (same summation order)
__device__ __forceinline__ void block_mean_var(const double* __restrict__ v, int P, double* s_red, double& mean, double& var) {
  double a = 0.0;
  for (int i = threadIdx.x; i < P; i += blockDim.x) a += v[i];
  mean = block_sum(a, s_red) / (double)P;
  a = 0.0;
  for (int i = threadIdx.x; i < P; i += blockDim.x) { const double d = v[i] - mean; a += d * d; }
  var = block_sum(a, s_red) / (double)P;
}

// z-score path in ONE launch: both vectors shaped (a zero-std vector shapes to 0), skip only when both stds are 0,
// coef[p] = lr/(P sigma) * ((1-w) F~_p + w N~_p) / 2
__global__ void __launch_bounds__(1024)
es_member_stats_coef_kernel(const double* __restrict__ r, const double* __restrict__ nov, int P, double* stats, int* status,
                            const double* __restrict__ lr, double sigma, double nw, double* __restrict__ coef) {
  __shared__ double s_red[32];
  double mr, vr, mn, vn;
  block_mean_var(r, P, s_red, mr, vr);
  block_mean_var(nov, P, s_red, mn, vn);
  const double sr = __dsqrt_rn(vr), sn = __dsqrt_rn(vn);
  const bool skip = (sr == 0.0) && (sn == 0.0);
  if (threadIdx.x == 0) {
    stats[0] = mr; stats[1] = sr; stats[2] = skip ? 1.0 : 0.0; stats[3] = mn; stats[4] = sn;
    if (status) *status = skip ? 1 : 0;
  }
  const double f = *lr / ((double)P * sigma);
  // F~ first, then N~ and the mix: each pass keeps few values live across the division's slow-path call (no spills)
  for (int p = threadIdx.x; p < P; p += blockDim.x) coef[p] = sr == 0.0 ? 0.0 : (r[p] - mr) / sr;
  for (int p = threadIdx.x; p < P; p += blockDim.x) {
    const double N = sn == 0.0 ? 0.0 : (nov[p] - mn) / sn;
    coef[p] = skip ? 0.0 : f * (((1.0 - nw) * coef[p] + nw * N) / 2.0);
  }
}

// centred-rank path, after rank_kernel on each vector: never skips
__global__ void __launch_bounds__(256)
es_member_rank_coef_kernel(const double* __restrict__ cf, const double* __restrict__ cn, int P, double* stats, int* status,
                           const double* __restrict__ lr, double sigma, double nw, double* __restrict__ coef) {
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p == 0) {
    stats[2] = 0.0;
    if (status) *status = 0;
  }
  if (p >= P) return;
  const double f = *lr / ((double)P * sigma);
  coef[p] = f * (((1.0 - nw) * cf[p] + nw * cn[p]) / 2.0);
}

int gemv_splits(int P, int D) {
  const int64_t colblocks = ceil_div(D, 512);
  int64_t s = ceil_div(16 * (int64_t)sm_count(), colblocks);      // measured at C5: 35 us with 16 CTAs per SM, 63 us with 4
  s = std::max<int64_t>(1, std::min<int64_t>(s, std::max(1, P / 32)));
  return (int)s;
}

}  // namespace
}  // namespace ppx

using namespace ppx;

extern "C" int ppx_noise_fill(float* table, int64_t n, uint64_t seed, void* stream) {
  PPX_REQUIRE(table && n >= 1, "noise_fill: bad arguments");
  noise_kernel<<<(unsigned)ceil_div(ceil_div(n, 4), 256), 256, 0, (cudaStream_t)stream>>>(table, n, seed);
  return after_launch("noise_fill");
}

extern "C" int ppx_es_perturb(const double* theta, const float* noise, const int64_t* offsets, double sigma, int P, int D,
                              void* out, int out_is_f64, void* stream) {
  PPX_REQUIRE(theta && noise && out && P >= 1 && D >= 1, "es_perturb: bad arguments");
  // fast path: 16-byte vectors (the table sampler hands out offsets that are multiples of 4; dense eps needs D % 4 == 0)
  bool vec = (D % 4 == 0) && ((uintptr_t)noise % 16 == 0) && ((uintptr_t)theta % 16 == 0) && ((uintptr_t)out % 16 == 0);
  if (vec && offsets) {
    // offsets live on the device: the caller promises 4-alignment through ppx_es_perturb's contract (see ppx.h)
  }
  if (vec) {
    const int64_t total = (int64_t)P * (D / 4);
    const unsigned g = (unsigned)std::min<int64_t>(ceil_div(total, 256), (int64_t)sm_count() * 16);
    if (out_is_f64) perturb_vec_kernel<double><<<g, 256, 0, (cudaStream_t)stream>>>(theta, noise, offsets, sigma, P, D / 4, (double*)out);
    else perturb_vec_kernel<float><<<g, 256, 0, (cudaStream_t)stream>>>(theta, noise, offsets, sigma, P, D / 4, (float*)out);
    return after_launch("es_perturb(vec)");
  }
  dim3 grid((unsigned)std::min<int64_t>(ceil_div(D, 256), 64), (unsigned)P);
  PPX_REQUIRE(P <= 65535, "es_perturb: P=%d exceeds grid.y limit; call in slices", P);
  if (out_is_f64) perturb_kernel<double><<<grid, 256, 0, (cudaStream_t)stream>>>(theta, noise, offsets, sigma, P, D, (double*)out);
  else perturb_kernel<float><<<grid, 256, 0, (cudaStream_t)stream>>>(theta, noise, offsets, sigma, P, D, (float*)out);
  return after_launch("es_perturb");
}

extern "C" int ppx_es_forward(const double* theta, const float* noise, const int64_t* offsets, double sigma, int P,
                              const int* layer_sizes, int n_layers, const double* obs, int squash_tanh, double* out,
                              void* stream) {
  PPX_REQUIRE(theta && noise && layer_sizes && obs && out, "es_forward: null pointer");
  PPX_REQUIRE(P >= 1, "es_forward: P=%d", P);
  EsFwdP p{};
  p.theta = theta; p.noise = noise; p.offsets = offsets; p.sigma = (float)sigma; p.P = P;
  p.obs = obs; p.out = out; p.squash = squash_tanh;
  int rc = es_plan(p, noise, offsets, layer_sizes, n_layers, "es_forward");
  if (rc) return rc;
  const int D = p.D;
  const size_t smem = sizeof(float) * ((size_t)((D + 3) & ~3) + 8 * 2 * kFwdMaxWidth);
  PPX_REQUIRE(smem <= 227 * 1024, "es_forward: %d parameters do not fit in shared memory", D);
  static size_t configured = 0;
  if (smem > configured) {
    PPX_CUDA(cudaFuncSetAttribute(es_forward_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    configured = smem;
  }
  // persistent grid with a WHOLE number of members per warp (1.4 members per warp = some warps doing 2 and the rest 1)
  static int per_sm = 0;
  if (!per_sm) {
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, es_forward_kernel, 256, smem) != cudaSuccess || per_sm < 1) per_sm = 1;
  }
  const int64_t resident = (int64_t)sm_count() * per_sm;
  const int64_t k = std::max<int64_t>(1, ceil_div(P, 8 * resident));
  const unsigned grid = (unsigned)ceil_div(P, 8 * k);
  es_forward_kernel<<<grid, 256, smem, (cudaStream_t)stream>>>(p);
  return after_launch("es_forward");
}

extern "C" int64_t ppx_es_update_workspace(int P, int D) {
  return (int64_t)sizeof(double) * (8 + 2 * (int64_t)P + (int64_t)gemv_splits(P, D) * D);
}

extern "C" int ppx_es_offsets(uint64_t seed, int64_t* draw_dev, int P, int64_t table_size, int D, int64_t* offsets_out, void* stream) {
  PPX_REQUIRE(draw_dev && offsets_out && P >= 1 && D >= 1 && table_size >= D + 4, "es_offsets: bad arguments");
  es_offsets_kernel<<<(unsigned)ceil_div(P, 256), 256, 0, (cudaStream_t)stream>>>(seed, draw_dev, P, (table_size - D) / 4, offsets_out);
  return after_launch("es_offsets");
}

namespace {
// the GEMV over members [p_lo, p_lo + p_n) of coef[0..P) with the column-sum tail: theta += update and lr *= decay
// (dtheta_out NULL), or this rank's partial update -> dtheta_out
int es_gemv_tail(double* theta, const float* noise, const int64_t* offsets, const double* coef, int P, int p_lo, int p_n, int D,
                 const double* stats, double decay, double* lr_inout, double* partial, double* dtheta_out, cudaStream_t st) {
  const int splits = gemv_splits(P, D);
  const int p_chunk = (int)ceil_div(p_n, splits);
  dim3 grid((unsigned)ceil_div(D, 512), (unsigned)splits);
  const bool vec = (D % 4 == 0) && ((uintptr_t)noise % 16 == 0);
  // with offsets, vector loads need every offset to be a multiple of 4 -- the table sampler guarantees it
  // (see host wrapper); dense parity inputs only need D % 4 == 0.
  const float* nz = offsets ? noise : noise + (int64_t)p_lo * D;
  if (vec) es_gemv_kernel<true><<<grid, 128, 0, st>>>(nz, offsets ? offsets + p_lo : nullptr, coef + p_lo, p_n, D, p_chunk, partial);
  else es_gemv_kernel<false><<<grid, 128, 0, st>>>(nz, offsets ? offsets + p_lo : nullptr, coef + p_lo, p_n, D, p_chunk, partial);
  int rc = after_launch("es_update(gemv)");
  if (rc) return rc;
  es_colsum_kernel<<<(unsigned)ceil_div(D, 32), 256, 0, st>>>(partial, splits, D, stats, theta, dtheta_out, decay, lr_inout);
  return after_launch("es_update(column sums)");
}

// stats + coefficients over ALL P rewards (replicated: every rank computes the identical z-scores), then the GEMV over
// members [p_lo, p_lo + p_n) with the column-sum tail
int es_update_core(double* theta, const float* noise, const int64_t* offsets, const double* rewards, int P, int p_lo, int p_n, int D,
                   double sigma, double novelty_param, double novelty, const double* novelty_dev, int use_novelty, double decay,
                   double* lr_inout, int* status_out, void* workspace, double* dtheta_out, cudaStream_t st) {
  double* stats = (double*)workspace;
  double* coef = stats + 8;
  double* partial = coef + 2 * (int64_t)P;
  es_stats_coef_kernel<<<1, 1024, 0, st>>>(rewards, P, stats, status_out, lr_inout, sigma, novelty_param, novelty, novelty_dev,
                                           use_novelty, coef);
  int rc = after_launch("es_update(stats+coef)");
  if (rc) return rc;
  return es_gemv_tail(theta, noise, offsets, coef, P, p_lo, p_n, D, stats, decay, lr_inout, partial, dtheta_out, st);
}
}  // namespace

extern "C" int ppx_es_update_sharded(double* theta, const float* noise, const int64_t* offsets, const double* rewards, int P, int p_lo,
                                     int p_n, int D, double sigma, double novelty_param, double novelty, const double* novelty_dev,
                                     int use_novelty, double decay, double* lr_inout, int* status_out, void* workspace,
                                     double* dtheta_local, const void* const* peer_dtheta_host, void* const* peer_flags_host, int W,
                                     int rank, uint32_t* seq_dev, uint32_t* status_dev, void* stream) {
  PPX_REQUIRE(theta && noise && rewards && lr_inout && workspace && dtheta_local, "es_update_sharded: null pointer");
  PPX_REQUIRE(P >= 2 && D >= 1 && sigma != 0.0 && p_lo >= 0 && p_n >= 1 && p_lo + p_n <= P, "es_update_sharded: P=%d p_lo=%d p_n=%d D=%d", P, p_lo, p_n, D);
  p2p::Peers PP;
  int rc = p2p::fill(&PP, peer_dtheta_host, peer_flags_host, W, rank, seq_dev, status_dev);
  if (rc) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  rc = es_update_core(theta, noise, offsets, rewards, P, p_lo, p_n, D, sigma, novelty_param, novelty, novelty_dev, use_novelty, decay,
                      lr_inout, status_out, workspace, dtheta_local, st);
  if (rc) return rc;
  es_apply_p2p_kernel<<<1, 1024, 0, st>>>(PP, theta, D, (const double*)workspace, decay, lr_inout);
  return after_launch("es_update(p2p apply)");
}

extern "C" int ppx_es_update(double* theta, const float* noise, const int64_t* offsets, const double* rewards, int P, int D,
                             double sigma, double novelty_param, double novelty, const double* novelty_dev, int use_novelty,
                             int rank_mode, double decay, double* lr_inout, int* status_out, void* workspace, void* stream) {
  PPX_REQUIRE(theta && noise && rewards && lr_inout && workspace, "es_update: null pointer");
  PPX_REQUIRE(P >= 2 && D >= 1 && sigma != 0.0, "es_update: P=%d D=%d sigma=%g", P, D, sigma);
  cudaStream_t st = (cudaStream_t)stream;
  double* stats = (double*)workspace;
  double* coef = stats + 8;
  double* centred = coef + P;
  double* partial = centred + P;
  int rc;
  if (rank_mode) {
    es_stats_kernel<<<1, 1024, 0, st>>>(rewards, P, rank_mode, stats, status_out);
    rc = after_launch("es_update(stats)");
    if (rc) return rc;
    rank_kernel<<<(unsigned)ceil_div(P, 256), 256, 0, st>>>(rewards, P, nullptr, centred);
    rc = after_launch("es_update(rank)");
    if (rc) return rc;
    es_coef_kernel<<<(unsigned)ceil_div(P, 256), 256, 0, st>>>(rewards, centred, P, stats, lr_inout, sigma, novelty_param, novelty,
                                                               novelty_dev, use_novelty, rank_mode, coef);
    rc = after_launch("es_update(coef)");
  } else {
    // z-score shaping (the reference's): stats + coefficients, then the GEMV whose last CTAs apply the update (2 launches)
    return es_update_core(theta, noise, offsets, rewards, P, 0, P, D, sigma, novelty_param, novelty, novelty_dev, use_novelty, decay,
                          lr_inout, status_out, workspace, nullptr, st);
  }
  if (rc) return rc;
  const int splits = gemv_splits(P, D);
  const int p_chunk = (int)ceil_div(P, splits);
  dim3 grid((unsigned)ceil_div(D, 512), (unsigned)splits);
  bool vec = (D % 4 == 0) && ((uintptr_t)noise % 16 == 0) && offsets == nullptr;
  // with offsets, vector loads need every offset to be a multiple of 4 -- the table sampler guarantees it
  // (see host wrapper); dense parity inputs only need D % 4 == 0.
  if (offsets) vec = (D % 4 == 0) && ((uintptr_t)noise % 16 == 0);
  if (vec) es_gemv_kernel<true><<<grid, 128, 0, st>>>(noise, offsets, coef, P, D, p_chunk, partial);
  else es_gemv_kernel<false><<<grid, 128, 0, st>>>(noise, offsets, coef, P, D, p_chunk, partial);
  rc = after_launch("es_update(gemv)");
  if (rc) return rc;
  es_apply_kernel<<<(unsigned)ceil_div(D, 256), 256, 0, st>>>(theta, partial, splits, D, stats, decay, lr_inout);
  return after_launch("es_update(apply)");
}

extern "C" int64_t ppx_es_update_member_workspace(int P, int D) {
  return (int64_t)sizeof(double) * (8 + 3 * (int64_t)P + (int64_t)gemv_splits(P, D) * D);
}

extern "C" int ppx_es_update_member(double* theta, const float* noise, const int64_t* offsets, const double* rewards,
                                    const double* novelties, int P, int p_lo, int p_n, int D, double sigma, double novelty_param,
                                    int rank_mode, double decay, double* lr_inout, int* status_out, void* workspace,
                                    double* dtheta_local, const void* const* peer_dtheta_host, void* const* peer_flags_host, int W,
                                    int rank, uint32_t* seq_dev, uint32_t* status_dev, void* stream) {
  PPX_REQUIRE(theta && noise && rewards && novelties && lr_inout && workspace, "es_update_member: null pointer");
  PPX_REQUIRE(P >= 2 && D >= 1 && sigma != 0.0 && W >= 1 && p_lo >= 0 && p_n >= 1 && p_lo + p_n <= P,
              "es_update_member: P=%d p_lo=%d p_n=%d D=%d W=%d", P, p_lo, p_n, D, W);
  PPX_REQUIRE(W >= 2 || (p_lo == 0 && p_n == P), "es_update_member: one rank updates all P members (p_lo=%d p_n=%d)", p_lo, p_n);
  p2p::Peers PP;
  if (W >= 2) {
    PPX_REQUIRE(dtheta_local, "es_update_member: W=%d needs dtheta_local", W);
    int rc = p2p::fill(&PP, peer_dtheta_host, peer_flags_host, W, rank, seq_dev, status_dev);
    if (rc) return rc;
  }
  cudaStream_t st = (cudaStream_t)stream;
  double* stats = (double*)workspace;
  double* coef = stats + 8;
  double* cf = coef + P;
  double* cn = cf + P;
  double* partial = cn + P;
  int rc;
  if (rank_mode) {
    rank_kernel<<<(unsigned)ceil_div(P, 256), 256, 0, st>>>(rewards, P, nullptr, cf);
    rc = after_launch("es_update_member(rank fitness)");
    if (rc) return rc;
    rank_kernel<<<(unsigned)ceil_div(P, 256), 256, 0, st>>>(novelties, P, nullptr, cn);
    rc = after_launch("es_update_member(rank novelty)");
    if (rc) return rc;
    es_member_rank_coef_kernel<<<(unsigned)ceil_div(P, 256), 256, 0, st>>>(cf, cn, P, stats, status_out, lr_inout, sigma,
                                                                           novelty_param, coef);
  } else {
    es_member_stats_coef_kernel<<<1, 1024, 0, st>>>(rewards, novelties, P, stats, status_out, lr_inout, sigma, novelty_param, coef);
  }
  rc = after_launch("es_update_member(coef)");
  if (rc) return rc;
  rc = es_gemv_tail(theta, noise, offsets, coef, P, p_lo, p_n, D, stats, decay, lr_inout, partial, W >= 2 ? dtheta_local : nullptr, st);
  if (rc || W == 1) return rc;
  es_apply_p2p_kernel<<<1, 1024, 0, st>>>(PP, theta, D, stats, decay, lr_inout);
  return after_launch("es_update_member(p2p apply)");
}

extern "C" int ppx_rank_center(const double* r, int P, int64_t* rank_out, double* centred_out, void* stream) {
  PPX_REQUIRE(r && P >= 2 && (rank_out || centred_out), "rank_center: bad arguments");
  rank_kernel<<<(unsigned)ceil_div(P, 256), 256, 0, (cudaStream_t)stream>>>(r, P, rank_out, centred_out);
  return after_launch("rank_center");
}

extern "C" int ppx_knn_novelty(const double* archive, int64_t M, const double* queries, int Q, int dim, int K, double* sum_out,
                               double* novelty_out, void* stream) {
  PPX_REQUIRE(archive && queries && M >= 1 && Q >= 1 && dim >= 1, "knn_novelty: bad arguments");
  PPX_REQUIRE(K >= 1 && K <= 32, "knn_novelty: K=%d (1..32)", K);
  // archive split: enough warps to fill the machine for few queries, >= 256 points per warp
  int splits = (int)std::max<int64_t>(1, std::min<int64_t>(ceil_div(M, 256), ceil_div(8 * (int64_t)sm_count(), Q)));
  splits = std::min(splits, 1024);
  PPX_REQUIRE(Q <= 65535, "knn_novelty: Q=%d exceeds grid.y; call in slices", Q);
  static GrowOnlyScratch scratch;                      // calls are stream-ordered (one learner thread)
  const int rs = grow_scratch(scratch, (size_t)Q * splits * K * sizeof(double));
  if (rs) return rs;
  double* cand = (double*)scratch.p;
  dim3 grid((unsigned)splits, (unsigned)Q);
  if (K <= 16) {
    knn_slice_kernel<16><<<grid, 32, 0, (cudaStream_t)stream>>>(archive, M, queries, dim, K, splits, cand);
    int rc = after_launch("knn_novelty(slices)");
    if (rc) return rc;
    knn_merge_kernel<16><<<(unsigned)Q, 32, 0, (cudaStream_t)stream>>>(cand, splits * K, M, K, sum_out, novelty_out);
  } else {
    knn_slice_kernel<32><<<grid, 32, 0, (cudaStream_t)stream>>>(archive, M, queries, dim, K, splits, cand);
    int rc = after_launch("knn_novelty(slices)");
    if (rc) return rc;
    knn_merge_kernel<32><<<(unsigned)Q, 32, 0, (cudaStream_t)stream>>>(cand, splits * K, M, K, sum_out, novelty_out);
  }
  return after_launch("knn_novelty");
}

extern "C" int ppx_knn_novelty_many(const double* archive, int64_t M, const double* queries, int Q, int dim, int K, double* sum_out,
                                    double* novelty_out, void* stream) {
  PPX_REQUIRE(archive && queries && M >= 1 && Q >= 1 && (sum_out || novelty_out), "knn_novelty_many: bad arguments");
  PPX_REQUIRE(dim >= 1 && dim <= kKnnManyMaxDim, "knn_novelty_many: dim=%d (1..%d)", dim, kKnnManyMaxDim);
  PPX_REQUIRE(K >= 1 && K <= 32, "knn_novelty_many: K=%d (1..32)", K);
  const unsigned grid = (unsigned)ceil_div(Q, kKnnManyThreads);
  if (K <= 16) knn_many_kernel<16><<<grid, kKnnManyThreads, 0, (cudaStream_t)stream>>>(archive, M, queries, Q, dim, K, sum_out, novelty_out);
  else knn_many_kernel<32><<<grid, kKnnManyThreads, 0, (cudaStream_t)stream>>>(archive, M, queries, Q, dim, K, sum_out, novelty_out);
  return after_launch("knn_novelty_many");
}
