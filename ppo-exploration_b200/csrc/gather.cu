// Minibatch shuffle-gather and advantage statistics.
//
// Replaces RolloutStorage.get/_get_samples (buffer.py:233-267, :365-394).  The reference first
// rewrites every array into the env-major flat layout (swap_and_flatten, buffer.py:40-52) and then
// fancy-indexes it; here the [T,N,...] arrays stay where they are and the flat index is decoded on
// the fly: flat i -> (t, n) = (i % T, i / T).  One launch gathers every field of the RolloutSample.
// Algorithmic traffic: 2 x row bytes per sample + the 8-byte index (SURVEY §8d).
#include "common.cuh"
#include "p2p.cuh"

namespace ppx {
namespace {

struct GatherArgs {
  const char* src[PPX_MAX_GATHER];
  char* dst[PPX_MAX_GATHER];
  int row_bytes[PPX_MAX_GATHER];
  int vec16[PPX_MAX_GATHER];
  // optional: {mean, unbiased std} of up to two gathered f32 [B] fields (the advantages, algorithms.py:219 / :431-434),
  // computed on the way so the minibatch needs no separate moments launch
  int stat_field[2];
  int order[PPX_MAX_GATHER];     // blockIdx.y (after the row-per-thread slice) -> field
  unsigned small_mask;           // fields with rows <= 32 bytes: ONE thread gathers all of them for a row (slice blockIdx.y == 0)
  int small_idx[8], n_small;     // the same fields as a list (at most kSmallMax)
  double* stat_out[2];
  double* stat_part;             // [2][kStatMax][2]
  unsigned int* stat_ticket;     // [2]
  int n_shard;                   // > 0: sources are all-gathered env shards [N / n_shard][T][n_shard][...]
  int64_t stat_lo, stat_n;       // statistics over idx[stat_lo .. stat_lo + stat_n)
  const int64_t* row_dev;        // optional step cursor
  int64_t n_mb, epoch_stride, mb_stride;
  // per-rank shuffles of a sharded learner (W >= 2): the finalising block merges the W ranks' moment records over peer memory
  int W, rank;
  uint64_t* xm[p2p::MAXW];       // rank r's staging [2 statistics slots][2 parities][W source ranks][8 words of {u32, u32 seq}]
  uint32_t* seq_dev;             // [2]: one sequence number per statistics slot
  uint32_t* status_dev;
};
constexpr int kStatMax = 4096;
constexpr int kSmallMax = 8;

// flat index of the (global) env-major flatten (buffer.py:49-52) -> storage row.  T*N < 2^31 (checked on the host): the
// index arithmetic is 32-bit -- a 64-bit division costs ~70 instructions, and this decode runs once per gathered word.
__device__ __forceinline__ int64_t row_of(int64_t i, int T, int N, int n_shard) {
  const uint32_t u = (uint32_t)i, n = u / (uint32_t)T, t = u - n * (uint32_t)T;
  if (n_shard <= 0) return (int64_t)(t * (uint32_t)N + n);
  const uint32_t r = n / (uint32_t)n_shard;
  return (int64_t)((r * (uint32_t)T + t) * (uint32_t)n_shard + (n - r * (uint32_t)n_shard));
}
// this launch's index slice (step cursor: one CUDA graph serves every minibatch of a train() call)
__device__ __forceinline__ const int64_t* idx_of(const GatherArgs& a, const int64_t* idx) {
  if (!a.row_dev) return idx;
  const int64_t row = *a.row_dev;
  return idx + (row / a.n_mb) * a.epoch_stride + (row % a.n_mb) * a.mb_stride;
}

template <typename V>
__device__ __forceinline__ void gather_rows(const char* __restrict__ src, char* __restrict__ dst, int row_bytes,
                                            const int64_t* __restrict__ idx, int64_t B, int T, int N, int n_shard) {
  const int words = row_bytes / (int)sizeof(V);
  const int64_t total = B * words;
  for (int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; g < total; g += (int64_t)gridDim.x * blockDim.x) {
    const int64_t b = g / words;
    const int w = (int)(g - b * words);
    const int64_t row = row_of(__ldg(idx + b), T, N, n_shard);
    reinterpret_cast<V*>(dst)[g] = __ldg(reinterpret_cast<const V*>(src + row * row_bytes) + w);
  }
}

// Block partials of one statistics slot -> {mean, unbiased std}: every block of the slice publishes (sum, sum of squares),
// the last one to arrive adds them in a fixed order and -- sharded with per-rank shuffles -- merges the ranks' records.
// All threads of the block call this; n_stat = rows the statistics cover on this rank.
__device__ void finish_stats(const GatherArgs& args, int slot, double s, double q, int64_t n_stat) {
  __shared__ double s_red[32];
  __shared__ bool s_last;
  s = block_sum(s, s_red);
  q = block_sum(q, s_red);
  double* part = args.stat_part + (size_t)slot * kStatMax * 2;
  if (threadIdx.x == 0) { part[2 * blockIdx.x] = s; part[2 * blockIdx.x + 1] = q; }
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) {
    const unsigned int t = atomicAdd(args.stat_ticket + slot, 1u);
    s_last = (t == gridDim.x - 1);
    if (s_last) args.stat_ticket[slot] = 0u;
  }
  __syncthreads();
  if (!s_last) return;
  __threadfence();
  s = 0.0; q = 0.0;
  for (int k = threadIdx.x; k < (int)gridDim.x; k += blockDim.x) { s += __ldcg(part + 2 * k); q += __ldcg(part + 2 * k + 1); }
  s = block_sum(s, s_red);
  q = block_sum(q, s_red);
  if (threadIdx.x >= 32) return;
  double mean = s / (double)n_stat;
  double M2 = fmax(q - s * mean, 0.0);
  double n_tot = (double)n_stat;
  if (args.W >= 2) {
    // Every rank shuffled its own rollout: the statistics of the GLOBAL minibatch are the merge of the W local records
    // {n, mean, M2} (Chan et al.), in rank order so that every rank gets the same bits.  Exchange = value + sequence
    // number in one 8-byte store per 32-bit half, pushed to every rank; then poll the own slots (no fence, no separate
    // kernel; same protocol as the loss sums and the gradient, ppo_loss.cu / mlp_fused.cu).
    const int lane = threadIdx.x, W = args.W;
    const uint32_t seq = args.seq_dev[slot] + 1u;
    const size_t base = ((size_t)slot * 2 + (seq & 1u)) * W * 8;
    if (lane < 6) {                                           // lane / 2 = which double, lane & 1 = which half
      const double v = lane < 2 ? n_tot : (lane < 4 ? mean : M2);
      const uint64_t bits = (uint64_t)__double_as_longlong(v);
      const uint32_t half = (lane & 1) ? (uint32_t)(bits >> 32) : (uint32_t)bits;
      for (int r = 0; r < W; ++r)
        asm volatile("st.relaxed.sys.global.v2.u32 [%0], {%1, %2};" ::"l"(args.xm[r] + base + (size_t)args.rank * 8 + lane), "r"(half), "r"(seq) : "memory");
    }
    double nr = 0.0, mr = 0.0, m2r = 0.0;                      // lane r < W holds rank r's record
    if (lane < W) {
      const uint64_t* src = args.xm[args.rank] + base + (size_t)lane * 8;
      uint32_t w[6];
      const uint64_t t0 = p2p::now_ns();
      for (int k = 0; k < 6; ++k) {
        uint32_t v, t;
        for (;;) {
          asm volatile("ld.volatile.global.v2.u32 {%0, %1}, [%2];" : "=r"(v), "=r"(t) : "l"(src + k) : "memory");
          if (t == seq) break;
          if (p2p::now_ns() - t0 > 4000000000ull) { atomicExch(args.status_dev, 1u); break; }
        }
        w[k] = v;
      }
      nr = __longlong_as_double((long long)(((uint64_t)w[1] << 32) | w[0]));
      mr = __longlong_as_double((long long)(((uint64_t)w[3] << 32) | w[2]));
      m2r = __longlong_as_double((long long)(((uint64_t)w[5] << 32) | w[4]));
    }
    double tot = 0.0, wsum = 0.0;
    for (int r = 0; r < W; ++r) {
      const double a = __shfl_sync(0xffffffffu, nr, r), b = __shfl_sync(0xffffffffu, mr, r);
      tot += a;
      wsum += a * b;
    }
    mean = wsum / tot;
    M2 = 0.0;
    for (int r = 0; r < W; ++r) {
      const double a = __shfl_sync(0xffffffffu, nr, r), b = __shfl_sync(0xffffffffu, mr, r), c = __shfl_sync(0xffffffffu, m2r, r);
      const double d = b - mean;
      M2 += c + a * d * d;
    }
    n_tot = tot;
    if (lane == 0) args.seq_dev[slot] = seq;
  }
  if (threadIdx.x == 0) {
    args.stat_out[slot][0] = mean;
    args.stat_out[slot][1] = sqrt(M2 / (n_tot - 1.0));       // unbiased, like torch.Tensor.std()
  }
}

// one f32 per row + running (sum, sum of squares) in f64; the last CTA of the field finishes the moments in a fixed order
__device__ void gather_scalar_with_stats(const GatherArgs& args, int a, int slot, const int64_t* __restrict__ idx, int64_t B,
                                         int T, int N) {
  const float* src = reinterpret_cast<const float*>(args.src[a]);
  float* dst = reinterpret_cast<float*>(args.dst[a]);
  double s = 0.0, q = 0.0;
  const int64_t lo = args.stat_n > 0 ? args.stat_lo : 0, n_stat = args.stat_n > 0 ? args.stat_n : B;
  for (int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; k < n_stat; k += (int64_t)gridDim.x * blockDim.x) {
    const int64_t b = lo + k;
    const float v = __ldg(src + row_of(__ldg(idx + b), T, N, args.n_shard));
    if (b >= 0 && b < B) dst[b] = v;
    s += (double)v;
    q += (double)v * (double)v;
  }
  if (args.stat_n > 0) {                                      // rows of the slice the statistics range does not cover
    for (int64_t b = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; b < B; b += (int64_t)gridDim.x * blockDim.x)
      if (b < lo || b >= lo + n_stat) dst[b] = __ldg(src + row_of(__ldg(idx + b), T, N, args.n_shard));
  }
  finish_stats(args, slot, s, q, n_stat);
}

// Narrow fields (rows of <= 32 bytes: at C2 every field of the RolloutSample): one thread per ROW reads the index once,
// decodes it once and has the loads of all fields in flight together (7 independent loads at C2) before it stores;
// the field-per-slice scheme below pays the index load, the decode and a dependent load per 4..16 bytes moved.
__device__ void gather_small_rows(const GatherArgs& args, const int64_t* __restrict__ idx, int64_t B, int T, int N) {
  double s0 = 0.0, q0 = 0.0, s1 = 0.0, q1 = 0.0;
  const bool st0 = args.stat_field[0] >= 0 && ((args.small_mask >> args.stat_field[0]) & 1u);
  const bool st1 = args.stat_field[1] >= 0 && ((args.small_mask >> args.stat_field[1]) & 1u);
  for (int64_t b = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; b < B; b += (int64_t)gridDim.x * blockDim.x) {
    const int64_t row = row_of(__ldg(idx + b), T, N, args.n_shard);
#pragma unroll
    for (int k0 = 0; k0 < kSmallMax; k0 += 4) {                // four fields' loads in flight, then their stores (32 registers)
      if (k0 >= args.n_small) break;
      int r[4][8];
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        if (k0 + k >= args.n_small) continue;
        const int f = args.small_idx[k0 + k], rb = args.row_bytes[f];
        const char* sp = args.src[f] + row * rb;
        if (args.vec16[f]) {
          const int4 v = __ldg(reinterpret_cast<const int4*>(sp));
          r[k][0] = v.x; r[k][1] = v.y; r[k][2] = v.z; r[k][3] = v.w;
          if (rb > 16) {
            const int4 u = __ldg(reinterpret_cast<const int4*>(sp) + 1);
            r[k][4] = u.x; r[k][5] = u.y; r[k][6] = u.z; r[k][7] = u.w;
          }
        } else {
#pragma unroll
          for (int w = 0; w < 8; ++w)
            if (4 * w < rb) r[k][w] = __ldg(reinterpret_cast<const int*>(sp) + w);
        }
      }
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        if (k0 + k >= args.n_small) continue;
        const int f = args.small_idx[k0 + k], rb = args.row_bytes[f];
        char* dp = args.dst[f] + b * rb;
        if (args.vec16[f]) {
          *reinterpret_cast<int4*>(dp) = make_int4(r[k][0], r[k][1], r[k][2], r[k][3]);
          if (rb > 16) *(reinterpret_cast<int4*>(dp) + 1) = make_int4(r[k][4], r[k][5], r[k][6], r[k][7]);
        } else {
#pragma unroll
          for (int w = 0; w < 8; ++w)
            if (4 * w < rb) reinterpret_cast<int*>(dp)[w] = r[k][w];
        }
        if (st0 && f == args.stat_field[0]) { const double v = (double)__int_as_float(r[k][0]); s0 += v; q0 += v * v; }
        if (st1 && f == args.stat_field[1]) { const double v = (double)__int_as_float(r[k][0]); s1 += v; q1 += v * v; }
      }
    }
  }
  if (st0) finish_stats(args, 0, s0, q0, B);
  if (st1) finish_stats(args, 1, s1, q1, B);
}

__global__ void __launch_bounds__(256, 4)
gather_kernel(GatherArgs args, const int64_t* __restrict__ idx_base, int64_t B, int T, int N) {
  const int64_t* idx = idx_of(args, idx_base);
  int y = blockIdx.y;
  if (args.small_mask) {
    if (y == 0) { gather_small_rows(args, idx, B, T, N); return; }
    --y;
  }
  const int a = args.order[y];                                // statistics fields first: their tail overlaps the other fields' rows
  if (a == args.stat_field[0]) { gather_scalar_with_stats(args, a, 0, idx, B, T, N); return; }
  if (a == args.stat_field[1]) { gather_scalar_with_stats(args, a, 1, idx, B, T, N); return; }
  if (args.vec16[a]) gather_rows<int4>(args.src[a], args.dst[a], args.row_bytes[a], idx, B, T, N, args.n_shard);
  else gather_rows<int>(args.src[a], args.dst[a], args.row_bytes[a], idx, B, T, N, args.n_shard);
}

constexpr int kStatBlocks = 256;
__device__ unsigned int g_stat_ticket = 0;
// mean / unbiased std in ONE launch: per-CTA f64 (sum, sum of squares) partials; the last CTA to finish combines
// them in a fixed order (deterministic).  sum x^2 - sum x * mean cancels a factor 1 + mean^2 / var, so the std is
// good to ~1e-14 for centred data and ~1e-12 relative at |mean| ~ 1e2 std (~1e-10 at 1e3 std).
__global__ void __launch_bounds__(256) moments_kernel(const float* __restrict__ x, int64_t n, double* __restrict__ part, double* __restrict__ out) {
  __shared__ double s_red[32];
  double s = 0.0, q = 0.0;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const double v = (double)x[i];
    s += v;
    q += v * v;
  }
  s = block_sum(s, s_red);
  q = block_sum(q, s_red);
  if (threadIdx.x == 0) { part[2 * blockIdx.x] = s; part[2 * blockIdx.x + 1] = q; }
  if (!last_block_done(&g_stat_ticket)) return;
  const int nb = gridDim.x;
  s = 0.0; q = 0.0;
  if ((int)threadIdx.x < nb) { s = __ldcg(part + 2 * threadIdx.x); q = __ldcg(part + 2 * threadIdx.x + 1); }
  s = block_sum(s, s_red);
  q = block_sum(q, s_red);
  if (threadIdx.x == 0) {
    const double mean = s / (double)n;
    out[0] = mean;
    out[1] = sqrt(fmax(q - s * mean, 0.0) / (double)(n - 1));          // unbiased, like torch.Tensor.std()
  }
}

// sharded minibatches: {mean, std(ddof 1)} of n local samples -> {n, mean, M2}; and the merge of W such records
// (in rank order, Chan's parallel-variance formula) back to the {mean, std} of the global minibatch
__global__ void moments_pack_kernel(const double* __restrict__ stats, double n, double* __restrict__ rec) {
  if (threadIdx.x == 0) { rec[0] = n; rec[1] = stats[0]; rec[2] = stats[1] * stats[1] * (n - 1.0); }
}
__global__ void moments_merge_kernel(const double* __restrict__ recs, int W, double* __restrict__ out) {
  if (threadIdx.x != 0) return;
  double tot = 0.0, wsum = 0.0;
  for (int r = 0; r < W; ++r) { tot += recs[3 * r]; wsum += recs[3 * r] * recs[3 * r + 1]; }
  const double mean = wsum / tot;
  double M2 = 0.0;
  for (int r = 0; r < W; ++r) { const double d = recs[3 * r + 1] - mean; M2 += recs[3 * r + 2] + recs[3 * r] * d * d; }
  out[0] = mean;
  out[1] = sqrt(M2 / (tot - 1.0));
}

}  // namespace
}  // namespace ppx

extern "C" int ppx_moments_pack(const double* stats2, int64_t n, double* rec3, void* stream) {
  PPX_REQUIRE(stats2 && rec3 && n >= 1, "moments_pack: bad arguments");
  ppx::moments_pack_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(stats2, (double)n, rec3);
  return ppx::after_launch("moments_pack");
}
extern "C" int ppx_moments_merge(const double* recs, int W, double* out2, void* stream) {
  PPX_REQUIRE(recs && out2 && W >= 1, "moments_merge: bad arguments");
  ppx::moments_merge_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(recs, W, out2);
  return ppx::after_launch("moments_merge");
}

namespace {
int gather_impl(const void* const* srcs_host, void* const* dsts_host, const int* row_bytes_host, int n_arrays, const int64_t* idx,
                int64_t B, int T, int N, const int* stat_fields, double* const* stat_outs, int n_stats, const ppx_gather_opts* opts,
                void* stream) {
  PPX_REQUIRE(srcs_host && dsts_host && row_bytes_host && idx, "gather_minibatch: null pointer");
  PPX_REQUIRE(n_arrays >= 1 && n_arrays <= PPX_MAX_GATHER, "gather_minibatch: n_arrays=%d (1..%d)", n_arrays, PPX_MAX_GATHER);
  PPX_REQUIRE(B >= 0 && T > 0 && N > 0 && (int64_t)T * N < (1ll << 31), "gather_minibatch: B=%lld T=%d N=%d", (long long)B, T, N);
  PPX_REQUIRE(n_stats >= 0 && n_stats <= 2, "gather_minibatch: at most two statistics fields");
  if (B == 0) return PPX_OK;
  ppx::GatherArgs args;
  int64_t max_words = 0;
  for (int a = 0; a < n_arrays; ++a) {
    PPX_REQUIRE(srcs_host[a] && dsts_host[a], "gather_minibatch: array %d null", a);
    PPX_REQUIRE(row_bytes_host[a] > 0 && row_bytes_host[a] % 4 == 0, "gather_minibatch: row_bytes[%d]=%d must be a positive multiple of 4", a, row_bytes_host[a]);
    args.src[a] = (const char*)srcs_host[a];
    args.dst[a] = (char*)dsts_host[a];
    args.row_bytes[a] = row_bytes_host[a];
    args.vec16[a] = (row_bytes_host[a] % 16 == 0) && ((uintptr_t)srcs_host[a] % 16 == 0) && ((uintptr_t)dsts_host[a] % 16 == 0);
    const int64_t words = B * (row_bytes_host[a] / (args.vec16[a] ? 16 : 4));
    if (words > max_words) max_words = words;
  }
  args.stat_field[0] = args.stat_field[1] = -1;
  args.stat_out[0] = args.stat_out[1] = nullptr;
  args.stat_part = nullptr; args.stat_ticket = nullptr;
  args.n_shard = 0; args.stat_lo = 0; args.stat_n = 0; args.row_dev = nullptr; args.n_mb = 1; args.epoch_stride = 0; args.mb_stride = 0;
  args.W = 0; args.rank = 0; args.seq_dev = nullptr; args.status_dev = nullptr;
  if (opts) {
    PPX_REQUIRE(opts->n_shard >= 0 && (opts->n_shard == 0 || N % opts->n_shard == 0), "gather_minibatch: n_shard=%d does not divide N=%d", opts->n_shard, N);
    PPX_REQUIRE(opts->stat_n >= 0 && (opts->stat_n == 0 || opts->stat_n >= 2), "gather_minibatch: stat_n=%lld", (long long)opts->stat_n);
    PPX_REQUIRE(!opts->row_dev || opts->n_mb >= 1, "gather_minibatch: cursor needs n_mb >= 1");
    args.n_shard = opts->n_shard; args.stat_lo = opts->stat_lo; args.stat_n = opts->stat_n;
    args.row_dev = opts->row_dev; args.n_mb = opts->n_mb; args.epoch_stride = opts->epoch_stride; args.mb_stride = opts->mb_stride;
    if (opts->stat_n > max_words) max_words = opts->stat_n;
    if (opts->W >= 2 && n_stats > 0) {
      PPX_REQUIRE(opts->W <= ppx::p2p::MAXW && opts->rank >= 0 && opts->rank < opts->W && opts->peer_moments_host && opts->seq_dev &&
                  opts->status_dev, "gather_minibatch: bad peer arguments (W=%d rank=%d)", opts->W, opts->rank);
      args.W = opts->W; args.rank = opts->rank; args.seq_dev = opts->seq_dev; args.status_dev = opts->status_dev;
      for (int q = 0; q < opts->W; ++q) {
        PPX_REQUIRE(opts->peer_moments_host[q], "gather_minibatch: null peer pointer for rank %d", q);
        args.xm[q] = (uint64_t*)opts->peer_moments_host[q];
      }
    }
  }
  int64_t gx = ppx::ceil_div(max_words, 256);
  const int64_t cap = (int64_t)ppx::sm_count() * 16;
  if (gx > cap) gx = cap;
  if (n_stats > 0) {
    static double* part = nullptr;                       // per-process scratch; calls are stream-ordered (one learner thread)
    static unsigned int* ticket = nullptr;
    if (!part) {
      PPX_CUDA(cudaMalloc((void**)&part, 2 * ppx::kStatMax * 2 * sizeof(double)));
      PPX_CUDA(cudaMalloc((void**)&ticket, 2 * sizeof(unsigned int)));
      PPX_CUDA(cudaMemset(ticket, 0, 2 * sizeof(unsigned int)));
    }
    PPX_REQUIRE(B >= 2 || (opts && opts->stat_n >= 2), "gather_minibatch: statistics need B >= 2");
    for (int k = 0; k < n_stats; ++k) {
      PPX_REQUIRE(stat_fields && stat_outs && stat_fields[k] >= 0 && stat_fields[k] < n_arrays && stat_outs[k] &&
                  row_bytes_host[stat_fields[k]] == 4, "gather_minibatch: statistics field %d must be an f32 [B] field", k);
      args.stat_field[k] = stat_fields[k];
      args.stat_out[k] = stat_outs[k];
    }
    args.stat_part = part; args.stat_ticket = ticket;
    if (gx > ppx::kStatMax) gx = ppx::kStatMax;
  }
  // narrow fields go to the row-per-thread slice (statistics fields too, unless their range differs from the gathered
  // rows: the "global" shard mode takes the moments over the whole global minibatch)
  args.small_mask = 0u;
  int n_small = 0;
  for (int a = 0; a < n_arrays; ++a) {
    const bool is_stat = a == args.stat_field[0] || a == args.stat_field[1];
    if (row_bytes_host[a] <= 32 && !(is_stat && args.stat_n > 0) && n_small < ppx::kSmallMax) {
      args.small_mask |= 1u << a;
      args.small_idx[n_small++] = a;
    }
  }
  if (n_small < 2) { args.small_mask = 0u; n_small = 0; }
  args.n_small = n_small;
  int n_slices = 0;
  for (int q = 0; q < 2; ++q)
    if (args.stat_field[q] >= 0 && !((args.small_mask >> args.stat_field[q]) & 1u)) args.order[n_slices++] = args.stat_field[q];
  for (int a = 0; a < n_arrays; ++a)
    if (a != args.stat_field[0] && a != args.stat_field[1] && !((args.small_mask >> a) & 1u)) args.order[n_slices++] = a;
  if (n_small) {
    int64_t big_words = 0;                                    // the slices share gridDim.x: size it for the rows and the wide fields
    for (int k = 0; k < n_slices; ++k) {
      const int a = args.order[k];
      big_words = std::max<int64_t>(big_words, B * (row_bytes_host[a] / (args.vec16[a] ? 16 : 4)));
    }
    if (opts && opts->stat_n > big_words) big_words = opts->stat_n;
    gx = std::min<int64_t>(std::max<int64_t>(ppx::ceil_div(std::max<int64_t>(B, big_words), 256), 1), cap);
    if (n_stats > 0 && gx > ppx::kStatMax) gx = ppx::kStatMax;
  }
  dim3 grid((unsigned)gx, (unsigned)(n_slices + (n_small ? 1 : 0)));
  ppx::gather_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(args, idx, B, T, N);
  return ppx::after_launch("gather_minibatch");
}
}  // namespace

extern "C" int ppx_gather_minibatch(const void* const* srcs_host, void* const* dsts_host, const int* row_bytes_host,
                                    int n_arrays, const int64_t* idx, int64_t B, int T, int N, void* stream) {
  return gather_impl(srcs_host, dsts_host, row_bytes_host, n_arrays, idx, B, T, N, nullptr, nullptr, 0, nullptr, stream);
}

extern "C" int ppx_gather_minibatch_stats(const void* const* srcs_host, void* const* dsts_host, const int* row_bytes_host,
                                          int n_arrays, const int64_t* idx, int64_t B, int T, int N, const int* stat_fields_host,
                                          double* const* stat_outs_host, int n_stats, const ppx_gather_opts* opts_host, void* stream) {
  return gather_impl(srcs_host, dsts_host, row_bytes_host, n_arrays, idx, B, T, N, stat_fields_host, stat_outs_host, n_stats, opts_host, stream);
}

extern "C" int ppx_mean_std(const float* x, int64_t n, double* out2, void* stream) {
  PPX_REQUIRE(x && out2 && n >= 1, "mean_std: bad arguments");
  static double* part = nullptr;                       // per-process scratch; calls are stream-ordered (one learner thread)
  if (!part) PPX_CUDA(cudaMalloc((void**)&part, 2 * ppx::kStatBlocks * sizeof(double)));
  const int nb = (int)std::max<int64_t>(1, std::min<int64_t>(ppx::kStatBlocks, ppx::ceil_div(n, 2048)));
  ppx::moments_kernel<<<nb, 256, 0, (cudaStream_t)stream>>>(x, n, part, out2);
  return ppx::after_launch("mean_std");
}
