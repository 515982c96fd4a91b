// SimHash codes + persistent open-addressing count table with the reference's sequential semantics.
//
// Replaces RolloutStorage.sim_hash (buffer.py:188-200) and the defaultdict count_table (buffer.py:136).
//
// Semantics that must survive parallelisation: the reference walks the batch in env order,
// `count[key] += 1; reward[i] += beta/sqrt(count[key])`, so the j-th occurrence of a key inside one
// batch sees count c+j.  A bare atomicAdd gives the right final table but hands the bonuses to the
// wrong envs.  Two launches, no inter-CTA ordering:
//   A. (parallel over observations)  codes: bit b = (A[b,:] . obs[i,:] > 0), f64 dot (buffer.py:194), plus a
//      16-bit BUCKET id = hash(code) % NB.  A is staged in shared memory, two observations per thread.
//   P. (stable partition by bucket, 3 small launches)  tiles of 4096 elements sort (bucket, local index) keys in
//      shared memory and emit per-tile bucket counts; an exclusive scan over tiles / buckets turns them into
//      offsets; the tiles scatter their element indices into one list per bucket, in index order.
//   B. (one CTA per bucket)  a bucket OWNS its codes, so everything order-dependent happens inside one CTA:
//      the CTA walks its list (index order) in batches of <= 4096, and per batch
//        1. bitonic sort of (code, position) in shared memory -> rank among equal codes in index order and
//           one representative (the run tail) that knows the run length m
//        2. representatives find / claim their slot (linear probing, 64-bit atomicCAS: other buckets claim
//           other keys in the same table concurrently), read base = count[slot] and store base + m (plain
//           accesses: nobody else touches this key during the launch)
//        3. count_i = base + rank_i + 1; reward_i += beta / sqrt(count_i)  (f64, buffer.py:199)
//      Batches of one bucket run in index order inside the CTA, so skewed inputs (few distinct codes) stay
//      exact -- they only serialise.  Inputs above 2^20 observations are cut into stream-ordered launches.
// All 2^64 codes are valid keys: the all-ones code (the EMPTY sentinel) lives in a dedicated extra slot.
// Algorithmic traffic: 4D + 8 + 8 + 16 B/obs (SURVEY §8d).
#include "common.cuh"

struct ppx_count_table {
  uint64_t* keys;        // [capacity + 1]
  uint32_t* counts;      // [capacity + 1]
  uint64_t capacity;     // power of two
  uint32_t* ctrl;        // [0] ticket, [1] chunks done, [2] keys in use, [3] overflow flag
  uint64_t used_bound;   // host-side upper bound of keys in use (avoids a sync per call)
  uint64_t* scratch_codes;   // [scratch_n] codes of the launch in flight
  uint16_t* scratch_bucket;  // [scratch_n] bucket ids
  uint32_t* scratch_sorted;  // [scratch_n] per-tile sorted (bucket << 12 | local index) keys
  uint32_t* scratch_list;    // [scratch_n] element indices grouped by bucket, index order inside a bucket
  uint32_t* scratch_hist;    // [tiles * nb] per-tile bucket counts -> exclusive offsets over tiles
  uint32_t* scratch_bstart;  // [2 * nb + 2] bucket totals | bucket starts
  int64_t scratch_n;
};

namespace ppx {
namespace {

constexpr uint64_t kEmpty = ~0ull;
constexpr int CAP = 4096;         // elements per sorted batch
constexpr int CT = 1024;          // threads per bucket CTA (4 elements each)
constexpr int64_t LMAX = 1 << 20; // observations per launch
constexpr int TARGET = 1536;      // expected elements per bucket (sorted as a 2048-wide bitonic network)

__device__ __forceinline__ uint64_t mix64(uint64_t x) {     // splitmix64 finaliser
  x ^= x >> 30; x *= 0xbf58476d1ce4e5b9ull;
  x ^= x >> 27; x *= 0x94d049bb133111ebull;
  x ^= x >> 31;
  return x;
}
__device__ __forceinline__ uint32_t bucket_of(uint64_t code, uint32_t nb) {
  return (uint32_t)(((mix64(code ^ 0x9e3779b97f4a7c15ull) >> 32) * (uint64_t)nb) >> 32);
}

__device__ __forceinline__ uint64_t find_or_claim(uint64_t* keys, uint64_t cap, uint32_t* ctrl, uint64_t code) {
  if (code == kEmpty) return cap;                            // dedicated slot
  const uint64_t mask = cap - 1;
  uint64_t h = mix64(code) & mask;
  for (uint64_t probe = 0; probe < cap; ++probe) {
    unsigned long long prev = keys[h];
    if (prev == code) return h;
    if (prev == kEmpty) {
      prev = atomicCAS((unsigned long long*)&keys[h], (unsigned long long)kEmpty, (unsigned long long)code);
      if (prev == kEmpty) { atomicAdd(&ctrl[2], 1u); return h; }
      if (prev == code) return h;
    }
    h = (h + 1) & mask;
  }
  atomicExch(&ctrl[3], 1u);                                  // table full: flagged, reported by the host
  return cap;
}

__device__ __forceinline__ uint64_t code_of(const double* __restrict__ A, const float* __restrict__ x, int k, int D) {
  uint64_t code = 0;
  for (int b = 0; b < k; ++b) {
    const double* a = A + (size_t)b * D;
    double acc = 0.0;
    for (int d = 0; d < D; ++d) acc = fma(__ldg(a + d), (double)__ldg(x + d), acc);
    code |= (uint64_t)(acc > 0.0) << b;
  }
  return code;
}

// codes (+ bucket ids).  The reference's sign test is on the f64 dot product (buffer.py:194: f64 A, f32 obs promoted).
// DMAX > 0 (D <= 16): the dot products run in F32 with a rigorous error bound and fall back to the exact f64 fma chain of
// code_of only when the f32 result is too close to zero to decide the sign -- bit-identical codes at FFMA instead of DFMA
// speed (VERDICT r1 item 9).  With a_f = fl32(a) (relative error u = 2^-24) and a D-term f32 fma chain,
//   |s_f32 - s_ref| <= (D + 2) u (1 + o(1)) sum_d |a_d| |x_d| <= (D + 3) u L1(a_b) max_d |x_d|  =: bound_b * xmax,
// so |s_f32| > bound decides; the reference's own f64 rounding (D 2^-53) is far inside the margin.  A (f32) and the
// per-bit bounds are staged in shared memory; a thread owns 4 observations (registers), so one 16-byte read of A feeds
// 16 FMAs.  DMAX == 0: any D, the exact chain straight from global / L1.
template <int DMAX>
__global__ void __launch_bounds__(128)
codes_kernel(const double* __restrict__ A, const float* __restrict__ obs, int k, int D, int64_t n,
             uint64_t* __restrict__ codes, uint16_t* __restrict__ bucket, uint32_t nb) {
  if (DMAX == 0) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) {
      const uint64_t c = code_of(A, obs + i * D, k, D);
      codes[i] = c;
      if (bucket) bucket[i] = (uint16_t)bucket_of(c, nb);
    }
    return;
  }
  constexpr int DM = DMAX > 0 ? DMAX : 4, OB = 4;
  __shared__ __align__(16) float Af[64 * DM];
  __shared__ float bnd[64];
  for (int e = threadIdx.x; e < k * DM; e += blockDim.x) {
    const int b = e / DM, d = e - b * DM;
    Af[e] = d < D ? (float)A[(size_t)b * D + d] : 0.f;
  }
  for (int b = threadIdx.x; b < k; b += blockDim.x) {
    double l1 = 0.0;
    for (int d = 0; d < D; ++d) l1 += fabs(A[(size_t)b * D + d]);
    bnd[b] = (float)(l1 * (double)(D + 3) * 5.9604644775390625e-08 * 1.0001);      // (D + 3) 2^-24 L1(a_b), rounded up
  }
  __syncthreads();
  const int64_t i0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) * OB;
  if (i0 >= n) return;
  float x[OB][DM], xmax[OB];
#pragma unroll
  for (int t = 0; t < OB; ++t) {
    xmax[t] = 0.f;
#pragma unroll
    for (int d = 0; d < DM; ++d) {
      x[t][d] = (i0 + t < n && d < D) ? ld_stream(obs + (i0 + t) * D + d) : 0.f;
      xmax[t] = fmaxf(xmax[t], fabsf(x[t][d]));
    }
  }
  uint64_t c[OB] = {0, 0, 0, 0};
  for (int b = 0; b < k; ++b) {
    float s[OB] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
    for (int d = 0; d < DM; d += 4) {
      const float4 a = *reinterpret_cast<const float4*>(&Af[b * DM + d]);
#pragma unroll
      for (int t = 0; t < OB; ++t)
        s[t] = fmaf(a.w, x[t][d + 3], fmaf(a.z, x[t][d + 2], fmaf(a.y, x[t][d + 1], fmaf(a.x, x[t][d], s[t]))));
    }
    const float bb = bnd[b];
#pragma unroll
    for (int t = 0; t < OB; ++t) {
      bool bit = s[t] > 0.f;
      if (!(fabsf(s[t]) > bb * xmax[t])) {                          // too close to call in f32 (rare): the reference's own chain
        double acc = 0.0;
        for (int d = 0; d < D; ++d) acc = fma(__ldg(A + (size_t)b * D + d), (double)__ldg(obs + (i0 + t) * D + d), acc);
        bit = acc > 0.0;
      }
      c[t] |= (uint64_t)bit << b;
    }
  }
#pragma unroll
  for (int t = 0; t < OB; ++t)
    if (i0 + t < n) {
      codes[i0 + t] = c[t];
      if (bucket) bucket[i0 + t] = (uint16_t)bucket_of(c[t], nb);
    }
}

__global__ void __launch_bounds__(256) bucket_ids_kernel(const uint64_t* __restrict__ codes, int64_t n, uint16_t* __restrict__ bucket, uint32_t nb) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) bucket[i] = (uint16_t)bucket_of(codes[i], nb);
}

__device__ __forceinline__ bool key_gt(uint64_t ca, uint16_t ia, uint64_t cb, uint16_t ib) {
  return ca > cb || (ca == cb && ia > ib);
}

struct BucketSmem {
  uint64_t code[CAP];
  uint32_t elem[CAP];       // element index inside the launch, in index order (the compacted list)
  uint32_t base[CAP];
  uint16_t pos[CAP];        // position in elem[] carried through the sort
  int warp[32];
  int total;
};

// one sorted batch: elements elem[0..m) (index order) of this bucket
__device__ void process_batch(BucketSmem& S, int m, uint64_t* __restrict__ keys, uint32_t* __restrict__ counts, uint64_t cap,
                              uint32_t* ctrl, const uint64_t* __restrict__ codes, int64_t e0, double beta, void* rewards,
                              int rewards_f64, uint32_t* __restrict__ counts_out) {
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  int SZ = 64;
  while (SZ < m) SZ <<= 1;                                   // sort size: next power of two (>= 64)
  for (int j = tid; j < SZ; j += CT) {
    const bool valid = j < m;
    S.code[j] = valid ? __ldg(codes + S.elem[j]) : kEmpty;
    S.pos[j] = valid ? (uint16_t)j : (uint16_t)0xFFFF;
  }
  __syncthreads();
  // 1. bitonic sort by (code, pos); padding (kEmpty, 0xFFFF) sorts last
  for (int kk = 2; kk <= SZ; kk <<= 1) {
    for (int j = kk >> 1; j > 0; j >>= 1) {
      for (int t = tid; t < SZ / 2; t += CT) {
        const int i = ((t & ~(j - 1)) << 1) | (t & (j - 1));
        const int l = i | j;
        const bool up = (i & kk) == 0;
        const uint64_t ci = S.code[i], cl = S.code[l];
        const uint16_t ii = S.pos[i], il = S.pos[l];
        if (key_gt(ci, ii, cl, il) == up) {
          S.code[i] = cl; S.code[l] = ci;
          S.pos[i] = il; S.pos[l] = ii;
        }
      }
      __syncthreads();
    }
  }
  // run starts: inclusive max-scan of (is_head ? p : 0); thread owns positions 4*tid .. 4*tid+3
  const int p0 = 4 * tid;
  uint64_t c[4];
  bool head[4], tail[4];
  int start[4];
#pragma unroll
  for (int q = 0; q < 4; ++q) c[q] = (p0 + q < SZ) ? S.code[p0 + q] : kEmpty;
  const uint64_t cprev = (p0 > 0 && p0 - 1 < SZ) ? S.code[p0 - 1] : kEmpty;
  const uint64_t cnext = (p0 + 4 < SZ) ? S.code[p0 + 4] : kEmpty;
  int run = 0;                                               // latest head position seen by this thread (0 if none)
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    const int p = p0 + q;
    const uint64_t before = q == 0 ? cprev : c[q - 1];
    const uint64_t after = q == 3 ? cnext : c[q + 1];
    head[q] = p < m && (p == 0 || before != c[q]);
    tail[q] = p < m && (p == m - 1 || after != c[q]);
    if (head[q]) run = p;
  }
  int incl = run;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    const int o = __shfl_up_sync(0xffffffffu, incl, d);
    if (lane >= d) incl = max(incl, o);
  }
  if (lane == 31) S.warp[wid] = incl;
  __syncthreads();
  if (wid == 0) {
    int x = S.warp[lane];
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const int o = __shfl_up_sync(0xffffffffu, x, d);
      if (lane >= d) x = max(x, o);
    }
    S.warp[lane] = x;
  }
  __syncthreads();
  int before = __shfl_up_sync(0xffffffffu, incl, 1);
  if (lane == 0) before = 0;
  if (wid > 0) before = max(before, S.warp[wid - 1]);
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    if (head[q]) before = p0 + q;
    start[q] = before;
  }
  // 2. run tails: slot, base count, new count (this CTA owns the key for the whole launch)
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    if (!tail[q]) continue;
    const uint64_t slot = find_or_claim(keys, cap, ctrl, c[q]);
    const uint32_t base = __ldcg(counts + slot);
    S.base[start[q]] = base;
    __stcg(counts + slot, base + (uint32_t)(p0 + q - start[q] + 1));
  }
  __syncthreads();
  // 3. counts and bonus, scattered back to element order
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    const int p = p0 + q;
    if (p >= m) continue;
    const uint32_t cnt = S.base[start[q]] + (uint32_t)(p - start[q]) + 1u;
    const int64_t e = e0 + S.elem[S.pos[p]];
    if (counts_out) counts_out[e] = cnt;
    if (rewards) {
      const double bonus = beta / sqrt((double)cnt);
      if (rewards_f64) ((double*)rewards)[e] += bonus;
      else ((float*)rewards)[e] = (float)((double)((float*)rewards)[e] + bonus);
    }
  }
  __syncthreads();
}

constexpr int TP = 4096;          // elements per partition tile

// block-wide inclusive max-scan of one int per thread (1024 threads); `warp_buf` is 32 ints of shared memory
__device__ __forceinline__ int block_prefix_max_excl(int v, int* warp_buf) {
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  int incl = v;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    const int o = __shfl_up_sync(0xffffffffu, incl, d);
    if (lane >= d) incl = max(incl, o);
  }
  if (lane == 31) warp_buf[wid] = incl;
  __syncthreads();
  if (wid == 0) {
    int x = warp_buf[lane];
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const int o = __shfl_up_sync(0xffffffffu, x, d);
      if (lane >= d) x = max(x, o);
    }
    warp_buf[lane] = x;
  }
  __syncthreads();
  int before = __shfl_up_sync(0xffffffffu, incl, 1);
  if (lane == 0) before = 0;
  if (wid > 0) before = max(before, warp_buf[wid - 1]);
  __syncthreads();
  return before;                                              // max over all EARLIER threads (0 if none)
}

// P1: sort the tile's (bucket, local index) keys; per-tile bucket counts
__global__ void __launch_bounds__(CT)
tile_sort_kernel(const uint16_t* __restrict__ bucket, int n, uint32_t nb, uint32_t* __restrict__ sorted, uint32_t* __restrict__ hist) {
  __shared__ uint32_t s_key[TP];
  const int tid = threadIdx.x, tile = blockIdx.x, e0 = tile * TP;
  for (uint32_t b = tid; b < nb; b += CT) hist[(size_t)tile * nb + b] = 0u;
#pragma unroll
  for (int q = 0; q < TP / CT; ++q) {
    const int j = tid + q * CT;
    s_key[j] = (e0 + j < n) ? (((uint32_t)__ldg(bucket + e0 + j) << 12) | (uint32_t)j) : 0xFFFFFFFFu;
  }
  __syncthreads();
  for (int kk = 2; kk <= TP; kk <<= 1) {
    for (int j = kk >> 1; j > 0; j >>= 1) {
#pragma unroll
      for (int t = tid; t < TP / 2; t += CT) {
        const int i = ((t & ~(j - 1)) << 1) | (t & (j - 1));
        const int l = i | j;
        const bool up = (i & kk) == 0;
        const uint32_t a = s_key[i], c = s_key[l];
        if ((a > c) == up) { s_key[i] = c; s_key[l] = a; }
      }
      __syncthreads();
    }
  }
  const int nv = min(TP, n - e0);
#pragma unroll
  for (int q = 0; q < TP / CT; ++q) {
    const int p = tid + q * CT;
    const uint32_t k = s_key[p];
    sorted[(size_t)e0 + p] = k;
    if (p < nv) {
      const uint32_t b = k >> 12;
      const bool tail = (p == nv - 1) || ((s_key[p + 1] >> 12) != b);
      if (tail) {                                            // run head = lower bound of (b << 12) in the sorted keys
        int lo = 0, hi = p;
        const uint32_t key0 = b << 12;
        while (lo < hi) { const int mid = (lo + hi) >> 1; if (s_key[mid] < key0) lo = mid + 1; else hi = mid; }
        hist[(size_t)tile * nb + b] = (uint32_t)(p - lo + 1);
      }
    }
  }
}

// P2: per bucket, exclusive scan of the tile counts (in place) and the bucket total; the last CTA turns the totals
// into bucket starts.  tiles <= 256 (LMAX / TP).
__device__ unsigned int g_part_ticket = 0;
__global__ void __launch_bounds__(256)
bucket_offsets_kernel(uint32_t* __restrict__ hist, int tiles, uint32_t nb, uint32_t* __restrict__ btot /*[nb]*/,
                      uint32_t* __restrict__ bstart /*[nb+1]*/) {
  __shared__ uint32_t s_w[8];
  __shared__ uint32_t s_scan[1024];
  const uint32_t b = blockIdx.x;
  const int t = threadIdx.x, lane = t & 31, wid = t >> 5;
  const uint32_t c = t < tiles ? hist[(size_t)t * nb + b] : 0u;
  uint32_t incl = c;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    const uint32_t o = __shfl_up_sync(0xffffffffu, incl, d);
    if (lane >= d) incl += o;
  }
  if (lane == 31) s_w[wid] = incl;
  __syncthreads();
  uint32_t base = 0;
  for (int w = 0; w < wid; ++w) base += s_w[w];
  if (t < tiles) hist[(size_t)t * nb + b] = base + incl - c;
  if (t == 255) btot[b] = base + incl;
  if (!last_block_done(&g_part_ticket)) return;
  // exclusive scan of the nb totals (nb <= 1024 checked on the host), 4 per thread
  uint32_t run = 0;
  uint32_t v[4];
#pragma unroll
  for (int q = 0; q < 4; ++q) { const uint32_t i = (uint32_t)t * 4 + q; v[q] = i < nb ? __ldcg(btot + i) : 0u; run += v[q]; }
  s_scan[t] = run;
  __syncthreads();
  if (t == 0) { uint32_t acc = 0; for (int i = 0; i < 256; ++i) { const uint32_t x = s_scan[i]; s_scan[i] = acc; acc += x; } }
  __syncthreads();
  uint32_t acc = s_scan[t];
#pragma unroll
  for (int q = 0; q < 4; ++q) { const uint32_t i = (uint32_t)t * 4 + q; if (i <= nb) bstart[i] = acc; acc += v[q]; }
}

// P3: scatter the tile's element indices to their bucket lists (stable: tile order, then index order)
__global__ void __launch_bounds__(CT)
tile_scatter_kernel(const uint32_t* __restrict__ sorted, int n, uint32_t nb, const uint32_t* __restrict__ tile_off,
                    const uint32_t* __restrict__ bstart, uint32_t* __restrict__ list) {
  __shared__ int s_warp[32];
  __shared__ uint32_t s_prev[CT];
  const int tid = threadIdx.x, tile = blockIdx.x, e0 = tile * TP;
  const int nv = min(TP, n - e0);
  // thread owns 4 CONSECUTIVE sorted positions
  const int p0 = 4 * tid;
  uint32_t k[4];
#pragma unroll
  for (int q = 0; q < 4; ++q) k[q] = sorted[(size_t)e0 + p0 + q];
  s_prev[tid] = k[3];
  __syncthreads();
  const uint32_t kprev = tid > 0 ? s_prev[tid - 1] : 0xFFFFFFFFu;
  bool head[4];
  int run = 0;
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    const uint32_t before = q == 0 ? kprev : k[q - 1];
    head[q] = (p0 + q < nv) && (p0 + q == 0 || (before >> 12) != (k[q] >> 12));
    if (head[q]) run = p0 + q;
  }
  int before = block_prefix_max_excl(run, s_warp);
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    const int p = p0 + q;
    if (head[q]) before = p;
    if (p < nv) {
      const uint32_t b = k[q] >> 12;
      list[bstart[b] + tile_off[(size_t)tile * nb + b] + (uint32_t)(p - before)] = (uint32_t)e0 + (k[q] & 0xFFFu);
    }
  }
}

__global__ void __launch_bounds__(CT)
bucket_update_kernel(uint64_t* __restrict__ keys, uint32_t* __restrict__ counts, uint64_t cap, uint32_t* ctrl,
                     const uint64_t* __restrict__ codes, const uint32_t* __restrict__ list, const uint32_t* __restrict__ bstart,
                     uint32_t n_direct, int64_t e0, double beta, void* rewards, int rewards_f64,
                     uint32_t* __restrict__ counts_out, int own_W, int own_rank) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  BucketSmem& S = *reinterpret_cast<BucketSmem*>(smem_raw);
  const int tid = threadIdx.x;
  // sharded table: this rank keeps (and counts) only the codes of the buckets it owns; the bucket count is a multiple of
  // own_W, so bucket % own_W == hash(code) % own_W whatever the call size
  if (own_W > 1 && (int)(blockIdx.x % (unsigned)own_W) != own_rank) return;
  // list == nullptr: a single bucket holding elements 0..n_direct-1 (small calls skip the partition)
  const uint32_t lo = list ? bstart[blockIdx.x] : 0u, hi = list ? bstart[blockIdx.x + 1] : n_direct;
  for (uint32_t b0 = lo; b0 < hi; b0 += CAP) {               // batches of one bucket run in index order
    const int m = (int)min((uint32_t)CAP, hi - b0);
    for (int j = tid; j < m; j += CT) S.elem[j] = list ? __ldg(list + b0 + j) : b0 + (uint32_t)j;
    __syncthreads();
    process_batch(S, m, keys, counts, cap, ctrl, codes, e0, beta, rewards, rewards_f64, counts_out);
  }
}

__global__ void bonus_kernel(const uint32_t* __restrict__ counts, int64_t n, double beta, void* rewards, int f64) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const double bonus = beta / sqrt((double)counts[i]);
  if (f64) ((double*)rewards)[i] += bonus;
  else ((float*)rewards)[i] = (float)((double)((float*)rewards)[i] + bonus);
}

__global__ void dump_kernel(const uint64_t* __restrict__ keys, const uint32_t* __restrict__ counts, uint64_t cap,
                            uint64_t* keys_out, uint32_t* counts_out, uint64_t max_out, unsigned long long* n_out) {
  const uint64_t s = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (s > cap) return;
  const bool used = (s < cap) ? (keys[s] != kEmpty) : (counts[cap] > 0);
  if (!used) return;
  const unsigned long long pos = atomicAdd(n_out, 1ull);
  if (pos < max_out) {
    if (keys_out) keys_out[pos] = (s < cap) ? keys[s] : kEmpty;
    if (counts_out) counts_out[pos] = counts[s];
  }
}

__global__ void rehash_kernel(const uint64_t* __restrict__ okeys, const uint32_t* __restrict__ ocounts, uint64_t ocap,
                              uint64_t* nkeys, uint32_t* ncounts, uint64_t ncap, uint32_t* ctrl) {
  const uint64_t s = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (s > ocap) return;
  if (s == ocap) { ncounts[ncap] = ocounts[ocap]; return; }
  const uint64_t key = okeys[s];
  if (key == kEmpty) return;
  const uint64_t slot = find_or_claim(nkeys, ncap, ctrl, key);
  ncounts[slot] = ocounts[s];
}

// checkpoint restore: pair i goes to its slot (the all-ones key to the dedicated slot cap) and its count is stored with a
// CAS from 0, so a key given twice -- and a zero count, which no table entry can hold -- raises `bad` instead of merging
__global__ void load_kernel(const uint64_t* __restrict__ keys_in, const uint32_t* __restrict__ counts_in, uint64_t n,
                            uint64_t* keys, uint32_t* counts, uint64_t cap, uint32_t* ctrl, uint32_t* bad) {
  const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const uint32_t c = counts_in[i];
  if (c == 0u) { atomicOr(bad, 2u); return; }
  const uint64_t slot = find_or_claim(keys, cap, ctrl, keys_in[i]);
  if (atomicCAS(&counts[slot], 0u, c) != 0u) atomicOr(bad, 1u);
}

int alloc_arrays(uint64_t cap, uint64_t** keys, uint32_t** counts) {
  PPX_CUDA(cudaMalloc((void**)keys, (cap + 1) * sizeof(uint64_t)));
  PPX_CUDA(cudaMalloc((void**)counts, (cap + 1) * sizeof(uint32_t)));
  return PPX_OK;
}

int clear_arrays(ppx_count_table* t, cudaStream_t st) {
  PPX_CUDA(cudaMemsetAsync(t->keys, 0xFF, (t->capacity + 1) * sizeof(uint64_t), st));
  PPX_CUDA(cudaMemsetAsync(t->counts, 0, (t->capacity + 1) * sizeof(uint32_t), st));
  PPX_CUDA(cudaMemsetAsync(t->ctrl, 0, 4 * sizeof(uint32_t), st));
  t->used_bound = 0;
  return PPX_OK;
}

// Make room for `incoming` new keys: sync + read the real fill only when the host bound says we might
// pass 50 % load; grow by rehashing into a table 2x (or more) the size.
int reserve(ppx_count_table* t, int64_t incoming, cudaStream_t st) {
  if (t->used_bound + (uint64_t)incoming <= t->capacity / 2) { t->used_bound += incoming; return PPX_OK; }
  uint32_t ctrl_h[4];
  PPX_CUDA(cudaMemcpyAsync(ctrl_h, t->ctrl, sizeof(ctrl_h), cudaMemcpyDeviceToHost, st));
  PPX_CUDA(cudaStreamSynchronize(st));
  if (ctrl_h[3]) return fail(PPX_ERR_CAPACITY, "count table overflowed (capacity %llu)", (unsigned long long)t->capacity);
  t->used_bound = ctrl_h[2];
  if (t->used_bound + (uint64_t)incoming > t->capacity / 2) {
    uint64_t ncap = t->capacity;
    while (t->used_bound + (uint64_t)incoming > ncap / 2) ncap <<= 1;
    uint64_t* nkeys; uint32_t* ncounts;
    int rc = alloc_arrays(ncap, &nkeys, &ncounts);
    if (rc) return rc;
    PPX_CUDA(cudaMemsetAsync(nkeys, 0xFF, (ncap + 1) * sizeof(uint64_t), st));
    PPX_CUDA(cudaMemsetAsync(ncounts, 0, (ncap + 1) * sizeof(uint32_t), st));
    PPX_CUDA(cudaMemsetAsync(t->ctrl + 2, 0, sizeof(uint32_t), st));
    rehash_kernel<<<(unsigned)ceil_div(t->capacity + 1, 256), 256, 0, st>>>(t->keys, t->counts, t->capacity, nkeys, ncounts,
                                                                         ncap, t->ctrl);
    rc = after_launch("count_table rehash");
    if (rc) return rc;
    PPX_CUDA(cudaStreamSynchronize(st));
    cudaFree(t->keys); cudaFree(t->counts);
    t->keys = nkeys; t->counts = ncounts; t->capacity = ncap;
  }
  t->used_bound += incoming;
  return PPX_OK;
}

int ensure_scratch(ppx_count_table* t, int64_t n) {
  if (t->scratch_n >= n) return PPX_OK;
  cudaFree(t->scratch_codes); cudaFree(t->scratch_bucket); cudaFree(t->scratch_sorted); cudaFree(t->scratch_list);
  cudaFree(t->scratch_hist); cudaFree(t->scratch_bstart);
  t->scratch_codes = nullptr; t->scratch_bucket = nullptr; t->scratch_sorted = nullptr; t->scratch_list = nullptr;
  t->scratch_hist = nullptr; t->scratch_bstart = nullptr; t->scratch_n = 0;
  const int64_t tiles = ceil_div(n, TP), nbmax = std::max<int64_t>(1, ceil_div(n, TARGET));
  PPX_CUDA(cudaMalloc((void**)&t->scratch_codes, (size_t)n * sizeof(uint64_t)));
  PPX_CUDA(cudaMalloc((void**)&t->scratch_bucket, (size_t)(n + 8) * sizeof(uint16_t)));
  PPX_CUDA(cudaMalloc((void**)&t->scratch_sorted, (size_t)tiles * TP * sizeof(uint32_t)));
  PPX_CUDA(cudaMalloc((void**)&t->scratch_list, (size_t)n * sizeof(uint32_t)));
  PPX_CUDA(cudaMalloc((void**)&t->scratch_hist, (size_t)tiles * nbmax * sizeof(uint32_t)));
  PPX_CUDA(cudaMalloc((void**)&t->scratch_bstart, (size_t)(2 * nbmax + 2) * sizeof(uint32_t)));
  t->scratch_n = n;
  return PPX_OK;
}

int launch_codes(const double* A, const float* obs, int k, int D, int64_t n, uint64_t* codes, uint16_t* bucket, uint32_t nb,
                 cudaStream_t st) {
  if (D <= 8) codes_kernel<8><<<(unsigned)ceil_div(n, 512), 128, 0, st>>>(A, obs, k, D, n, codes, bucket, nb);
  else if (D <= 16) codes_kernel<16><<<(unsigned)ceil_div(n, 512), 128, 0, st>>>(A, obs, k, D, n, codes, bucket, nb);
  else codes_kernel<0><<<(unsigned)ceil_div(n, 128), 128, 0, st>>>(A, obs, k, D, n, codes, bucket, nb);
  return after_launch("simhash codes");
}

int run_update(ppx_count_table* t, const double* A, const float* obs, int k, int D, const uint64_t* codes_in, int64_t n,
               double beta, void* rewards, int rewards_f64, uint64_t* codes_out, uint32_t* counts_out, cudaStream_t st,
               int own_W = 1, int own_rank = 0) {
  if (n == 0) return PPX_OK;
  int rc = reserve(t, n, st);
  if (rc) return rc;
  rc = ensure_scratch(t, std::min<int64_t>(n, LMAX));
  if (rc) return rc;
  static bool configured = false;
  if (!configured) {
    PPX_CUDA(cudaFuncSetAttribute(bucket_update_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(BucketSmem)));
    configured = true;
  }
  for (int64_t e0 = 0; e0 < n; e0 += LMAX) {                  // stream-ordered launches keep the index order
    const int64_t nl = std::min<int64_t>(LMAX, n - e0);
    // <= 1024 buckets: one-CTA scan of the totals; a call that fits one sorted batch needs no partition at all
    uint32_t nb = nl <= CAP ? 1u : (uint32_t)std::max<int64_t>(1, std::min<int64_t>(ceil_div(nl, TARGET), 1024));
    if (own_W > 1) nb = std::max<uint32_t>((uint32_t)own_W, nb / (uint32_t)own_W * (uint32_t)own_W);   // always partitioned, W | nb
    const uint64_t* codes = codes_in ? codes_in + e0 : (codes_out ? codes_out + e0 : t->scratch_codes);
    const size_t sz = rewards_f64 ? sizeof(double) : sizeof(float);
    void* rew = rewards ? (char*)rewards + e0 * sz : nullptr;
    uint32_t* cnt = counts_out ? counts_out + e0 : nullptr;
    if (obs) {
      rc = launch_codes(A, obs + e0 * D, k, D, nl, const_cast<uint64_t*>(codes), nb > 1 ? t->scratch_bucket : nullptr, nb, st);
      if (rc) return rc;
    } else if (nb > 1) {
      bucket_ids_kernel<<<(unsigned)ceil_div(nl, 256), 256, 0, st>>>(codes, nl, t->scratch_bucket, nb);
      rc = after_launch("simhash bucket ids");
      if (rc) return rc;
    }
    if (nb == 1) {                                            // one bucket: no partition, elements in index order
      bucket_update_kernel<<<1, CT, sizeof(BucketSmem), st>>>(t->keys, t->counts, t->capacity, t->ctrl, codes, nullptr, nullptr,
                                                             (uint32_t)nl, 0, beta, rew, rewards_f64, cnt, 1, 0);
    } else {
      const int tiles = (int)ceil_div(nl, TP);
      uint32_t* btot = t->scratch_bstart;
      uint32_t* bstart = t->scratch_bstart + nb;
      tile_sort_kernel<<<tiles, CT, 0, st>>>(t->scratch_bucket, (int)nl, nb, t->scratch_sorted, t->scratch_hist);
      bucket_offsets_kernel<<<nb, 256, 0, st>>>(t->scratch_hist, tiles, nb, btot, bstart);
      tile_scatter_kernel<<<tiles, CT, 0, st>>>(t->scratch_sorted, (int)nl, nb, t->scratch_hist, bstart, t->scratch_list);
      rc = after_launch("simhash partition", 3);
      if (rc) return rc;
      bucket_update_kernel<<<nb, CT, sizeof(BucketSmem), st>>>(t->keys, t->counts, t->capacity, t->ctrl, codes, t->scratch_list,
                                                              bstart, 0u, 0, beta, rew, rewards_f64, cnt, own_W, own_rank);
    }
    rc = after_launch("simhash update");
    if (rc) return rc;
  }
  return PPX_OK;
}

}  // namespace
}  // namespace ppx

extern "C" int ppx_simhash_codes(const double* A, const float* obs, int k, int D, int64_t n, uint64_t* codes, void* stream) {
  PPX_REQUIRE(A && obs && codes, "simhash_codes: null pointer");
  PPX_REQUIRE(k >= 1 && k <= 64 && D >= 1 && n >= 0, "simhash_codes: k=%d (1..64) D=%d n=%lld", k, D, (long long)n);
  if (n == 0) return PPX_OK;
  return ppx::launch_codes(A, obs, k, D, n, codes, nullptr, 1, (cudaStream_t)stream);
}

extern "C" int ppx_count_table_create(uint64_t capacity, ppx_count_table** out) {
  PPX_REQUIRE(out, "count_table_create: null out");
  uint64_t cap = 1024;
  while (cap < capacity) cap <<= 1;
  ppx_count_table* t = new ppx_count_table();
  t->capacity = cap;
  int rc = ppx::alloc_arrays(cap, &t->keys, &t->counts);
  if (rc) { delete t; return rc; }
  if (cudaMalloc((void**)&t->ctrl, 4 * sizeof(uint32_t)) != cudaSuccess) { delete t; return ppx::fail(PPX_ERR_CUDA, "cudaMalloc ctrl"); }
  rc = ppx::clear_arrays(t, 0);
  if (rc) { delete t; return rc; }
  PPX_CUDA(cudaStreamSynchronize(0));
  *out = t;
  return PPX_OK;
}

extern "C" int ppx_count_table_destroy(ppx_count_table* t) {
  if (!t) return PPX_OK;
  cudaFree(t->keys); cudaFree(t->counts); cudaFree(t->ctrl); cudaFree(t->scratch_codes); cudaFree(t->scratch_bucket);
  cudaFree(t->scratch_sorted); cudaFree(t->scratch_list); cudaFree(t->scratch_hist); cudaFree(t->scratch_bstart);
  delete t;
  return PPX_OK;
}

extern "C" int ppx_count_table_clear(ppx_count_table* t, void* stream) {
  PPX_REQUIRE(t, "count_table_clear: null table");
  return ppx::clear_arrays(t, (cudaStream_t)stream);
}

extern "C" int ppx_count_table_update(ppx_count_table* t, const uint64_t* codes, int64_t n, uint32_t* counts_out, void* stream) {
  PPX_REQUIRE(t && codes && counts_out && n >= 0, "count_table_update: bad arguments");
  return ppx::run_update(t, nullptr, nullptr, 0, 0, codes, n, 0.0, nullptr, 0, nullptr, counts_out, (cudaStream_t)stream);
}

extern "C" int ppx_count_table_update_owned(ppx_count_table* t, const uint64_t* codes, int64_t n, uint32_t* counts_out, int W,
                                           int rank, void* stream) {
  PPX_REQUIRE(t && codes && counts_out && n >= 0 && W >= 1 && W <= 1024 && rank >= 0 && rank < W, "count_table_update_owned: bad arguments");
  if (n > 0) PPX_CUDA(cudaMemsetAsync(counts_out, 0, sizeof(uint32_t) * (size_t)n, (cudaStream_t)stream));
  return ppx::run_update(t, nullptr, nullptr, 0, 0, codes, n, 0.0, nullptr, 0, nullptr, counts_out, (cudaStream_t)stream, W, rank);
}

extern "C" int ppx_simhash_update(ppx_count_table* t, const double* A, const float* obs, int k, int D, int64_t n, double beta,
                                  void* rewards_inout, int rewards_are_f64, uint64_t* codes_out, uint32_t* counts_out,
                                  void* stream) {
  PPX_REQUIRE(t && A && obs && n >= 0, "simhash_update: bad arguments");
  PPX_REQUIRE(k >= 1 && k <= 64 && D >= 1, "simhash_update: k=%d (1..64) D=%d", k, D);
  return ppx::run_update(t, A, obs, k, D, nullptr, n, beta, rewards_inout, rewards_are_f64, codes_out, counts_out,
                         (cudaStream_t)stream);
}

extern "C" int ppx_simhash_bonus(const uint32_t* counts, int64_t n, double beta, void* rewards_inout, int rewards_are_f64,
                                 void* stream) {
  PPX_REQUIRE(counts && rewards_inout && n >= 0, "simhash_bonus: bad arguments");
  if (n == 0) return PPX_OK;
  ppx::bonus_kernel<<<(unsigned)ppx::ceil_div(n, 256), 256, 0, (cudaStream_t)stream>>>(counts, n, beta, rewards_inout,
                                                                                       rewards_are_f64);
  return ppx::after_launch("simhash_bonus");
}

extern "C" int ppx_count_table_size(ppx_count_table* t, uint64_t* n_keys_host) {
  PPX_REQUIRE(t && n_keys_host, "count_table_size: bad arguments");
  uint32_t ctrl_h[4];
  uint32_t special = 0;
  PPX_CUDA(cudaDeviceSynchronize());
  PPX_CUDA(cudaMemcpy(ctrl_h, t->ctrl, sizeof(ctrl_h), cudaMemcpyDeviceToHost));
  PPX_CUDA(cudaMemcpy(&special, t->counts + t->capacity, sizeof(uint32_t), cudaMemcpyDeviceToHost));
  if (ctrl_h[3]) return ppx::fail(PPX_ERR_CAPACITY, "count table overflowed");
  *n_keys_host = (uint64_t)ctrl_h[2] + (special > 0 ? 1 : 0);
  return PPX_OK;
}

extern "C" int ppx_count_table_dump(ppx_count_table* t, uint64_t* keys_dev, uint32_t* counts_dev, uint64_t max_out,
                                    uint64_t* n_out_host) {
  PPX_REQUIRE(t && n_out_host, "count_table_dump: bad arguments");
  unsigned long long* n_dev;
  PPX_CUDA(cudaDeviceSynchronize());
  PPX_CUDA(cudaMalloc((void**)&n_dev, sizeof(unsigned long long)));
  PPX_CUDA(cudaMemset(n_dev, 0, sizeof(unsigned long long)));
  ppx::dump_kernel<<<(unsigned)ppx::ceil_div(t->capacity + 1, 256), 256>>>(t->keys, t->counts, t->capacity, keys_dev, counts_dev,
                                                                         max_out, n_dev);
  int rc = ppx::after_launch("count_table_dump");
  unsigned long long n_h = 0;
  if (!rc && cudaMemcpy(&n_h, n_dev, sizeof(n_h), cudaMemcpyDeviceToHost) != cudaSuccess) rc = ppx::fail(PPX_ERR_CUDA, "dump memcpy");
  cudaFree(n_dev);
  *n_out_host = n_h;
  return rc;
}

extern "C" int ppx_count_table_capacity(ppx_count_table* t, uint64_t* capacity_host) {
  PPX_REQUIRE(t && capacity_host, "count_table_capacity: bad arguments");
  *capacity_host = t->capacity;
  return PPX_OK;
}

extern "C" int ppx_count_table_load(ppx_count_table* t, const uint64_t* keys_dev, const uint32_t* counts_dev, uint64_t n,
                                    void* stream) {
  PPX_REQUIRE(t && (n == 0 || (keys_dev && counts_dev)), "count_table_load: bad arguments");
  PPX_REQUIRE(n < (1ull << 31), "count_table_load: %llu keys (at most 2^31 - 1)", (unsigned long long)n);
  const cudaStream_t st = (cudaStream_t)stream;
  uint32_t ctrl_h[4], special = 0;
  PPX_CUDA(cudaMemcpyAsync(ctrl_h, t->ctrl, sizeof(ctrl_h), cudaMemcpyDeviceToHost, st));
  PPX_CUDA(cudaMemcpyAsync(&special, t->counts + t->capacity, sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
  PPX_CUDA(cudaStreamSynchronize(st));
  PPX_REQUIRE(ctrl_h[2] == 0 && special == 0 && ctrl_h[3] == 0, "count_table_load: the table is not empty (%u keys)",
              ctrl_h[2] + (special > 0 ? 1u : 0u));
  if (n == 0) return PPX_OK;
  t->used_bound = 0;
  int rc = ppx::reserve(t, (int64_t)n, st);                   // grows until n keys fit at <= 50 % load
  if (rc) return rc;
  uint32_t* bad;
  PPX_CUDA(cudaMalloc((void**)&bad, sizeof(uint32_t)));
  rc = cudaMemsetAsync(bad, 0, sizeof(uint32_t), st) == cudaSuccess ? PPX_OK : ppx::fail(PPX_ERR_CUDA, "count_table_load memset");
  if (!rc) {
    ppx::load_kernel<<<(unsigned)ppx::ceil_div(n, 256), 256, 0, st>>>(keys_dev, counts_dev, n, t->keys, t->counts, t->capacity,
                                                                    t->ctrl, bad);
    rc = ppx::after_launch("count_table_load");
  }
  uint32_t bad_h = 0;
  if (!rc && (cudaMemcpyAsync(&bad_h, bad, sizeof(bad_h), cudaMemcpyDeviceToHost, st) != cudaSuccess ||
              cudaMemcpyAsync(ctrl_h, t->ctrl, sizeof(ctrl_h), cudaMemcpyDeviceToHost, st) != cudaSuccess ||
              cudaStreamSynchronize(st) != cudaSuccess))
    rc = ppx::fail(PPX_ERR_CUDA, "count_table_load readback");
  cudaFree(bad);
  if (rc) return rc;
  if (bad_h || ctrl_h[3]) {                                   // no half-loaded table: back to empty, then report
    rc = ppx::clear_arrays(t, st);
    if (rc) return rc;
    PPX_CUDA(cudaStreamSynchronize(st));
    if (bad_h & 1u) return ppx::fail(PPX_ERR_ARG, "count_table_load: duplicate key");
    if (bad_h & 2u) return ppx::fail(PPX_ERR_ARG, "count_table_load: zero count");
    return ppx::fail(PPX_ERR_CAPACITY, "count_table_load: table overflowed");
  }
  t->used_bound = ctrl_h[2];                                  // exact: later growth checks see the keys in use
  return PPX_OK;
}
