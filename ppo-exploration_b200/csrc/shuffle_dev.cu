// Fisher-Yates swaps of np.random.permutation applied ON THE DEVICE, in parallel, bit-exactly.
//
// buffer.py:239 draws one np.random.permutation(T*N) per epoch.  Its draws are inherently sequential (host_rng.cpp
// restates numpy's legacy MT19937 stream); its swaps  for i = n-1 .. 1: swap(a[i], a[j_i])  look sequential too, and
// cost 0.9 ms per 524 288 on a host core -- the one thing that does not shrink when 8 ranks share 16 cores.  They can
// be resolved in parallel:
//   * position i is final after its own step (later steps only touch positions < i), and receives the content
//     position j_i had just before step i;
//   * the content of a position p before step i is what the most recent earlier step that TARGETED p put there,
//     i.e. step s = min{ s > i : j_s = p } moved in the old content of position s -- or p itself if there is none.
// So with the steps grouped by target and each (tiny: mean 1, ~ln(n/p) for position p) group sorted by index,
//   first[p] = smallest step targeting p,  nxt[s] = next larger step with the same target,
//   V(s) = content of position s before its own step = V(first[s]) if first[s] exists else s   (a strictly increasing chain)
//   out[i] = V(nxt[i]) if nxt[i] exists else j_i          (self-swaps j_i = i and position 0:  out[i] = V(i)).
// Five small kernels over n elements (count, scan, scatter, per-group sort + links, resolve): the group order produced by
// the atomics is re-sorted, so the result does not depend on their timing.  Checked bit-exactly against numpy
// (tests/test_gpu_gather.py).
#include "common.cuh"

namespace ppx {
namespace {

constexpr int kScanBlock = 1024;       // elements per scan block (256 threads x 4)

// n < 2^31: every index, count and scan offset fits an int (the offsets sum to at most n - 1 steps).  The grid-stride
// loops count in int64_t because their last step may pass 2^31.
__global__ void __launch_bounds__(256) fy_count_kernel(const int32_t* __restrict__ j, int n, int rev, int32_t* __restrict__ cnt) {
  for (int64_t i = blockIdx.x * blockDim.x + threadIdx.x + 1; i < n; i += gridDim.x * blockDim.x) {
    const int t = j[rev ? n - 1 - i : i];
    if (t != i) atomicAdd(&cnt[t], 1);
  }
}

// exclusive scan, pass 1: per-block exclusive scan of 1024 elements + the block total
__global__ void __launch_bounds__(256) fy_scan1_kernel(const int32_t* __restrict__ in, int n, int32_t* __restrict__ out, int32_t* __restrict__ bsum) {
  __shared__ int32_t s_w[8];
  const int base = blockIdx.x * kScanBlock + threadIdx.x * 4;
  int v[4];
#pragma unroll
  for (int k = 0; k < 4; ++k) v[k] = base + k < n ? in[base + k] : 0;
  const int tsum = v[0] + v[1] + v[2] + v[3];
  int x = tsum;                                              // inclusive warp scan of the thread sums
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) { const int y = __shfl_up_sync(0xffffffffu, x, d); if (lane >= d) x += y; }
  if (lane == 31) s_w[warp] = x;
  __syncthreads();
  int woff = 0, total = 0;
#pragma unroll
  for (int w = 0; w < 8; ++w) { if (w < warp) woff += s_w[w]; total += s_w[w]; }
  int run = woff + x - tsum;
#pragma unroll
  for (int k = 0; k < 4; ++k) { if (base + k < n) out[base + k] = run; run += v[k]; }
  if (threadIdx.x == 0) bsum[blockIdx.x] = total;
}
// pass 2: one block turns the block totals into exclusive offsets (any nb: each thread scans `per` of them)
__global__ void __launch_bounds__(1024) fy_scan2_kernel(int32_t* __restrict__ bsum, int nb) {
  __shared__ int32_t s_w[32];
  const int per = (nb + 1023) / 1024, b0 = threadIdx.x * per;
  int tsum = 0;
  for (int k = 0; k < per; ++k) if (b0 + k < nb) tsum += bsum[b0 + k];
  int x = tsum;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) { const int y = __shfl_up_sync(0xffffffffu, x, d); if (lane >= d) x += y; }
  if (lane == 31) s_w[warp] = x;
  __syncthreads();
  int woff = 0;
  for (int w = 0; w < warp; ++w) woff += s_w[w];
  int run = woff + x - tsum;
  for (int k = 0; k < per; ++k)
    if (b0 + k < nb) { const int t = bsum[b0 + k]; bsum[b0 + k] = run; run += t; }
}
// pass 3 fused into the scatter: start[t] = local[t] + bsum[t / 1024]
__global__ void __launch_bounds__(256) fy_scatter_kernel(const int32_t* __restrict__ j, int n, int rev, const int32_t* __restrict__ local,
                                                         const int32_t* __restrict__ bsum, int32_t* __restrict__ cursor,
                                                         int32_t* __restrict__ grp) {
  for (int64_t i = blockIdx.x * blockDim.x + threadIdx.x + 1; i < n; i += gridDim.x * blockDim.x) {
    const int t = j[rev ? n - 1 - i : i];
    if (t != i) grp[local[t] + bsum[t / kScanBlock] + atomicAdd(&cursor[t], 1)] = (int)i;
  }
}
// one thread per target: sort its (tiny) group by step index, emit first[p] and the nxt links
__global__ void __launch_bounds__(256) fy_links_kernel(int n, const int32_t* __restrict__ cnt, const int32_t* __restrict__ local,
                                                       const int32_t* __restrict__ bsum, int32_t* __restrict__ grp,
                                                       int32_t* __restrict__ first, int32_t* __restrict__ nxt) {
  for (int64_t p = blockIdx.x * blockDim.x + threadIdx.x; p < n; p += gridDim.x * blockDim.x) {
    const int m = cnt[p];
    if (m == 0) { first[p] = -1; continue; }
    int32_t* g = grp + local[p] + bsum[p / kScanBlock];
    for (int a = 1; a < m; ++a) {                            // insertion sort (groups average one element)
      const int key = g[a];
      int b = a - 1;
      while (b >= 0 && g[b] > key) { g[b + 1] = g[b]; --b; }
      g[b + 1] = key;
    }
    first[p] = g[0];
    for (int a = 0; a + 1 < m; ++a) nxt[g[a]] = g[a + 1];
    nxt[g[m - 1]] = -1;
  }
}
// out[i]: follow the (strictly increasing) first[] chain from the step that last wrote the source position
__global__ void __launch_bounds__(256) fy_resolve_kernel(const int32_t* __restrict__ j, int n, int rev, const int32_t* __restrict__ first,
                                                         const int32_t* __restrict__ nxt, int64_t* __restrict__ out) {
  for (int64_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const int t = i ? j[rev ? n - 1 - i : i] : 0;
    int q;
    if (t == i) q = (int)i;                                 // self-swap (and position 0): the content position i ends up with
    else { q = nxt[i]; if (q < 0) { out[i] = t; continue; } }
    int f;
    while ((f = first[q]) >= 0) q = f;
    out[i] = q;
  }
}

}  // namespace
}  // namespace ppx

using namespace ppx;

extern "C" int64_t ppx_np_shuffle_apply_device_workspace(int64_t n) {
  if (n < 0 || n >= (1ll << 31)) return -1;
  const int64_t nb = ceil_div(std::max<int64_t>(n, 1), kScanBlock);
  return (int64_t)sizeof(int32_t) * (6 * std::max<int64_t>(n, 1) + nb + 64);
}

extern "C" int ppx_np_shuffle_apply_device(const int32_t* j_dev, int64_t n, int acceptance_order, void* workspace, int64_t* out_dev,
                                           void* stream) {
  PPX_REQUIRE(n >= 0 && n < (1ll << 31), "np_shuffle_apply_device: n=%lld (supported below 2^31)", (long long)n);
  if (n == 0) return PPX_OK;
  PPX_REQUIRE(j_dev && workspace && out_dev, "np_shuffle_apply_device: null pointer");
  cudaStream_t st = (cudaStream_t)stream;
  const int N = (int)n, nb = (int)ceil_div(n, kScanBlock), rev = acceptance_order ? 1 : 0;
  int32_t* cnt = (int32_t*)workspace;                        // [n] steps targeting p (self-swaps excluded)
  int32_t* cursor = cnt + n;                                 // [n]
  int32_t* local = cursor + n;                               // [n] exclusive scan inside the 1024-block
  int32_t* grp = local + n;                                  // [n] steps grouped by target
  int32_t* first = grp + n;                                  // [n]
  int32_t* nxt = first + n;                                  // [n]
  int32_t* bsum = nxt + n;                                   // [nb]
  PPX_CUDA(cudaMemsetAsync(cnt, 0, sizeof(int32_t) * 2 * n, st));          // cnt + cursor
  const unsigned g = (unsigned)std::min<int64_t>(ceil_div(n, 256), (int64_t)sm_count() * 8);
  fy_count_kernel<<<g, 256, 0, st>>>(j_dev, N, rev, cnt);
  fy_scan1_kernel<<<(unsigned)nb, 256, 0, st>>>(cnt, N, local, bsum);
  fy_scan2_kernel<<<1, 1024, 0, st>>>(bsum, nb);
  fy_scatter_kernel<<<g, 256, 0, st>>>(j_dev, N, rev, local, bsum, cursor, grp);
  fy_links_kernel<<<g, 256, 0, st>>>(N, cnt, local, bsum, grp, first, nxt);
  fy_resolve_kernel<<<g, 256, 0, st>>>(j_dev, N, rev, first, nxt, out_dev);
  return after_launch("np_shuffle_apply_device", 6);
}

// One call for a whole staging step of a permutation (made from the host thread that drew it): H2D of the pinned partner
// list, the swaps above, and the two event records the consumer needs -- `copied` (the pinned list may be re-used) and
// `ready` (out_dev holds the permutation).  Selects the device that owns j_dev for the calling thread first, so a
// worker thread of a rank > 0 needs no device bookkeeping of its own.
extern "C" int ppx_np_shuffle_stage(const int32_t* j_host_pinned, int64_t n, int32_t* j_dev, void* workspace, int64_t* out_dev,
                                    void* stream, void* copied_event, void* ready_event) {
  PPX_REQUIRE(n >= 1 && n < (1ll << 31), "np_shuffle_stage: n=%lld (supported: 1 .. 2^31 - 1)", (long long)n);
  PPX_REQUIRE(j_host_pinned && j_dev && workspace && out_dev, "np_shuffle_stage: null pointer");
  cudaPointerAttributes at;
  PPX_CUDA(cudaPointerGetAttributes(&at, j_dev));
  PPX_REQUIRE(at.type == cudaMemoryTypeDevice, "np_shuffle_stage: j_dev is not device memory");
  PPX_CUDA(cudaSetDevice(at.device));
  cudaStream_t st = (cudaStream_t)stream;
  PPX_CUDA(cudaMemcpyAsync(j_dev, j_host_pinned, sizeof(int32_t) * (size_t)n, cudaMemcpyHostToDevice, st));
  if (copied_event) PPX_CUDA(cudaEventRecord((cudaEvent_t)copied_event, st));
  const int rc = ppx_np_shuffle_apply_device(j_dev, n, 1, workspace, out_dev, stream);
  if (rc != PPX_OK) return rc;
  if (ready_event) PPX_CUDA(cudaEventRecord((cudaEvent_t)ready_event, st));
  return PPX_OK;
}
