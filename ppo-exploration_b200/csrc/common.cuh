// Shared host/device helpers for libppx (sm_100a).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdarg.h>
#include <stdio.h>
#include <algorithm>

#include "../../include/ppx.h"

namespace ppx {

int fail(int code, const char* fmt, ...);          // sets the thread-local message, returns code
void count_launch(int n = 1);                      // bumps ppx_launch_count()
int sm_count();                                    // cached cudaDevAttrMultiProcessorCount

inline int after_launch(const char* what, int n = 1) {
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return fail(PPX_ERR_CUDA, "%s: %s", what, cudaGetErrorString(e));
  count_launch(n);
  return PPX_OK;
}

inline int64_t ceil_div(int64_t a, int64_t b) { return (a + b - 1) / b; }

// Per-process device scratch of an entry point that only grows.  A CUDA graph captured by an earlier call holds the
// address of the block it saw, so a call that needs more allocates a new block and never frees the old one (at least
// doubling, so the retired blocks add up to less than the live one).  Nothing is synchronised.  A learner's warm pass
// sizes the block before it captures a graph; a block a graph holds is never freed.
struct GrowOnlyScratch {
  void* p = nullptr;
  size_t cap = 0;
};
inline int grow_scratch(GrowOnlyScratch& s, size_t bytes) {
  if (bytes <= s.cap) return PPX_OK;
  const size_t n = std::max(bytes, 2 * s.cap);
  void* q = nullptr;
  const cudaError_t e = cudaMalloc(&q, n);
  if (e != cudaSuccess) return fail(PPX_ERR_CUDA, "scratch of %zu bytes: %s", n, cudaGetErrorString(e));
  s.p = q;
  s.cap = n;
  return PPX_OK;
}

}  // namespace ppx

#define PPX_REQUIRE(cond, ...)                                    \
  do {                                                            \
    if (!(cond)) return ppx::fail(PPX_ERR_ARG, __VA_ARGS__);      \
  } while (0)

#define PPX_CUDA(expr)                                                                         \
  do {                                                                                         \
    cudaError_t e__ = (expr);                                                                  \
    if (e__ != cudaSuccess) return ppx::fail(PPX_ERR_CUDA, "%s: %s", #expr, cudaGetErrorString(e__)); \
  } while (0)

#ifdef __CUDACC__
namespace ppx {

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// Block-wide sum (any blockDim multiple of 32, <= 1024).  Result valid in every thread.
template <typename T>
__device__ __forceinline__ T block_sum(T v, T* smem32) {
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
  v = warp_sum(v);
  __syncthreads();                       // protect smem32 reuse across calls
  if (lane == 0) smem32[wid] = v;
  __syncthreads();
  T r = (lane < nw) ? smem32[lane] : T(0);
  r = warp_sum(r);
  return r;
}

// "Last block done" reduction tail: every thread of every block calls this after writing its block's partial
// results to global memory; it returns true in exactly one block -- the last to arrive -- whose threads may
// then read all partials (use __ldcg) and finish the reduction in a fixed order.  The ticket (zero before the
// first launch) is re-armed by the last block, so stream-ordered launches can share one counter.
__device__ __forceinline__ bool last_block_done(unsigned int* ticket) {
  __shared__ bool s_last;
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) {
    const unsigned int total = gridDim.x * gridDim.y * gridDim.z;
    const unsigned int t = atomicAdd(ticket, 1u);
    s_last = (t == total - 1);
    if (s_last) *ticket = 0u;
  }
  __syncthreads();
  if (s_last) __threadfence();
  return s_last;
}

// streaming (read-once) loads: keep them out of L1
__device__ __forceinline__ float ld_stream(const float* p) {
  float v;
  asm volatile("ld.global.nc.L1::no_allocate.f32 %0, [%1];" : "=f"(v) : "l"(p));
  return v;
}
__device__ __forceinline__ float4 ld_stream4(const float4* p) {
  float4 v;
  asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
               : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w)
               : "l"(p));
  return v;
}

}  // namespace ppx
#endif
