// Per-member layer walk of the ES population forward (FeedForwardNetwork.predict, evolution_strategies.py:48-61), shared by
// ppx_es_forward (es.cu) and ppx_es_act (es_eval.cu): both kernels run this code on the same weights and inputs, so a member's
// logits are bit-identical whichever of the two computed them.
//
// One warp per member: theta is staged once per CTA in shared memory (`th`, f32); a layer  out = a . W  (W [in, out] row-major
// inside the flat vector, bias-free) is walked 8 inputs at a time -- lane j owns output columns j, j+32, ... so a warp reads
// 128 contiguous bytes of eps per input, all loads of a step in flight before the math.  fp32 arithmetic: hidden layers
// arctan (:57), last layer linear; column j of the last layer (width `no`) goes to `emit(j, no, logit)`.
#pragma once
#include <stdint.h>

#include "common.cuh"

namespace ppx {

constexpr int kFwdMaxLayers = 8, kFwdMaxWidth = 256;

// the layer plan of both kernels' parameter blocks: sizes[0..n_layers], D, per-layer load path
//   vec[l] = 4: 16-byte slot path, 1: scalar slot path (narrow layer), 0: generic
template <class Prm>
int es_plan(Prm& p, const float* noise, const int64_t* offsets, const int* layer_sizes, int n_layers, const char* what) {
  PPX_REQUIRE(n_layers >= 1 && n_layers <= kFwdMaxLayers, "%s: n_layers=%d", what, n_layers);
  int D = 0;
  for (int l = 0; l <= n_layers; ++l) {
    PPX_REQUIRE(layer_sizes[l] >= 1 && layer_sizes[l] <= kFwdMaxWidth, "%s: layer width %d not in [1, %d]", what, layer_sizes[l], kFwdMaxWidth);
    p.sizes[l] = layer_sizes[l];
    if (l) D += layer_sizes[l - 1] * layer_sizes[l];
  }
  p.D = D;
  p.n_layers = n_layers;
  int woff = 0;
  const bool base_ok = (((uintptr_t)noise & 15) == 0) && (offsets != nullptr || D % 4 == 0);   // table offsets are multiples of 4
  for (int l = 0; l < n_layers; ++l) {
    const int no = layer_sizes[l + 1], nq = no / 4;
    if (base_ok && no % 4 == 0 && nq <= 32 && (nq & (nq - 1)) == 0 && woff % 4 == 0) p.vec[l] = 4;
    else if (no <= 32 && (no & (no - 1)) == 0) p.vec[l] = 1;
    else p.vec[l] = 0;
    woff += layer_sizes[l] * no;
  }
  return PPX_OK;
}

#ifdef __CUDACC__
// Runs the member whose noise row is `eps` with its input already in a0[0..sizes[0]) (a0 / a1: this warp's two activation
// buffers of kFwdMaxWidth floats).  Every lane returns after a final __syncwarp.
template <class Prm, class Emit>
__device__ __forceinline__ void es_member_walk(const Prm& p, const float* eps, const float* th, float* a0, float* a1, int lane,
                                               Emit emit) {
  float* in = a0;
  float* outv = a1;
  int woff = 0;
  for (int l = 0; l < p.n_layers; ++l) {
    const int ni = p.sizes[l], no = p.sizes[l + 1];
    if (p.vec[l] == 4) {
      // 16-byte path (no = 4 nq, nq a power of two <= 32): lane = (row slot rs = lane / nq, column quad q = lane % nq), a warp
      // instruction covers 32 / nq consecutive input rows = 512 contiguous bytes; 8 steps of loads in flight before the math
      const int nq = no >> 2, rps = 32 / nq, rs = lane / nq, q = lane - rs * nq;
      float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
      for (int i0 = 0; i0 < ni; i0 += 8 * rps) {
        float4 e[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) {
          const int i = i0 + u * rps + rs;
          e[u] = i < ni ? ld_stream4(reinterpret_cast<const float4*>(eps + woff + (size_t)i * no) + q) : make_float4(0.f, 0.f, 0.f, 0.f);
        }
#pragma unroll
        for (int u = 0; u < 8; ++u) {
          const int i = i0 + u * rps + rs;
          if (i < ni) {
            const float ai = in[i];
            const float4 t = *reinterpret_cast<const float4*>(th + woff + (size_t)i * no + 4 * q);
            acc.x = fmaf(ai, fmaf(p.sigma, e[u].x, t.x), acc.x); acc.y = fmaf(ai, fmaf(p.sigma, e[u].y, t.y), acc.y);
            acc.z = fmaf(ai, fmaf(p.sigma, e[u].z, t.z), acc.z); acc.w = fmaf(ai, fmaf(p.sigma, e[u].w, t.w), acc.w);
          }
        }
      }
      for (int d = nq; d < 32; d <<= 1) {                  // combine the row slots (fixed order)
        acc.x += __shfl_xor_sync(0xffffffffu, acc.x, d); acc.y += __shfl_xor_sync(0xffffffffu, acc.y, d);
        acc.z += __shfl_xor_sync(0xffffffffu, acc.z, d); acc.w += __shfl_xor_sync(0xffffffffu, acc.w, d);
      }
      if (rs == 0) {
        const float v[4] = {acc.x, acc.y, acc.z, acc.w};
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          const int j = 4 * q + c;
          if (l + 1 < p.n_layers) outv[j] = atanf(v[c]);
          else emit(j, no, v[c]);
        }
      }
    } else if (p.vec[l] == 1) {
      // narrow layer (no a power of two <= 32, e.g. the action head): the same slot scheme with one column per lane, so the
      // whole warp streams the layer's contiguous weights instead of `no` lanes walking them row by row
      const int rps = 32 / no, rs = lane / no, j = lane - rs * no;
      float acc = 0.f;
      for (int i0 = 0; i0 < ni; i0 += 8 * rps) {
        float e[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) {
          const int i = i0 + u * rps + rs;
          e[u] = i < ni ? ld_stream(eps + woff + (size_t)i * no + j) : 0.f;
        }
#pragma unroll
        for (int u = 0; u < 8; ++u) {
          const int i = i0 + u * rps + rs;
          if (i < ni) acc = fmaf(in[i], fmaf(p.sigma, e[u], th[woff + (size_t)i * no + j]), acc);
        }
      }
      for (int d = no; d < 32; d <<= 1) acc += __shfl_xor_sync(0xffffffffu, acc, d);
      if (rs == 0) {
        if (l + 1 < p.n_layers) outv[j] = atanf(acc);
        else emit(j, no, acc);
      }
    } else
    for (int j0 = 0; j0 < no; j0 += 64) {                 // scalar path: 2 output columns per lane per sweep
      const bool l0 = j0 + lane < no, l1 = j0 + lane + 32 < no;
      float acc0 = 0.f, acc1 = 0.f;
      for (int i0 = 0; i0 < ni; i0 += 8) {
        float e0[8], e1[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) {
          const float* er = eps + woff + (size_t)(i0 + u) * no + j0 + lane;
          e0[u] = (i0 + u < ni && l0) ? ld_stream(er) : 0.f;
          e1[u] = (i0 + u < ni && l1) ? ld_stream(er + 32) : 0.f;
        }
#pragma unroll
        for (int u = 0; u < 8; ++u) {
          if (i0 + u < ni) {
            const float ai = in[i0 + u];
            const float* tr = th + woff + (size_t)(i0 + u) * no + j0 + lane;
            if (l0) acc0 = fmaf(ai, fmaf(p.sigma, e0[u], tr[0]), acc0);
            if (l1) acc1 = fmaf(ai, fmaf(p.sigma, e1[u], tr[32]), acc1);
          }
        }
      }
#pragma unroll
      for (int c = 0; c < 2; ++c) {
        const int j = j0 + lane + 32 * c;
        if (j < no) {
          float v = c ? acc1 : acc0;
          if (l + 1 < p.n_layers) outv[j] = atanf(v);
          else emit(j, no, v);
        }
      }
    }
    __syncwarp();
    woff += ni * no;
    float* t = in; in = outv; outv = t;
  }
}
#endif

}  // namespace ppx
