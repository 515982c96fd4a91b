// Fused forward and backward of the policy networks: G independent  D -> H -> H -> o_g  tanh MLPs over one
// minibatch (actor | critic | int_critic of models.py:137-213), exact fp32.
//
// The layer-by-layer path (linear.cu) launches ~30 kernels per minibatch and moves every activation through
// HBM several times; at the reference's widths (H = 64 / 128, D <= 32) the whole chain for a tile of 128
// samples fits in shared memory, so:
//   forward   one persistent kernel: X tile -> H1 = tanh(X W1 + b1) -> H2 = tanh(H1 W2 + b2) -> out = H2 W3 + b3;
//             H1 / H2 are written once (the backward pass needs them), outputs go to the loss head.
//   backward  one persistent kernel per tile:  dP2 = (dOut W3^T) (1-H2^2),  dW3 += H2^T dOut,
//             dW2 += H1^T dP2,  dP1 = (dP2 W2^T) (1-H1^2),  dW1 += X^T dP1  and the bias column sums; the weight
//             gradients stay in registers / shared memory across all tiles of a CTA and leave as ONE partial
//             per CTA, reduced in a fixed order by a second small kernel (deterministic, no float atomics).
// Both are FP32-FMA bound (the 1e-5 parity bound rules out one-pass tf32/bf16, and at K = 64 the hi/lo split
// of a 3xTF32 tensor-core pass costs as many instructions per element as the FMAs it saves): 8x4 (H=64) or
// 8x8 (H=128) register tiles fed by float4 shared-memory loads with warp-broadcast A fragments.
//
// Replaces, for these shapes, the nn.Linear/Tanh stacks + autograd of Policy.evaluate inside train()
// (models.py:52-73, 101-124; algorithms.py:213, 242, 425, 464, 665, 696).
#include "common.cuh"
#include "p2p.cuh"

namespace ppx {
namespace mf {

constexpr int TM = 128;      // samples per tile
constexpr int NT = 256;      // threads per CTA
constexpr int MAXG = 4, MAXO = 32, MAXD = 32;

struct FwdP {
  const float* X; int ldx; int M, D, G;
  const float* W1; const float* b1; const float* W2; const float* b2;     // W1 [D, G*H], b1 [G*H], W2 [G,H,H], b2 [G,H]
  const float* W3[MAXG]; const float* b3[MAXG]; int o[MAXG];              // W3.g [H, o_g], b3.g [o_g]
  float* H1; float* H2; int ldh;                                          // [M, G*H]
  float* out[MAXG];                                                       // [M, o_g]
};

struct BwdP {
  const float* X; int ldx; int M, D, G;
  const float* W2; const float* W3[MAXG]; int o[MAXG];
  const float* H1; const float* H2; int ldh;
  const float* dOut[MAXG];
  // value heads (o = 1) whose output gradient is evaluated here from the loss inputs instead of being read:
  // d = scale * (w1 * -2(R - v) + w2 * -2(R - v_clip) * [|v - v_old| <= clip]) / B_total   (ppo_loss.cu dvalue)
  const float* vh_v[MAXG]; const float* vh_ov[MAXG]; const float* vh_R[MAXG]; const double* vh_branch[MAXG];
  float vh_scale[MAXG]; float vh_clip; float vh_Bt;
  float* ws2;        // [G][nCta][H*H]        dW2 partials
  float* wsr;        // [G][nCta][RS]         dW1 | db1 | db2 | dW3 | db3 partials
  int RS;
};

struct RedP {
  const float* ws2; const float* wsr; int n2, nr, RS;      // partial counts per net
  int D, G;
  float* dW1; float* db1; float* dW2; float* db2; float* dW3[MAXG]; float* db3[MAXG]; int o[MAXG];
  double* sumsq;             // optional [G * gridDim.x]: per-block sum of squares of the final gradients (clip_grad_norm_)
  int64_t* step_dev;         // optional: optimiser step counter, bumped here when the sumsq launch is skipped
  ppx_fused_adam adam;       // adam.params != nullptr: the last block applies clip + Adam to the whole bank
  uint64_t* xg[p2p::MAXW];   // adam.W >= 2: rank r's staging area [2][W][n] of {value, seq} (device copies of adam.peer_xg_host)
};

__host__ __device__ constexpr int round4(int x) { return (x + 3) & ~3; }

// tanh(x) = 1 - 2 / (1 + e^{2x}) with ex2.approx / rcp.approx: 5 instructions instead of ~17 for tanhf, ABSOLUTE
// error <= 3e-7 on [-1, 1] outputs (the hidden activations enter the next layer as absolute values).  The bound: about
// one ulp of r = 1 / (1 + e) from rcp.approx and half an ulp of 1 + e (each worth up to 1.2e-7 once doubled), two ulp
// of e from ex2.approx (up to 1.2e-7 near x = 0), the final fma's rounding.  Measured maximum 2.2e-7 (at x = -2.66) on
// exact arguments over [-32, 32] in tests/test_gpu_mlp_edges.py.  Saturates correctly: e -> inf gives 1, e -> 0 gives -1.
__device__ __forceinline__ float tanh_fast(float x) {
  float e, r;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(x * 2.8853900817779268f));
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(e + 1.f));
  return fmaf(-2.f, r, 1.f);
}

// acc[i][q*4+c] += a_i * b[q].c  for one k
template <int CQ>
__device__ __forceinline__ void outer(float (&acc)[8][CQ * 4], const float (&a)[8], const float4 (&b)[CQ]) {
#pragma unroll
  for (int i = 0; i < 8; ++i)
#pragma unroll
    for (int q = 0; q < CQ; ++q) {
      acc[i][q * 4 + 0] = fmaf(a[i], b[q].x, acc[i][q * 4 + 0]);
      acc[i][q * 4 + 1] = fmaf(a[i], b[q].y, acc[i][q * 4 + 1]);
      acc[i][q * 4 + 2] = fmaf(a[i], b[q].z, acc[i][q * 4 + 2]);
      acc[i][q * 4 + 3] = fmaf(a[i], b[q].w, acc[i][q * 4 + 3]);
    }
}

// acc[8][CT] += A[rows ty*8.., 0..K) . B[0..K, cols]   A row-major (lda), B row-major (ldb = H), K % 4 == 0
template <int H>
__device__ __forceinline__ void tile_gemm(float (&acc)[8][H / 16], const float* __restrict__ As, int lda,
                                          const float* __restrict__ Bs, int K, int ty, int tx) {
  constexpr int CQ = H / 64;
#pragma unroll 2
  for (int k4 = 0; k4 < K; k4 += 4) {
    float4 a4[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) a4[i] = *reinterpret_cast<const float4*>(&As[(ty * 8 + i) * lda + k4]);
#pragma unroll
    for (int kk = 0; kk < 4; ++kk) {
      float4 b[CQ];
#pragma unroll
      for (int q = 0; q < CQ; ++q) b[q] = *reinterpret_cast<const float4*>(&Bs[(k4 + kk) * H + q * 64 + tx * 4]);
      float a[8];
#pragma unroll
      for (int i = 0; i < 8; ++i) a[i] = reinterpret_cast<const float*>(&a4[i])[kk];
      outer<CQ>(acc, a, b);
    }
  }
}

template <int H>
__global__ void __launch_bounds__(NT, H == 64 ? 2 : 1) mlp3_fwd_kernel(FwdP p) {
  constexpr int CT = H / 16, CQ = H / 64;
  extern __shared__ __align__(16) float sm[];
  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4, lane = tid & 31, warp = tid >> 5;
  const int g = blockIdx.y, o = p.o[g], D = p.D, Dp = round4(D);
  float* W2s = sm;                         // [H][H]
  float* W1s = W2s + H * H;                // [Dp][H]
  float* W3s = W1s + Dp * H;               // [H][o]
  float* b1s = W3s + round4(H * o);
  float* b2s = b1s + H;
  float* b3s = b2s + H;                    // [MAXO]
  float* Xs = b3s + MAXO;                  // [TM][Dp]
  float* As = Xs + TM * Dp;                // [TM][H]  H1, then H2

  for (int e = tid; e < H * H / 4; e += NT)
    reinterpret_cast<float4*>(W2s)[e] = __ldg(reinterpret_cast<const float4*>(p.W2 + (size_t)g * H * H) + e);
  for (int e = tid; e < Dp * H; e += NT) {
    const int k = e / H, c = e % H;
    W1s[e] = k < D ? __ldg(p.W1 + (size_t)k * p.ldh + g * H + c) : 0.f;
  }
  for (int e = tid; e < H * o; e += NT) W3s[e] = __ldg(p.W3[g] + e);
  for (int e = tid; e < H; e += NT) { b1s[e] = __ldg(p.b1 + g * H + e); b2s[e] = __ldg(p.b2 + g * H + e); }
  if (tid < o) b3s[tid] = __ldg(p.b3[g] + tid);

  const int nTiles = (p.M + TM - 1) / TM;
  for (int tile = blockIdx.x; tile < nTiles; tile += gridDim.x) {
    const int m0 = tile * TM;
    __syncthreads();                                        // staging done / previous tile finished with Xs, As
    if (Dp == D && p.ldx == D) {                            // dense rows: the tile is one contiguous run (no div/mod)
      const int lim = min(TM, p.M - m0) * D;
      const float* src = p.X + (size_t)m0 * D;
      for (int e = tid; e < TM * Dp; e += NT) Xs[e] = e < lim ? ld_stream(src + e) : 0.f;
    } else {
      for (int e = tid; e < TM * Dp; e += NT) {
        const int r = e / Dp, k = e % Dp;
        Xs[e] = (m0 + r < p.M && k < D) ? ld_stream(p.X + (size_t)(m0 + r) * p.ldx + k) : 0.f;
      }
    }
    __syncthreads();

    float acc[8][CT];
    // ---- layer 1 ----
#pragma unroll
    for (int q = 0; q < CQ; ++q) {
      const float4 bv = *reinterpret_cast<const float4*>(&b1s[q * 64 + tx * 4]);
#pragma unroll
      for (int i = 0; i < 8; ++i) { acc[i][q * 4] = bv.x; acc[i][q * 4 + 1] = bv.y; acc[i][q * 4 + 2] = bv.z; acc[i][q * 4 + 3] = bv.w; }
    }
    tile_gemm<H>(acc, Xs, Dp, W1s, Dp, ty, tx);
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const int r = ty * 8 + i;
#pragma unroll
      for (int q = 0; q < CQ; ++q) {
        const float4 v = make_float4(tanh_fast(acc[i][q * 4]), tanh_fast(acc[i][q * 4 + 1]), tanh_fast(acc[i][q * 4 + 2]), tanh_fast(acc[i][q * 4 + 3]));
        *reinterpret_cast<float4*>(&As[r * H + q * 64 + tx * 4]) = v;
        if (m0 + r < p.M) *reinterpret_cast<float4*>(&p.H1[(size_t)(m0 + r) * p.ldh + g * H + q * 64 + tx * 4]) = v;
      }
    }
    __syncthreads();
    // ---- layer 2 ----
#pragma unroll
    for (int q = 0; q < CQ; ++q) {
      const float4 bv = *reinterpret_cast<const float4*>(&b2s[q * 64 + tx * 4]);
#pragma unroll
      for (int i = 0; i < 8; ++i) { acc[i][q * 4] = bv.x; acc[i][q * 4 + 1] = bv.y; acc[i][q * 4 + 2] = bv.z; acc[i][q * 4 + 3] = bv.w; }
    }
    tile_gemm<H>(acc, As, H, W2s, H, ty, tx);
    if (o <= 4) {
      // ---- layer 3, narrow head: per-thread partial dot over its CT columns, fixed-order reduction over the 16
      //      column groups of a half-warp (xor 1,2,4,8), no shared-memory round trip ----
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const int r = ty * 8 + i;
        float po[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
        for (int q = 0; q < CQ; ++q) {
          const float4 v = make_float4(tanh_fast(acc[i][q * 4]), tanh_fast(acc[i][q * 4 + 1]), tanh_fast(acc[i][q * 4 + 2]), tanh_fast(acc[i][q * 4 + 3]));
          if (m0 + r < p.M) *reinterpret_cast<float4*>(&p.H2[(size_t)(m0 + r) * p.ldh + g * H + q * 64 + tx * 4]) = v;
          const float* w = &W3s[(q * 64 + tx * 4) * o];
#pragma unroll
          for (int j = 0; j < 4; ++j)
            if (j < o) po[j] = fmaf(v.w, w[3 * o + j], fmaf(v.z, w[2 * o + j], fmaf(v.y, w[o + j], fmaf(v.x, w[j], po[j]))));
        }
#pragma unroll
        for (int j = 0; j < 4; ++j)
          if (j < o) {                                      // o is CTA-uniform: no divergence around the shuffles
            float x = po[j];
            x += __shfl_xor_sync(0xffffffffu, x, 1);
            x += __shfl_xor_sync(0xffffffffu, x, 2);
            x += __shfl_xor_sync(0xffffffffu, x, 4);
            x += __shfl_xor_sync(0xffffffffu, x, 8);
            if (tx == 0 && m0 + r < p.M) p.out[g][(size_t)(m0 + r) * o + j] = x + b3s[j];
          }
      }
      continue;                                             // the loop-top barrier protects Xs / As
    }
    __syncthreads();                                        // every read of H1 done before H2 overwrites it
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const int r = ty * 8 + i;
#pragma unroll
      for (int q = 0; q < CQ; ++q) {
        const float4 v = make_float4(tanh_fast(acc[i][q * 4]), tanh_fast(acc[i][q * 4 + 1]), tanh_fast(acc[i][q * 4 + 2]), tanh_fast(acc[i][q * 4 + 3]));
        *reinterpret_cast<float4*>(&As[r * H + q * 64 + tx * 4]) = v;
        if (m0 + r < p.M) *reinterpret_cast<float4*>(&p.H2[(size_t)(m0 + r) * p.ldh + g * H + q * 64 + tx * 4]) = v;
      }
    }
    __syncthreads();
    // ---- layer 3, wide head (4 < o <= 32): one warp per row, lanes split the H inputs, fixed-order warp reduction ----
    for (int r = warp; r < TM; r += NT / 32) {
      if (m0 + r >= p.M) break;
      float res = 0.f;
      for (int j = 0; j < o; ++j) {
        float s = 0.f;
#pragma unroll
        for (int c = 0; c < H / 32; ++c) s = fmaf(As[r * H + c * 32 + lane], W3s[(c * 32 + lane) * o + j], s);
        s = warp_sum(s);
        if (lane == j) res = s;
      }
      if (lane < o) p.out[g][(size_t)(m0 + r) * o + lane] = res + b3s[lane];
    }
  }
}

// Sum v[n] over the 16 row groups (ty) of the CTA for every column group tx, in a fixed order:
// lane ^ 16 inside the warp, then the 8 warps through `part`; sink(n, tx, sum) runs once per (n, tx).
// Ends with a barrier (callers rely on it to publish their shared-memory writes as well).
template <int NV, typename F>
__device__ __forceinline__ void cross_reduce(float (&v)[NV], float* part, int tid, F&& sink) {
  const int lane = tid & 31, warp = tid >> 5;
#pragma unroll
  for (int n = 0; n < NV; ++n) v[n] += __shfl_xor_sync(0xffffffffu, v[n], 16);
  if (lane < 16) {
#pragma unroll
    for (int n = 0; n < NV; ++n) part[(warp * NV + n) * 16 + lane] = v[n];
  }
  __syncthreads();
  for (int e = tid; e < NV * 16; e += NT) {
    float s = 0.f;
#pragma unroll
    for (int w = 0; w < NT / 32; ++w) s += part[w * NV * 16 + e];
    sink(e >> 4, e & 15, s);
  }
  __syncthreads();
}

template <int H> struct BwdCfg {
  static constexpr int KC = (H == 64) ? 8 : 4;          // inputs d handled per dW1 pass
  static constexpr int KO = 4;                          // outputs j handled per dW3 pass
  static constexpr int NV = (H / 16) * (KC + 1);        // part[] is sized for the larger of the two
};

template <int H>
__global__ void __launch_bounds__(NT, H == 64 ? 2 : 1) mlp3_bwd_kernel(BwdP p) {
  constexpr int CT = H / 16, CQ = H / 64;
  constexpr int NG = NT / (2 * H);            // row groups of the dW2 accumulation (2 for H=64, 1 for H=128)
  constexpr int KC = BwdCfg<H>::KC, NV = BwdCfg<H>::NV, KS = KC + 1;
  constexpr int KO = BwdCfg<H>::KO, NVO = CT * (KO + 1), KSO = KO + 1;
  extern __shared__ __align__(16) float sm[];
  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
  const int g = blockIdx.y, o = p.o[g], D = p.D, Dp = round4(D);
  float* W2Ts = sm;                          // [H][H]   W2Ts[j][i] = W2[i][j]
  float* W3s = W2Ts + H * H;                 // [o][H]   W3s[j][c] = W3[c][j]
  float* H1s = W3s + round4(H * o);          // [TM][H]  H1
  float* H2s = H1s + TM * H;                 // [TM][H]  H2, then dP2
  float* Xs = H2s + TM * H;                  // [TM][Dp]
  float* dOs = Xs + TM * Dp;                 // [TM][o]
  float* accR = dOs + round4(TM * o);        // [RS]     dW1 | db1 | db2 | dW3 | db3
  float* part = accR + p.RS;                 // [8][NV][16]
  const int offW1 = 0, offb1 = D * H, offb2 = offb1 + H, offW3 = offb2 + H, offb3 = offW3 + H * o;

  for (int e = tid; e < H * H; e += NT) {
    const int i = e / H, j = e % H;
    W2Ts[j * H + i] = __ldg(p.W2 + (size_t)g * H * H + e);
  }
  for (int e = tid; e < H * o; e += NT) W3s[(e % o) * H + e / o] = __ldg(p.W3[g] + e);
  for (int e = tid; e < p.RS; e += NT) accR[e] = 0.f;

  float dW2[8][CT];
#pragma unroll
  for (int i = 0; i < 8; ++i)
#pragma unroll
    for (int c = 0; c < CT; ++c) dW2[i][c] = 0.f;
  // dW2 mapping: group gr takes rows [gr*TM/NG, (gr+1)*TM/NG); thread tile: inputs ti*8..+7, outputs q*64+tx*4..+3
  const int t2 = tid % (2 * H), gr = tid / (2 * H), ti = t2 >> 4;
  auto col_of = [&](int cidx, int txx) { return (cidx >> 2) * 64 + txx * 4 + (cidx & 3); };

  const int nTiles = (p.M + TM - 1) / TM;
  for (int tile = blockIdx.x; tile < nTiles; tile += gridDim.x) {
    const int m0 = tile * TM;
    __syncthreads();
    for (int e = tid; e < TM * H / 4; e += NT) {
      const int r = e / (H / 4), c4 = e % (H / 4);
      float4 v1 = make_float4(0.f, 0.f, 0.f, 0.f), v2 = v1;
      if (m0 + r < p.M) {
        const size_t off = (size_t)(m0 + r) * p.ldh + g * H + c4 * 4;
        v1 = ld_stream4(reinterpret_cast<const float4*>(p.H1 + off));
        v2 = ld_stream4(reinterpret_cast<const float4*>(p.H2 + off));
      }
      reinterpret_cast<float4*>(H1s)[e] = v1;
      reinterpret_cast<float4*>(H2s)[e] = v2;
    }
    if (Dp == D && p.ldx == D) {                            // dense rows: the tile is one contiguous run (no div/mod)
      const int lim = min(TM, p.M - m0) * D;
      const float* src = p.X + (size_t)m0 * D;
      for (int e = tid; e < TM * Dp; e += NT) Xs[e] = e < lim ? ld_stream(src + e) : 0.f;
    } else {
      for (int e = tid; e < TM * Dp; e += NT) {
        const int r = e / Dp, k = e % Dp;
        Xs[e] = (m0 + r < p.M && k < D) ? ld_stream(p.X + (size_t)(m0 + r) * p.ldx + k) : 0.f;
      }
    }
    if (p.vh_v[g] != nullptr) {                            // o == 1 (checked on the host)
      if (tid < TM) {
        float dv = 0.f;
        const int b = m0 + tid;
        if (b < p.M) {
          const float w1 = (float)p.vh_branch[g][0], w2 = (float)p.vh_branch[g][1], clip = p.vh_clip;
          const float v = ld_stream(p.vh_v[g] + b), ov = ld_stream(p.vh_ov[g] + b), R = ld_stream(p.vh_R[g] + b);
          const float d = v - ov;
          const float vc = ov + fminf(fmaxf(d, -clip), clip);
          const float pass = (d >= -clip && d <= clip) ? 1.f : 0.f;
          const float gv = w1 * (-2.f * (R - v)) + w2 * (-2.f * (R - vc)) * pass;
          dv = p.vh_scale[g] * gv / p.vh_Bt;
        }
        dOs[tid] = dv;
      }
    } else {
      const int lim = min(TM, p.M - m0) * o;
      for (int e = tid; e < TM * o; e += NT) dOs[e] = e < lim ? ld_stream(p.dOut[g] + (size_t)m0 * o + e) : 0.f;
    }
    __syncthreads();

    // ---- db3 += colsum(dOut) (o threads, 4 independent partial sums) ----
    if (tid < o) {
      float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
      for (int r = 0; r < TM; r += 4) {
        s0 += dOs[r * o + tid]; s1 += dOs[(r + 1) * o + tid]; s2 += dOs[(r + 2) * o + tid]; s3 += dOs[(r + 3) * o + tid];
      }
      accR[offb3 + tid] += (s0 + s1) + (s2 + s3);
    }
    // ---- wide heads only (o > KO): dW3 columns j >= KO, while H2s still holds H2 ----
    for (int jc = KO; jc < o; jc += KO) {
      float v[NVO];
#pragma unroll
      for (int n = 0; n < NVO; ++n) v[n] = 0.f;
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const int r = ty * 8 + i;
        float d[KO];
#pragma unroll
        for (int jj = 0; jj < KO; ++jj) d[jj] = (jc + jj < o) ? dOs[r * o + jc + jj] : 0.f;
#pragma unroll
        for (int q = 0; q < CQ; ++q) {
          const float4 h = *reinterpret_cast<const float4*>(&H2s[r * H + q * 64 + tx * 4]);
          const float hv[4] = {h.x, h.y, h.z, h.w};
#pragma unroll
          for (int cc = 0; cc < 4; ++cc)
#pragma unroll
            for (int jj = 0; jj < KO; ++jj) v[(q * 4 + cc) * KSO + jj] = fmaf(hv[cc], d[jj], v[(q * 4 + cc) * KSO + jj]);
        }
      }
      cross_reduce<NVO>(v, part, tid, [&](int n, int txx, float s) {
        const int k = n % KSO;
        if (k < KO && jc + k < o) accR[offW3 + col_of(n / KSO, txx) * o + jc + k] += s;
      });
    }
    // ---- A: dP2 = (dOut W3^T)(1 - H2^2) in place over H2s;  dW3[:, j < KO] += H2^T dOut;  db2 += colsum(dP2) ----
    {
      float v[NVO];
#pragma unroll
      for (int n = 0; n < NVO; ++n) v[n] = 0.f;
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const int r = ty * 8 + i;
        float d[KO];
#pragma unroll
        for (int jj = 0; jj < KO; ++jj) d[jj] = (jj < o) ? dOs[r * o + jj] : 0.f;
#pragma unroll
        for (int q = 0; q < CQ; ++q) {
          const int c0 = q * 64 + tx * 4;
          const float4 h = *reinterpret_cast<const float4*>(&H2s[r * H + c0]);
          const float hv[4] = {h.x, h.y, h.z, h.w};
          float sp[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
          for (int jj = 0; jj < KO; ++jj)
            if (jj < o) {                                   // CTA-uniform
              const float4 w = *reinterpret_cast<const float4*>(&W3s[jj * H + c0]);
              sp[0] = fmaf(d[jj], w.x, sp[0]); sp[1] = fmaf(d[jj], w.y, sp[1]);
              sp[2] = fmaf(d[jj], w.z, sp[2]); sp[3] = fmaf(d[jj], w.w, sp[3]);
            }
          for (int j = KO; j < o; ++j) {
            const float dj = dOs[r * o + j];
            const float4 w = *reinterpret_cast<const float4*>(&W3s[j * H + c0]);
            sp[0] = fmaf(dj, w.x, sp[0]); sp[1] = fmaf(dj, w.y, sp[1]); sp[2] = fmaf(dj, w.z, sp[2]); sp[3] = fmaf(dj, w.w, sp[3]);
          }
          float dp[4];
#pragma unroll
          for (int cc = 0; cc < 4; ++cc) {
            dp[cc] = sp[cc] * (1.f - hv[cc] * hv[cc]);
#pragma unroll
            for (int jj = 0; jj < KO; ++jj) v[(q * 4 + cc) * KSO + jj] = fmaf(hv[cc], d[jj], v[(q * 4 + cc) * KSO + jj]);
            v[(q * 4 + cc) * KSO + KO] += dp[cc];
          }
          *reinterpret_cast<float4*>(&H2s[r * H + c0]) = make_float4(dp[0], dp[1], dp[2], dp[3]);
        }
      }
      cross_reduce<NVO>(v, part, tid, [&](int n, int txx, float s) {
        const int k = n % KSO, c = col_of(n / KSO, txx);
        if (k < KO) { if (k < o) accR[offW3 + c * o + k] += s; }
        else accR[offb2 + c] += s;
      });
    }
    // ---- B: dW2 += H1^T dP2 ----
    {
      const int r0 = gr * (TM / NG);
#pragma unroll 2
      for (int r = r0; r < r0 + TM / NG; ++r) {
        const float4 a0 = *reinterpret_cast<const float4*>(&H1s[r * H + ti * 8]);
        const float4 a1 = *reinterpret_cast<const float4*>(&H1s[r * H + ti * 8 + 4]);
        float4 b[CQ];
#pragma unroll
        for (int q = 0; q < CQ; ++q) b[q] = *reinterpret_cast<const float4*>(&H2s[r * H + q * 64 + tx * 4]);
        const float a[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
        outer<CQ>(dW2, a, b);
      }
    }
    // ---- C: dP1 = (dP2 W2^T)(1 - H1^2) kept in registers;  dW1 += X^T dP1;  db1 += colsum(dP1) ----
    {
      float acc[8][CT];
#pragma unroll
      for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int c = 0; c < CT; ++c) acc[i][c] = 0.f;
      tile_gemm<H>(acc, H2s, H, W2Ts, H, ty, tx);
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const int r = ty * 8 + i;
#pragma unroll
        for (int q = 0; q < CQ; ++q) {
          const float4 h = *reinterpret_cast<const float4*>(&H1s[r * H + q * 64 + tx * 4]);
          acc[i][q * 4] *= (1.f - h.x * h.x); acc[i][q * 4 + 1] *= (1.f - h.y * h.y);
          acc[i][q * 4 + 2] *= (1.f - h.z * h.z); acc[i][q * 4 + 3] *= (1.f - h.w * h.w);
        }
      }
      for (int dc = 0; dc < D; dc += KC) {
        float v[NV];
#pragma unroll
        for (int n = 0; n < NV; ++n) v[n] = 0.f;
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const int r = ty * 8 + i;
          float x[KC];
#pragma unroll
          for (int k4 = 0; k4 < KC; k4 += 4) {
            const float4 xv = (dc + k4 < Dp) ? *reinterpret_cast<const float4*>(&Xs[r * Dp + dc + k4]) : make_float4(0.f, 0.f, 0.f, 0.f);
            x[k4] = xv.x; x[k4 + 1] = xv.y; x[k4 + 2] = xv.z; x[k4 + 3] = xv.w;
          }
#pragma unroll
          for (int c = 0; c < CT; ++c) {
#pragma unroll
            for (int dd = 0; dd < KC; ++dd) v[c * KS + dd] = fmaf(acc[i][c], x[dd], v[c * KS + dd]);
            v[c * KS + KC] += acc[i][c];
          }
        }
        cross_reduce<NV>(v, part, tid, [&](int n, int txx, float s) {
          const int k = n % KS, c = col_of(n / KS, txx);
          if (k < KC) { if (dc + k < D) accR[offW1 + (dc + k) * H + c] += s; }
          else if (dc == 0) accR[offb1 + c] += s;
        });
      }
    }
  }
  __syncthreads();
  float* wr = p.wsr + ((size_t)g * gridDim.x + blockIdx.x) * p.RS;
  for (int e = tid; e < p.RS; e += NT) wr[e] = accR[e];
  // dW2: the NG row groups are combined here in a fixed order (through H1s, free by now) -> one partial per CTA
  float* w2 = p.ws2 + (size_t)(g * gridDim.x + blockIdx.x) * H * H;
  if (NG > 1) {
    if (gr == 1) {
#pragma unroll
      for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int q = 0; q < CQ; ++q)
          *reinterpret_cast<float4*>(&H1s[(ti * 8 + i) * H + q * 64 + tx * 4]) =
              make_float4(dW2[i][q * 4], dW2[i][q * 4 + 1], dW2[i][q * 4 + 2], dW2[i][q * 4 + 3]);
    }
    __syncthreads();
  }
  if (gr == 0) {
#pragma unroll
    for (int i = 0; i < 8; ++i)
#pragma unroll
      for (int q = 0; q < CQ; ++q) {
        float4 o4 = make_float4(dW2[i][q * 4], dW2[i][q * 4 + 1], dW2[i][q * 4 + 2], dW2[i][q * 4 + 3]);
        if (NG > 1) {
          const float4 t = *reinterpret_cast<const float4*>(&H1s[(ti * 8 + i) * H + q * 64 + tx * 4]);
          o4.x += t.x; o4.y += t.y; o4.z += t.z; o4.w += t.w;
        }
        *reinterpret_cast<float4*>(&w2[(ti * 8 + i) * H + q * 64 + tx * 4]) = o4;
      }
  }
}

template <int H>
__device__ __forceinline__ float* mlp3_reduce_finish(const RedP& p, float (&sl)[8][33], float s, int e, int R, int g, int o, int D, int el,
                                                     float* grad_value) {
  const bool live = e < H * H + R;
  if (live) {
#pragma unroll
    for (int q = 1; q < 8; ++q) s += sl[q][el];
  } else {
    s = 0.f;
  }
  if (p.sumsq) {                                              // first warp: fixed-order sum of squares of this block's 32 gradients
    const double ss = warp_sum((double)s * (double)s);
    if (el == 0) p.sumsq[(size_t)g * gridDim.x + blockIdx.x] = ss;
    if (p.step_dev && el == 0 && blockIdx.x == 0 && g == 0) *p.step_dev += 1;
  }
  float* dst = nullptr;
  if (live) {
    if (e < H * H) dst = p.dW2 + (size_t)g * H * H + e;
    else {
      const int r = e - H * H;
      if (r < D * H) dst = p.dW1 + (size_t)(r / H) * (p.G * H) + g * H + r % H;
      else if (r < D * H + H) dst = p.db1 + g * H + (r - D * H);
      else if (r < D * H + 2 * H) dst = p.db2 + g * H + (r - D * H - H);
      else if (r < D * H + 2 * H + H * o) dst = p.dW3[g] + (r - D * H - 2 * H);
      else dst = p.db3[g] + (r - D * H - 2 * H - H * o);
    }
    *dst = s;
  }
  *grad_value = s;
  return dst;
}

// Optimiser tail (ppx_fused_adam).  clip_grad_norm_ needs the norm over ALL gradients, i.e. a grid-wide dependency inside
// the reduce kernel.  (First version: the last block to finish applied Adam to the whole bank -- one CTA walking 9732
// parameters with dependent loads cost 53 us, more than the separate Adam launch it replaced.)  Now every block publishes
// its sum of squares, the grid meets at a counter (the launch is COOPERATIVE, so all blocks are resident and the spin
// cannot deadlock), every block re-reads the partials in the same fixed order -- identical clip coefficient everywhere --
// and its first warp applies Adam to the 32 parameters whose gradients it has just produced; block (0,0) also takes the
// parameters outside the MLP (action_log_std) and bumps the step counter.  ticket[0] = arrivals, ticket[1] = departures
// (the last block to leave re-arms both).
// Sharded (a.W >= 2): the gradient all-reduce happens in the same place, per block, over peer memory, with the
// low-latency "value + tag in one 8-byte store" protocol: the first warp PUSHES the 32 gradients it has just reduced into
// every rank's staging area (remote stores over NVLink, slot [seq parity][own rank][param] = {f32 value, u32 seq}), then
// polls its own W slots until each carries this launch's sequence number and sums them in rank order -- every rank
// computes bit-identical sums, so the weights stay replicas.  No fence, no flag hop, no remote load, no separate exchange
// kernel: the cost is one one-way NVLink latency plus the skew between the ranks.  (An 8-byte aligned store is delivered
// whole; the parity double-buffering keeps a fast rank's launch k+1 from overwriting a slot of launch k: it cannot reach
// launch k+2 before every peer has finished launch k.)
__device__ __forceinline__ void st_ll(uint64_t* p, float v, uint32_t tag) {
  asm volatile("st.relaxed.sys.global.v2.u32 [%0], {%1, %2};" ::"l"(p), "r"(__float_as_uint(v)), "r"(tag) : "memory");
}
__device__ __forceinline__ float ld_ll_wait(const uint64_t* p, uint32_t tag, uint32_t* status) {
  uint32_t v, t;
  const uint64_t t0 = p2p::now_ns();
  for (;;) {
    asm volatile("ld.volatile.global.v2.u32 {%0, %1}, [%2];" : "=r"(v), "=r"(t) : "l"(p) : "memory");
    if (t == tag) break;
    if (p2p::now_ns() - t0 > 4000000000ull) { atomicExch(status, 1u); break; }
  }
  return __uint_as_float(v);
}

__device__ void fused_adam_tail(const RedP& p, int n_partials, float* gptr, float gval, bool first_warp) {
  const ppx_fused_adam& a = p.adam;
  __shared__ double s_red[32];
  __shared__ float s_coef, s_step_size, s_bc2_sqrt;
  const unsigned int total = gridDim.x * gridDim.y;
  const bool lead = blockIdx.x == 0 && blockIdx.y == 0;
  const int64_t t_ = *a.step_dev + 1;                          // read before the rendezvous, written (block 0) after it
  const int extra_off = (int)(a.extra_grads - a.grads);
  uint32_t seq = 0;
  if (a.W >= 2) {
    seq = *a.seq_dev + 1u;                                     // same protocol as step_dev
    if (first_warp) {
      const int lane = threadIdx.x & 31, W = a.W, rank = a.rank;
      const int blk = blockIdx.y * gridDim.x + blockIdx.x;
      const size_t slot = (size_t)(seq & 1u) * W * a.n;
      const int64_t idx = gptr ? (int64_t)(gptr - a.grads) : -1;
      if (gptr)
        for (int r = 0; r < W; ++r) st_ll(p.xg[r] + slot + (size_t)rank * a.n + idx, gval, seq);
      if (lead)
        for (int k = lane; k < a.n_extra; k += 32) {
          const float v = a.extra_grads[k];
          for (int r = 0; r < W; ++r) st_ll(p.xg[r] + slot + (size_t)rank * a.n + extra_off + k, v, seq);
        }
      const uint64_t* mine_xg = p.xg[rank] + slot;
      double ss = 0.0;
      if (gptr) {
        float g = 0.f;
        for (int r = 0; r < W; ++r) g += ld_ll_wait(mine_xg + (size_t)r * a.n + idx, seq, a.status_dev);
        *gptr = g;                                             // the bank's gradient vector holds the global gradient
        gval = g;
        ss = (double)g * (double)g;
      }
      if (lead)
        for (int k = lane; k < a.n_extra; k += 32) {
          float g = 0.f;
          for (int r = 0; r < W; ++r) g += ld_ll_wait(mine_xg + (size_t)r * a.n + extra_off + k, seq, a.status_dev);
          const_cast<float*>(a.extra_grads)[k] = g;            // read back (ldcg) after the grid rendezvous
        }
      ss = warp_sum(ss);
      if (lane == 0) p.sumsq[blk] = ss;                        // replaces the local-gradient partial written by reduce_finish
    }
  }
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) {
    atomicAdd(a.ticket, 1u);
    unsigned int seen;
    do {
      asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(seen) : "l"(a.ticket) : "memory");
      if (seen < total) __nanosleep(64);
    } while (seen < total);
  }
  __syncthreads();
  double ss = 0.0;
  if (a.max_norm > 0.0) {
    for (int k = threadIdx.x; k < n_partials; k += blockDim.x) ss += __ldcg(p.sumsq + k);
    for (int k = threadIdx.x; k < a.n_extra; k += blockDim.x) { const double v = (double)__ldcg(a.extra_grads + k); ss += v * v; }
    ss = block_sum(ss, s_red);
  }
  if (threadIdx.x == 0) {
    const double t = (double)t_;
    s_step_size = (float)(a.lr / (1.0 - pow(a.beta1, t)));
    s_bc2_sqrt = (float)sqrt(1.0 - pow(a.beta2, t));
    float coef = 1.f;
    if (a.max_norm > 0.0) {
      const float norm = (float)sqrt(ss);
      coef = fminf((float)a.max_norm / (norm + 1e-6f), 1.f);   // clip_grad_norm_: clamp(max_norm/(norm+1e-6), max=1)
      if (lead && a.norm_out) *a.norm_out = sqrt(ss);
    }
    s_coef = coef;
    if (lead) *a.step_dev = t_;
    if (lead && a.W >= 2) *a.seq_dev = seq;
    if (atomicAdd(a.ticket + 1, 1u) == total - 1) { a.ticket[0] = 0u; a.ticket[1] = 0u; __threadfence(); }
  }
  __syncthreads();
  const float coef = s_coef, step_size = s_step_size, bc2_sqrt = s_bc2_sqrt;
  const float w1 = (float)(1.0 - a.beta1), beta2 = (float)a.beta2, w2 = (float)(1.0 - a.beta2), eps = (float)a.eps;
  auto upd = [&](int64_t i, float gi) {
    gi *= coef;
    float mi = a.exp_avg[i], vi = a.exp_avg_sq[i];
    mi = mi + w1 * (gi - mi);                                 // exp_avg.lerp_(grad, 1-beta1)
    vi = vi * beta2 + w2 * gi * gi;                           // exp_avg_sq.mul_(beta2).addcmul_(grad, grad, 1-beta2)
    const float denom = sqrtf(vi) / bc2_sqrt + eps;
    a.params[i] = a.params[i] - step_size * (mi / denom);     // param.addcdiv_(exp_avg, denom, -step_size)
    a.exp_avg[i] = mi;
    a.exp_avg_sq[i] = vi;
  };
  if (first_warp && gptr) upd((int64_t)(gptr - a.grads), gval);
  if (lead)
    for (int k = threadIdx.x; k < a.n_extra; k += blockDim.x) upd((int64_t)extra_off + k, __ldcg(a.extra_grads + k));
}

// grads[e] = sum over CTA partials in a fixed order.  Block = 32 consecutive parameters x 8 slices of the
// partial list (slice s takes partials s, s+8, ...: many independent loads in flight), slices combined 0..7.
template <int H>
__global__ void __launch_bounds__(256) mlp3_reduce_kernel(RedP p) {
  __shared__ float sl[8][33];
  const int g = blockIdx.y, o = p.o[g], D = p.D;
  const int el = threadIdx.x & 31, slice = threadIdx.x >> 5;
  const int e = blockIdx.x * 32 + el;
  const int R = D * H + 2 * H + H * o + o;
  float s = 0.f;
  if (e < H * H + R) {
    const bool w2 = e < H * H;
    const int n = w2 ? p.n2 : p.nr;
    const size_t stride = w2 ? (size_t)H * H : (size_t)p.RS;
    const float* src = w2 ? p.ws2 + (size_t)g * p.n2 * H * H + e : p.wsr + (size_t)g * p.nr * p.RS + (e - H * H);
    float s0 = 0.f, s1 = 0.f;
    int k = slice;
    for (; k + 8 < n; k += 16) { s0 += src[(size_t)k * stride]; s1 += src[(size_t)(k + 8) * stride]; }
    if (k < n) s0 += src[(size_t)k * stride];
    s = s0 + s1;
  }
  sl[slice][el] = s;
  __syncthreads();
  float* gptr = nullptr;
  float gval = 0.f;
  if (slice == 0) gptr = mlp3_reduce_finish<H>(p, sl, s, e, R, g, o, D, el, &gval);
  if (p.adam.params) fused_adam_tail(p, (int)(gridDim.x * gridDim.y), gptr, gval, slice == 0);
}

inline size_t fwd_smem(int H, int D, int o) {
  const int Dp = round4(D);
  return sizeof(float) * ((size_t)H * H + (size_t)Dp * H + round4(H * o) + 2 * H + MAXO + (size_t)TM * Dp + (size_t)TM * H);
}
inline int rest_size(int H, int D, int o) { return D * H + 2 * H + H * o + o; }
inline size_t bwd_smem(int H, int D, int o, int RS) {
  const int Dp = round4(D);
  const int NV = H == 64 ? BwdCfg<64>::NV : BwdCfg<128>::NV;
  return sizeof(float) * ((size_t)H * H + round4(H * o) + 2 * (size_t)TM * H + (size_t)TM * Dp + round4(TM * o) + RS +
                          (size_t)(NT / 32) * NV * 16);
}
constexpr size_t kMaxSmem = 227 * 1024;

struct Shape { int H, D, G, omax, RS; };
inline bool shape_ok(int D, int H, int G, const int* outs, Shape* s) {
  if (!(H == 64 || H == 128) || D < 1 || D > MAXD || G < 1 || G > MAXG) return false;
  int omax = 0;
  for (int g = 0; g < G; ++g) { if (outs[g] < 1 || outs[g] > MAXO) return false; omax = std::max(omax, outs[g]); }
  const int RS = round4(rest_size(H, D, omax));
  if (fwd_smem(H, D, omax) > kMaxSmem || bwd_smem(H, D, omax, RS) > kMaxSmem) return false;
  if (s) *s = Shape{H, D, G, omax, RS};
  return true;
}

template <typename K>
int ctas_per_sm(K kernel, size_t smem) {
  int n = 0;
  if (cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) return 0;
  if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, kernel, NT, smem) != cudaSuccess) return 0;
  return n;
}

// persistent grid: CTAs per net so that all G nets fill the machine once
inline int grid_x(int M, int G, int per_sm) {
  const int nTiles = (M + TM - 1) / TM;
  const int slots = std::max(1, sm_count() * std::max(per_sm, 1) / G);
  return std::max(1, std::min(nTiles, slots));
}

// fixed-order sum of the per-CTA partials of a backward kernel (this file's or mlp_tc.cu's) into the gradient tensors
int mlp3_reduce_launch(int H, int D, int G, const int* outs, const float* ws2, const float* wsr, int n, int RS, float* dW1,
                       float* db1, float* dW2, float* db2, float* const* dW3, float* const* db3, double* sumsq,
                       int64_t* step_dev, const ppx_fused_adam* adam, cudaStream_t st) {
  int omax = 0;
  for (int g = 0; g < G; ++g) omax = std::max(omax, outs[g]);
  RedP r{};
  r.ws2 = ws2; r.wsr = wsr; r.n2 = n; r.nr = n; r.RS = RS; r.D = D; r.G = G;
  r.dW1 = dW1; r.db1 = db1; r.dW2 = dW2; r.db2 = db2; r.sumsq = sumsq; r.step_dev = step_dev;
  if (adam) {
    PPX_REQUIRE(adam->params && adam->grads && adam->exp_avg && adam->exp_avg_sq && adam->step_dev && adam->ticket && adam->n >= 1 &&
                adam->n_extra >= 0 && (adam->n_extra == 0 || adam->extra_grads), "mlp3 fused adam: bad arguments");
    r.adam = *adam;
    if (adam->W >= 2) {
      PPX_REQUIRE(adam->W <= p2p::MAXW && adam->rank >= 0 && adam->rank < adam->W && adam->peer_xg_host && adam->seq_dev &&
                  adam->status_dev && sumsq, "mlp3 fused adam: bad peer arguments (W=%d rank=%d)", adam->W, adam->rank);
      for (int q = 0; q < adam->W; ++q) {
        PPX_REQUIRE(adam->peer_xg_host[q], "mlp3 fused adam: null peer pointer for rank %d", q);
        r.xg[q] = (uint64_t*)adam->peer_xg_host[q];
      }
    }
  }
  for (int g = 0; g < G; ++g) { r.dW3[g] = dW3[g]; r.db3[g] = db3[g]; r.o[g] = outs[g]; }
  dim3 rgrid((unsigned)ceil_div(H * H + rest_size(H, D, omax), 32), (unsigned)G);
  if (adam) {                                                 // grid-wide rendezvous inside: all blocks must be resident
    const void* fn = H == 64 ? (const void*)mlp3_reduce_kernel<64> : (const void*)mlp3_reduce_kernel<128>;
    static int per_sm[2] = {0, 0};
    int& occ = per_sm[H == 64 ? 0 : 1];
    if (!occ) PPX_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, fn, 256, 0));
    PPX_REQUIRE(adam->W < 2 || (int64_t)rgrid.x * rgrid.y <= (int64_t)occ * sm_count(),
                "mlp3 fused adam: the sharded tail needs %lld co-resident blocks (ppx_mlp3_fused_adam_blocks)", (long long)rgrid.x * rgrid.y);
    if ((int64_t)rgrid.x * rgrid.y > (int64_t)occ * sm_count()) {
      // more blocks than can be resident (h = 128, three nets): plain reduce + the stand-alone clip+Adam launch
      r.adam = ppx_fused_adam{};
      if (H == 64) mlp3_reduce_kernel<64><<<rgrid, 256, 0, st>>>(r);
      else mlp3_reduce_kernel<128><<<rgrid, 256, 0, st>>>(r);
      int rc = after_launch("mlp3_reduce");
      if (rc) return rc;
      return ppx_clip_adam(adam->params, adam->grads, adam->exp_avg, adam->exp_avg_sq, adam->n, adam->max_norm,
                           adam->max_norm > 0.0 ? adam->n : 0, adam->lr, adam->beta1, adam->beta2, adam->eps, 0, adam->step_dev,
                           adam->norm_out, sumsq, (void*)st);
    }
    void* args[] = {&r};
    PPX_CUDA(cudaLaunchCooperativeKernel(fn, rgrid, dim3(256), args, 0, st));
  } else if (H == 64) mlp3_reduce_kernel<64><<<rgrid, 256, 0, st>>>(r);
  else mlp3_reduce_kernel<128><<<rgrid, 256, 0, st>>>(r);
  return after_launch("mlp3_reduce");
}

}  // namespace mf
}  // namespace ppx

using namespace ppx;

extern "C" int ppx_mlp3_fused_adam_blocks(int D, int H, int G, const int* outs) {
  if (!outs || !mf::shape_ok(D, H, G, outs, nullptr)) return 0;
  int omax = 0;
  for (int g = 0; g < G; ++g) omax = std::max(omax, outs[g]);
  const int64_t blocks = (int64_t)ceil_div(H * H + mf::rest_size(H, D, omax), 32) * G;
  const void* fn = H == 64 ? (const void*)mf::mlp3_reduce_kernel<64> : (const void*)mf::mlp3_reduce_kernel<128>;
  int occ = 0;
  if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, fn, 256, 0) != cudaSuccess) return 0;
  return blocks <= (int64_t)occ * sm_count() ? (int)blocks : 0;
}

extern "C" int ppx_mlp3_supported(int D, int H, int G, const int* outs) {
  return (outs && mf::shape_ok(D, H, G, outs, nullptr)) ? 1 : 0;
}

extern "C" int ppx_mlp3_fwd(const float* X, int ldx, int M, int D, int H, int G, const int* outs, const float* W1,
                            const float* b1, const float* W2, const float* b2, const float* const* W3,
                            const float* const* b3, float* H1, float* H2, float* const* out, void* stream) {
  mf::Shape s;
  PPX_REQUIRE(X && outs && W1 && b1 && W2 && b2 && W3 && b3 && H1 && H2 && out, "mlp3_fwd: null pointer");
  PPX_REQUIRE(mf::shape_ok(D, H, G, outs, &s), "mlp3_fwd: unsupported shape D=%d H=%d G=%d", D, H, G);
  PPX_REQUIRE(M >= 0 && ldx >= D, "mlp3_fwd: M=%d ldx=%d", M, ldx);
  if (M == 0) return PPX_OK;
  mf::FwdP p{};
  p.X = X; p.ldx = ldx; p.M = M; p.D = D; p.G = G; p.W1 = W1; p.b1 = b1; p.W2 = W2; p.b2 = b2; p.H1 = H1; p.H2 = H2; p.ldh = G * H;
  for (int g = 0; g < G; ++g) { p.W3[g] = W3[g]; p.b3[g] = b3[g]; p.o[g] = outs[g]; p.out[g] = out[g]; }
  const size_t smem = mf::fwd_smem(H, D, s.omax);
  cudaStream_t st = (cudaStream_t)stream;
  if (H == 64) {
    static int occ = 0;
    if (!occ) occ = mf::ctas_per_sm(mf::mlp3_fwd_kernel<64>, mf::kMaxSmem);
    PPX_REQUIRE(occ > 0, "mlp3_fwd: kernel cannot be resident");
    dim3 grid((unsigned)mf::grid_x(M, G, 2), (unsigned)G);
    mf::mlp3_fwd_kernel<64><<<grid, mf::NT, smem, st>>>(p);
  } else {
    static int occ = 0;
    if (!occ) occ = mf::ctas_per_sm(mf::mlp3_fwd_kernel<128>, mf::kMaxSmem);
    PPX_REQUIRE(occ > 0, "mlp3_fwd: kernel cannot be resident");
    dim3 grid((unsigned)mf::grid_x(M, G, 1), (unsigned)G);
    mf::mlp3_fwd_kernel<128><<<grid, mf::NT, smem, st>>>(p);
  }
  return after_launch("mlp3_fwd");
}

namespace {
int bwd_grid(int M, int H, int G) {
  return mf::grid_x(M, G, H == 64 ? 2 : 1);
}
}  // namespace

extern "C" int ppx_mlp3_sumsq_partials(int D, int H, int G, const int* outs) {
  mf::Shape s;
  if (!outs || !mf::shape_ok(D, H, G, outs, &s)) return -1;
  return G * (int)ceil_div(H * H + mf::rest_size(H, D, s.omax), 32);
}

extern "C" int64_t ppx_mlp3_bwd_workspace(int M, int D, int H, int G, const int* outs) {
  mf::Shape s;
  if (!outs || !mf::shape_ok(D, H, G, outs, &s)) return -1;
  const int n = bwd_grid(M, H, G);
  return (int64_t)G * n * ((int64_t)H * H + s.RS);
}

extern "C" int ppx_mlp3_bwd(const float* X, int ldx, int M, int D, int H, int G, const int* outs, const float* W2,
                            const float* const* W3, const float* H1, const float* H2, const float* const* dOut,
                            const ppx_value_head* vh, float clip_range, int64_t B_total,
                            float* dW1, float* db1, float* dW2, float* db2, float* const* dW3, float* const* db3,
                            float* workspace, double* sumsq_partials, int64_t* step_dev, const ppx_fused_adam* adam,
                            void* stream) {
  mf::Shape s;
  PPX_REQUIRE(X && outs && W2 && W3 && H1 && H2 && dOut && dW1 && db1 && dW2 && db2 && dW3 && db3 && workspace, "mlp3_bwd: null pointer");
  PPX_REQUIRE(!adam || sumsq_partials, "mlp3_bwd: the fused optimiser tail needs sumsq_partials");
  PPX_REQUIRE(mf::shape_ok(D, H, G, outs, &s), "mlp3_bwd: unsupported shape D=%d H=%d G=%d", D, H, G);
  PPX_REQUIRE(M >= 1 && ldx >= D, "mlp3_bwd: M=%d ldx=%d", M, ldx);
  const int n = bwd_grid(M, H, G);
  const int NG = mf::NT / (2 * H);
  mf::BwdP p{};
  p.X = X; p.ldx = ldx; p.M = M; p.D = D; p.G = G; p.W2 = W2; p.H1 = H1; p.H2 = H2; p.ldh = G * H;
  p.ws2 = workspace; p.wsr = workspace + (size_t)G * n * H * H; p.RS = s.RS;
  p.vh_clip = clip_range; p.vh_Bt = (float)(B_total > 0 ? B_total : M);
  for (int g = 0; g < G; ++g) {
    p.W3[g] = W3[g]; p.o[g] = outs[g]; p.dOut[g] = dOut[g];
    if (vh && vh[g].values) {
      PPX_REQUIRE(outs[g] == 1 && vh[g].old_values && vh[g].returns && vh[g].branch, "mlp3_bwd: value head %d needs o=1 and all inputs", g);
      p.vh_v[g] = vh[g].values; p.vh_ov[g] = vh[g].old_values; p.vh_R[g] = vh[g].returns; p.vh_branch[g] = vh[g].branch;
      p.vh_scale[g] = vh[g].scale;
    } else {
      PPX_REQUIRE(dOut[g], "mlp3_bwd: dOut[%d] is null", g);
    }
  }
  const size_t smem = mf::bwd_smem(H, D, s.omax, s.RS);
  cudaStream_t st = (cudaStream_t)stream;
  dim3 grid((unsigned)n, (unsigned)G);
  if (H == 64) {
    static int occ = 0;
    if (!occ) occ = mf::ctas_per_sm(mf::mlp3_bwd_kernel<64>, mf::kMaxSmem);
    PPX_REQUIRE(occ > 0, "mlp3_bwd: kernel cannot be resident");
    mf::mlp3_bwd_kernel<64><<<grid, mf::NT, smem, st>>>(p);
  } else {
    static int occ = 0;
    if (!occ) occ = mf::ctas_per_sm(mf::mlp3_bwd_kernel<128>, mf::kMaxSmem);
    PPX_REQUIRE(occ > 0, "mlp3_bwd: kernel cannot be resident");
    mf::mlp3_bwd_kernel<128><<<grid, mf::NT, smem, st>>>(p);
  }
  int rc = after_launch("mlp3_bwd");
  if (rc) return rc;
  return mf::mlp3_reduce_launch(H, D, G, outs, p.ws2, p.wsr, n, s.RS, dW1, db1, dW2, db2, dW3, db3, sumsq_partials,
                                (sumsq_partials && !adam) ? step_dev : nullptr, adam, st);
}
