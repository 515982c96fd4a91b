// Policy MLPs on the Blackwell tensor cores: forward and backward of G independent  D -> 64 -> 64 -> o_g  tanh MLPs
// (actor | critic | int_critic of models.py:137-213) with the two 64x64 GEMMs of every pass on tcgen05.mma kind::tf32
// in fp32-equivalent precision (3xTF32: A_lo.B_hi + A_hi.B_lo + A_hi.B_hi, the lo.lo term ~2^-22 dropped).
//
// The SIMT kernels of mlp_fused.cu spend ~90 % of their instructions on the FMAs of those GEMMs.  Here a thread owns
// (sample s, 32 hidden columns) -- the tcgen05.ld 32x32b register layout -- and only does the elementwise work (first
// layer with K = D <= 32, tanh, hi/lo split, head layer, thin reductions); the GEMM operands are written by the same
// threads straight into 128-byte-swizzled K-major shared-memory images and the accumulators live in TMEM.
//   * kind::tf32 truncates its operands, so the RAW fp32 image is the "hi" operand; only lo = x - trunc(x) is extra
//     (tools/umma_probe.cu: identical results with and without the explicit mask).
//   * MN-major tf32 operands need the 32-byte-atom swizzle and cannot share an image with a K-major use of the same
//     data, so the weight-gradient GEMM (reduction over the samples) gets TRANSPOSED images, written with
//     conflict-free scalar stores (lanes = consecutive samples = consecutive words of a 128-byte row).
//   * the saved activations are private to this pair of kernels and are kept per tile in HBM as
//     Ht [G][tile][16 column quads][128 samples][4]: a thread moves its 32 columns of a sample as 8 float4 and a warp
//     instruction covers 512 contiguous bytes in both kernels.
//   * the tensor core's fp32 accumulator truncates on every MMA; small terms are accumulated first and dW2 is drained
//     into fp32 registers after every tile (48 MMAs), so the drift stays ~1e-6 (tests/test_gpu_mlp_tc.py).
// Forward: 2 CTAs/SM (96 KB of images each) so one CTA's MMA + epilogue overlaps the other's first layer.
// Backward: 1 CTA/SM (198 KB); GEMM 2 (dP1 = dP2 W2^T) runs under the H1^T image writes and the dW3/db2 sums,
// GEMM 1 (dW2 += H1^T dP2) under the dW1/db1 sums and the next tile's loads.  Partials leave in the same format as
// mlp_fused.cu's backward and go through the same fixed-order reduce kernel (deterministic, no float atomics).
//
// Replaces, for H = 64, the nn.Linear/Tanh stacks + autograd of Policy.evaluate inside train()
// (models.py:52-73, 101-124; algorithms.py:213, 242, 425, 464, 665, 696).
#include <atomic>
#include <cstdlib>
#include <type_traits>
#include "tc_common.cuh"

namespace ppx {
namespace mf {
// defined in mlp_fused.cu: fixed-order sum of the per-CTA partials (+ optional clip_grad_norm_ partial sums)
int mlp3_reduce_launch(int H, int D, int G, const int* outs, const float* ws2, const float* wsr, int n, int RS, float* dW1,
                       float* db1, float* dW2, float* db2, float* const* dW3, float* const* db3, double* sumsq,
                       int64_t* step_dev, const ppx_fused_adam* adam, cudaStream_t st);
}  // namespace mf

namespace mt {
using namespace tc;

constexpr int H = 64, TM = 128, NT = 256, MAXG = 4, MAXO = 4, MAXD = 32;
__host__ __device__ constexpr int round4(int x) { return (x + 3) & ~3; }

__device__ __forceinline__ float tanh_fast(float x) {   // same 5-instruction form as mlp_fused.cu (abs error <= 3e-7)
  float e, r;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(x * 2.8853900817779268f));
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(e + 1.f));
  return fmaf(-2.f, r, 1.f);
}
__device__ __forceinline__ float lo_of(float x) { return x - __uint_as_float(__float_as_uint(x) & 0xFFFFE000u); }
// shared-memory accesses by 32-bit shared-window address (the image bases come from a run-time 1024-byte alignment, which
// would otherwise turn every access into a generic LD/ST with 64-bit address arithmetic)
__device__ __forceinline__ void sts32(uint32_t a, float v) { asm volatile("st.shared.f32 [%0], %1;" ::"r"(a), "f"(v) : "memory"); }
__device__ __forceinline__ void sts128(uint32_t a, float x, float y, float z, float w) {
  asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(a), "f"(x), "f"(y), "f"(z), "f"(w) : "memory");
}
__device__ __forceinline__ float lds32(uint32_t a) {
  float v;
  asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(a) : "memory");
  return v;
}
__device__ __forceinline__ float4 lds128(uint32_t a) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(a) : "memory");
  return v;
}

struct FwdP {
  const float* X; int ldx; int M, D, G, nTiles;
  const float* W1; const float* b1; const float* W2; const float* b2;     // W1 [D, G*H], b1 [G*H], W2 [G,H,H] in-major, b2 [G,H]
  const float* W3[MAXG]; const float* b3[MAXG]; int o[MAXG];
  float* H1t; float* H2t;                                                  // [G][nTiles][H][TM]
  float* out[MAXG];
};

// row `row` of X (zero beyond M / D) into registers
template <int DP>
__device__ __forceinline__ void load_x_row(const float* __restrict__ X, int ldx, int D, bool live, float (&x)[DP]) {
  const bool vec = ((ldx & 3) == 0) && ((D & 3) == 0) && ((reinterpret_cast<uintptr_t>(X) & 15) == 0);
  if (vec) {
#pragma unroll
    for (int k = 0; k < DP; k += 4) {
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      if (live && k < D) v = __ldg(reinterpret_cast<const float4*>(X + k));
      x[k] = v.x; x[k + 1] = v.y; x[k + 2] = v.z; x[k + 3] = v.w;
    }
  } else {
#pragma unroll
    for (int k = 0; k < DP; ++k) x[k] = (live && k < D) ? __ldg(X + k) : 0.f;
  }
}

// one thread: v[32] = 32 consecutive columns (c0..c0+31, block kb = c0/32) of row s -> raw and lo K-major images
__device__ __forceinline__ void store_row_images(uint32_t raw, uint32_t lo, int s, const float (&v)[32]) {
  const uint32_t row = (uint32_t)(s * 128), x = (uint32_t)(s & 7);
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    const uint32_t off = row + ((j ^ x) << 4);
    sts128(raw + off, v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
    sts128(lo + off, lo_of(v[4 * j]), lo_of(v[4 * j + 1]), lo_of(v[4 * j + 2]), lo_of(v[4 * j + 3]));
  }
}
// one thread: v[32] = elements (row r0+c, column s) of a transposed image with 64-row k-blocks (block = s/32)
// (r0 is a multiple of 32 and every other term of the base has zero bits [4,7), so the row swizzle is an XOR of the base
// with the compile-time constant (c & 7) << 4 and the row pitch is an immediate offset)
__device__ __forceinline__ void store_col_images(uint32_t raw, uint32_t lo_delta, int r0, int s, const float (&v)[32]) {
  const uint32_t l = (uint32_t)(s & 31);
  const uint32_t base = raw + (uint32_t)((s >> 5) * 8192 + r0 * 128) + ((l & 3) << 2) + ((l >> 2) << 4);
#pragma unroll
  for (int c = 0; c < 32; ++c) {
    const uint32_t a = (base ^ (uint32_t)((c & 7) << 4)) + (uint32_t)(c * 128);
    sts32(a, v[c]);
    sts32(a + lo_delta, lo_of(v[c]));
  }
}

// W [64][64] row-major (global) -> K-major image of B[n][k] = W[n][k] (transpose = false) or W[k][n] (transpose = true)
__device__ __forceinline__ void stage_weight(uint32_t raw, uint32_t lo, const float* __restrict__ W, bool transpose, int tid) {
  float w[H * H / NT];
#pragma unroll
  for (int r = 0; r < H * H / NT; ++r) w[r] = __ldg(W + tid + r * NT);          // all loads in flight before the first store
#pragma unroll
  for (int r = 0; r < H * H / NT; ++r) {
    const int e = tid + r * NT, a = e >> 6, b = e & 63;                          // W[a][b]
    const int n = transpose ? b : a, k = transpose ? a : b;
    const uint32_t off = (uint32_t)((k >> 5) * 8192) + sw128_off(n, k & 31);
    sts32(raw + off, w[r]);
    sts32(lo + off, lo_of(w[r]));
  }
}

// 3xTF32 product of two K-major image pairs: D[128 x 64] (+)= A . B^T over KSTEPS k-steps of 8.
// Blocks of 32 k are A_KB / B_KB bytes apart.  Small terms first, then the hi.hi pass.  The four base descriptors are
// built once; every MMA only adds a compile-time constant to the 14-bit address field.
template <int A_KB, int B_KB, int KSTEPS, int MM = 128>
__device__ __forceinline__ void issue_3xtf32(uint32_t tacc, uint32_t a_raw, uint32_t a_lo, uint32_t b_raw, uint32_t b_lo) {
  constexpr uint32_t idesc = make_idesc(64, MM);
  const uint64_t dar = make_desc(a_raw), dal = make_desc(a_lo), dbr = make_desc(b_raw), dbl = make_desc(b_lo);
#pragma unroll
  for (int ks = 0; ks < KSTEPS; ++ks) {
    const uint64_t oa = (uint64_t)(((ks >> 2) * A_KB + (ks & 3) * 32) >> 4), ob = (uint64_t)(((ks >> 2) * B_KB + (ks & 3) * 32) >> 4);
    umma_tf32(tacc, dal + oa, dbr + ob, idesc, ks ? 1u : 0u);
    umma_tf32(tacc, dar + oa, dbl + ob, idesc, 1u);
  }
#pragma unroll
  for (int ks = 0; ks < KSTEPS; ++ks) {
    const uint64_t oa = (uint64_t)(((ks >> 2) * A_KB + (ks & 3) * 32) >> 4), ob = (uint64_t)(((ks >> 2) * B_KB + (ks & 3) * 32) >> 4);
    umma_tf32(tacc, dar + oa, dbr + ob, idesc, 1u);
  }
}

// ------------------------------------------------------------------------------------------------ forward
template <int DP>
__global__ void __launch_bounds__(NT, 2) mlp3_tc_fwd_kernel(FwdP p) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem = (smem_u32(smem_raw) + 1023u) & ~1023u;   // 32-bit shared-window addresses from here on
  const uint32_t Wb_raw = smem;              // B[n = j][k = i] = W2[i][j]: 2 k-blocks x [64 rows][128 B]
  const uint32_t Wb_lo = smem + 16384;
  const uint32_t A_raw = smem + 32768;       // H1 [s][i]: 2 k-blocks x [128 rows][128 B]
  const uint32_t A_lo = smem + 65536;
  __shared__ __align__(16) float W1s[DP * H];
  __shared__ __align__(16) float b1s[H], b2s[H], W3s[H * MAXO], b3s[MAXO];
  __shared__ __align__(16) float part[TM * MAXO];
  __shared__ __align__(8) uint64_t bar;
  __shared__ uint32_t tmem_slot;

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int q = warp & 3, ch = warp >> 2, s = q * 32 + lane, c0 = ch * 32;
  const int g = blockIdx.y, o = p.o[g], D = p.D, ldw = p.G * H;

  if (tid == 0) { mbar_init(smem_u32(&bar), 1); asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
  if (warp == 0) tmem_alloc<64>(&tmem_slot);
  stage_weight(Wb_raw, Wb_lo, p.W2 + (size_t)g * H * H, true, tid);
  for (int e = tid; e < DP * H; e += NT) {
    const int k = e >> 6, c = e & 63;
    W1s[e] = k < D ? __ldg(p.W1 + (size_t)k * ldw + g * H + c) : 0.f;
  }
  for (int e = tid; e < H * MAXO; e += NT) {                // W3s [j][c]: one 16-byte read = 4 columns of output j
    const int j = e >> 6, c = e & 63;
    W3s[e] = j < o ? __ldg(p.W3[g] + c * o + j) : 0.f;
  }
  if (tid < H) { b1s[tid] = __ldg(p.b1 + g * H + tid); b2s[tid] = __ldg(p.b2 + g * H + tid); }
  if (tid < MAXO) b3s[tid] = tid < o ? __ldg(p.b3[g] + tid) : 0.f;
  fence_async_smem();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = tmem_slot;
  const uint32_t taddr = tmem + ((uint32_t)(q * 32) << 16) + (uint32_t)c0;

  uint32_t phase = 0;
  float x[DP];                               // this tile's X row; the next tile's is loaded under the MMA
  if ((int)blockIdx.x < p.nTiles)
    load_x_row<DP>(p.X + (size_t)(blockIdx.x * TM + s) * p.ldx, p.ldx, D, blockIdx.x * TM + s < p.M, x);
  for (int tile = blockIdx.x; tile < p.nTiles; tile += gridDim.x) {
    const int m0 = tile * TM;
    const bool live = m0 + s < p.M;
    float4* h1t = reinterpret_cast<float4*>(p.H1t + ((size_t)(g * p.nTiles + tile) * H + c0) * TM) + s;   // quad (c0/4 + j): + j*TM
    float4* h2t = reinterpret_cast<float4*>(p.H2t + ((size_t)(g * p.nTiles + tile) * H + c0) * TM) + s;
    // ---- layer 1 (K = D): registers, W1 by broadcast shared-memory reads ----
    float v[32];
    {
#pragma unroll
      for (int c = 0; c < 32; c += 4) {
        const float4 b = *reinterpret_cast<const float4*>(&b1s[c0 + c]);
        v[c] = b.x; v[c + 1] = b.y; v[c + 2] = b.z; v[c + 3] = b.w;
      }
#pragma unroll
      for (int k = 0; k < DP; ++k) {
        if (k < D) {
#pragma unroll
          for (int c = 0; c < 32; c += 4) {
            const float4 w = *reinterpret_cast<const float4*>(&W1s[k * H + c0 + c]);
            v[c] = fmaf(x[k], w.x, v[c]); v[c + 1] = fmaf(x[k], w.y, v[c + 1]);
            v[c + 2] = fmaf(x[k], w.z, v[c + 2]); v[c + 3] = fmaf(x[k], w.w, v[c + 3]);
          }
        }
      }
#pragma unroll
      for (int c = 0; c < 32; ++c) v[c] = tanh_fast(v[c]);
    }
#pragma unroll
    for (int j = 0; j < 8; ++j) __stcs(h1t + j * TM, make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]));   // warp = 512 contiguous bytes
    store_row_images(A_raw + ch * 16384, A_lo + ch * 16384, s, v);
    fence_async_smem();
    tc_fence_before();
    __syncthreads();
    // ---- layer 2 on the tensor core: Z2[s][j] = sum_i H1[s][i] W2[i][j] ----
    if (warp == 0) {
      tc_fence_after();
      if (elect_one()) {
        issue_3xtf32<16384, 8192, 8>(tmem, A_raw, A_lo, Wb_raw, Wb_lo);
        umma_commit(smem_u32(&bar));
      }
      __syncwarp();
    }
    {
      const int nt = tile + (int)gridDim.x;
      if (nt < p.nTiles) load_x_row<DP>(p.X + (size_t)(nt * TM + s) * p.ldx, p.ldx, D, nt * TM + s < p.M, x);
    }
    mbar_wait(smem_u32(&bar), phase);
    phase ^= 1;
    tc_fence_after();
    uint32_t z[32];
    tmem_ld32(taddr, z);
    // ---- epilogue: bias + tanh, H2 out, head layer (o <= 4) ----
    float po[MAXO] = {0.f, 0.f, 0.f, 0.f};
    float h2v[32];
#pragma unroll
    for (int c = 0; c < 32; ++c) {
      h2v[c] = tanh_fast(__uint_as_float(z[c]) + b2s[c0 + c]);
    }
#pragma unroll
    for (int j = 0; j < 8; ++j) __stcs(h2t + j * TM, make_float4(h2v[4 * j], h2v[4 * j + 1], h2v[4 * j + 2], h2v[4 * j + 3]));
    auto head = [&](auto oc) {               // only the o live outputs (o is CTA-uniform)
      constexpr int OC = decltype(oc)::value;
#pragma unroll
      for (int c = 0; c < 32; c += 4) {
#pragma unroll
        for (int j = 0; j < OC; ++j) {
          const float4 w = *reinterpret_cast<const float4*>(&W3s[j * H + c0 + c]);
          po[j] = fmaf(h2v[c + 3], w.w, fmaf(h2v[c + 2], w.z, fmaf(h2v[c + 1], w.y, fmaf(h2v[c], w.x, po[j]))));
        }
      }
    };
    switch (o) {
      case 1: head(std::integral_constant<int, 1>{}); break;
      case 2: head(std::integral_constant<int, 2>{}); break;
      case 3: head(std::integral_constant<int, 3>{}); break;
      default: head(std::integral_constant<int, 4>{}); break;
    }
    if (ch == 1) *reinterpret_cast<float4*>(&part[s * MAXO]) = make_float4(po[0], po[1], po[2], po[3]);
    tc_fence_before();                       // the tcgen05.ld above is ordered before the next tile's MMAs
    __syncthreads();
    if (ch == 0 && live) {
      const float4 t = *reinterpret_cast<const float4*>(&part[s * MAXO]);
      const float r[MAXO] = {po[0] + t.x + b3s[0], po[1] + t.y + b3s[1], po[2] + t.z + b3s[2], po[3] + t.w + b3s[3]};
      float* dst = p.out[g] + (size_t)(m0 + s) * o;
#pragma unroll
      for (int j = 0; j < MAXO; ++j)
        if (j < o) dst[j] = r[j];
    }
    // `part` is rewritten only after the next tile's first barrier; the images only after this barrier + the MMA wait
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) { tc_fence_after(); tmem_dealloc<64>(tmem); }
}

// ------------------------------------------------------------------------------------------------ forward, v2
// Round 2: BOTH dense layers of the forward on the tensor pipe, A operands in TENSOR MEMORY (tools/umma_probe3.cu):
//   * layer 1: Z1 = [X | 1] [W1 ; b1] -- the thread that owns a sample writes its X row (raw | lo) and a ones column with
//     tcgen05.st; B = a small K-major image of [W1 ; b1]^T staged once per CTA.  (K = DP + 8; v1 spent 256 FMAs and 72
//     shared-memory reads per thread and tile here.)
//   * layer 2: H1 (raw | lo) goes back into tensor memory with tcgen05.st -- no shared-memory images, no swizzle
//     arithmetic, and the MMA reads only W2 from shared memory (32 instead of 48 cycles at M 128, N 64).
// 48 KB of shared memory and 256 TMEM columns per CTA: two CTAs per SM, one covers the other's MMA round trips.
namespace f2 {
constexpr uint32_t ACC = 0, A2_RAW = 64, A2_LO = 128, A1 = 192;      // tensor-memory columns (A1: raw K1 columns, then lo)
}

template <int DP>
__global__ void __launch_bounds__(NT, 2) mlp3_tc_fwd2_kernel(FwdP p) {
  using namespace f2;
  constexpr int K1 = DP + 8;                      // layer-1 reduction: D inputs (padded to DP) | ones | 7 zeros
  static_assert(2 * K1 <= 64, "layer-1 operand must fit its tensor-memory columns");
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t W2_raw = smem, W2_lo = smem + 16384;            // B[n = j][k = i] = W2[i][j]: 2 k-blocks x [64 rows][128 B]
  const uint32_t W1_raw = smem + 32768, W1_lo = smem + 40960;    // B[n = i][k] = W1[k][i] (k < D), b1[i] (k == DP): [64 rows][128 B]
  __shared__ __align__(16) float b2s[H], W3s[H * MAXO], b3s[MAXO];
  __shared__ __align__(16) float part[TM * MAXO];
  __shared__ __align__(8) uint64_t bar;
  __shared__ uint32_t tmem_slot;

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int q = warp & 3, ch = warp >> 2, s = q * 32 + lane, c0 = ch * 32;
  const int g = blockIdx.y, o = p.o[g], D = p.D, ldw = p.G * H;

  if (tid == 0) { mbar_init(smem_u32(&bar), 1); asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
  if (warp == 0) tmem_alloc<256>(&tmem_slot);
  stage_weight(W2_raw, W2_lo, p.W2 + (size_t)g * H * H, true, tid);
  for (int e = tid; e < H * 32; e += NT) {                   // the whole 128-byte rows (unused k columns = 0)
    const int n = e >> 5, k = e & 31;
    float w = 0.f;
    if (k < D) w = __ldg(p.W1 + (size_t)k * ldw + g * H + n);
    else if (k == DP) w = __ldg(p.b1 + g * H + n);
    const uint32_t off = sw128_off(n, k);
    sts32(W1_raw + off, w);
    sts32(W1_lo + off, lo_of(w));
  }
  for (int e = tid; e < H * MAXO; e += NT) {                 // W3s [j][c]: one 16-byte read = 4 columns of output j
    const int j = e >> 6, c = e & 63;
    W3s[e] = j < o ? __ldg(p.W3[g] + c * o + j) : 0.f;
  }
  if (tid < H) b2s[tid] = __ldg(p.b2 + g * H + tid);
  if (tid < MAXO) b3s[tid] = tid < o ? __ldg(p.b3[g] + tid) : 0.f;
  fence_async_smem();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = tmem_slot;
  const uint32_t tlane = tmem + ((uint32_t)(q * 32) << 16);

  uint32_t phase = 0;
  float x[DP];                                   // this tile's X row; the next tile's is loaded under the MMAs
  if ((int)blockIdx.x < p.nTiles)
    load_x_row<DP>(p.X + (size_t)(blockIdx.x * TM + s) * p.ldx, p.ldx, D, blockIdx.x * TM + s < p.M, x);
  for (int tile = blockIdx.x; tile < p.nTiles; tile += gridDim.x) {
    const int m0 = tile * TM;
    const bool live = m0 + s < p.M;
    float4* h1t = reinterpret_cast<float4*>(p.H1t + ((size_t)(g * p.nTiles + tile) * H + c0) * TM) + s;   // quad (c0/4 + j): + j*TM
    float4* h2t = reinterpret_cast<float4*>(p.H2t + ((size_t)(g * p.nTiles + tile) * H + c0) * TM) + s;
    // ---- layer 1 operand: [x | 1 | 0] raw (column half 0) and its lo part (column half 1) -> tensor memory ----
    {
#pragma unroll
      for (int k0 = 0; k0 < K1; k0 += 8) {
        uint32_t u[8];
#pragma unroll
        for (int k = 0; k < 8; ++k) {
          const int kk = k0 + k;
          const float v = kk < DP ? x[kk < DP ? kk : 0] : (kk == DP ? 1.f : 0.f);
          u[k] = __float_as_uint(ch == 0 ? v : lo_of(v));
        }
        tmem_st8(tlane + A1 + (uint32_t)(ch * K1 + k0), u);
      }
      tmem_st_wait();
    }
    tc_fence_before();
    __syncthreads();                         // [A] operand complete; every thread has read the previous tile's accumulator
    if (warp == 0) {
      tc_fence_after();
      if (elect_one()) {
        constexpr uint32_t id = make_idesc_full(128, 64, 0, 0);
        const uint64_t dr = make_desc(W1_raw), dl = make_desc(W1_lo);
#pragma unroll
        for (int ks = 0; ks < K1 / 8; ++ks) {
          umma_tf32_ts(tmem + ACC, tmem + A1 + K1 + ks * 8, dr + (uint64_t)(ks * 2), id, ks ? 1u : 0u);
          umma_tf32_ts(tmem + ACC, tmem + A1 + ks * 8, dl + (uint64_t)(ks * 2), id, 1u);
        }
#pragma unroll
        for (int ks = 0; ks < K1 / 8; ++ks) umma_tf32_ts(tmem + ACC, tmem + A1 + ks * 8, dr + (uint64_t)(ks * 2), id, 1u);
        umma_commit(smem_u32(&bar));
      }
      __syncwarp();
    }
    {
      const int nt = tile + (int)gridDim.x;
      if (nt < p.nTiles) load_x_row<DP>(p.X + (size_t)(nt * TM + s) * p.ldx, p.ldx, D, nt * TM + s < p.M, x);
    }
    mbar_wait(smem_u32(&bar), phase);
    phase ^= 1;
    tc_fence_after();
    // ---- H1 = tanh(Z1) (bias came through the ones column): out to HBM, raw | lo back into tensor memory ----
    float v[32];
    {
      uint32_t z[32];
      tmem_ld32(tlane + ACC + c0, z);
#pragma unroll
      for (int c = 0; c < 32; ++c) v[c] = tanh_fast(__uint_as_float(z[c]));
    }
#pragma unroll
    for (int j = 0; j < 8; ++j) __stcs(h1t + j * TM, make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]));   // warp = 512 contiguous bytes
#pragma unroll
    for (int hh = 0; hh < 32; hh += 16) {
      uint32_t u[16];
#pragma unroll
      for (int c = 0; c < 16; ++c) u[c] = __float_as_uint(v[hh + c]);
      tmem_st16(tlane + A2_RAW + c0 + hh, u);
#pragma unroll
      for (int c = 0; c < 16; ++c) u[c] = __float_as_uint(lo_of(v[hh + c]));
      tmem_st16(tlane + A2_LO + c0 + hh, u);
    }
    tmem_st_wait();
    tc_fence_before();
    __syncthreads();                         // [B] layer-2 operand complete; Z1 read by everyone
    // ---- layer 2 on the tensor core: Z2[s][j] = sum_i H1[s][i] W2[i][j] ----
    if (warp == 0) {
      tc_fence_after();
      if (elect_one()) {
        constexpr uint32_t id = make_idesc_full(128, 64, 0, 0);
        const uint64_t dr = make_desc(W2_raw), dl = make_desc(W2_lo);
#pragma unroll
        for (int ks = 0; ks < 8; ++ks) {
          const uint64_t ob = (uint64_t)(((ks >> 2) * 8192 + (ks & 3) * 32) >> 4);
          umma_tf32_ts(tmem + ACC, tmem + A2_LO + ks * 8, dr + ob, id, ks ? 1u : 0u);
          umma_tf32_ts(tmem + ACC, tmem + A2_RAW + ks * 8, dl + ob, id, 1u);
        }
#pragma unroll
        for (int ks = 0; ks < 8; ++ks) {
          const uint64_t ob = (uint64_t)(((ks >> 2) * 8192 + (ks & 3) * 32) >> 4);
          umma_tf32_ts(tmem + ACC, tmem + A2_RAW + ks * 8, dr + ob, id, 1u);
        }
        umma_commit(smem_u32(&bar));
      }
      __syncwarp();
    }
    mbar_wait(smem_u32(&bar), phase);
    phase ^= 1;
    tc_fence_after();
    // ---- epilogue: bias + tanh, H2 out, head layer (o <= 4) ----
    float po[MAXO] = {0.f, 0.f, 0.f, 0.f};
    {
      uint32_t z[32];
      tmem_ld32(tlane + ACC + c0, z);
#pragma unroll
      for (int c = 0; c < 32; ++c) v[c] = tanh_fast(__uint_as_float(z[c]) + b2s[c0 + c]);
    }
#pragma unroll
    for (int j = 0; j < 8; ++j) __stcs(h2t + j * TM, make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]));
    auto head = [&](auto oc) {               // only the o live outputs (o is CTA-uniform)
      constexpr int OC = decltype(oc)::value;
#pragma unroll
      for (int c = 0; c < 32; c += 4) {
#pragma unroll
        for (int j = 0; j < OC; ++j) {
          const float4 w = *reinterpret_cast<const float4*>(&W3s[j * H + c0 + c]);
          po[j] = fmaf(v[c + 3], w.w, fmaf(v[c + 2], w.z, fmaf(v[c + 1], w.y, fmaf(v[c], w.x, po[j]))));
        }
      }
    };
    switch (o) {
      case 1: head(std::integral_constant<int, 1>{}); break;
      case 2: head(std::integral_constant<int, 2>{}); break;
      case 3: head(std::integral_constant<int, 3>{}); break;
      default: head(std::integral_constant<int, 4>{}); break;
    }
    if (ch == 1) *reinterpret_cast<float4*>(&part[s * MAXO]) = make_float4(po[0], po[1], po[2], po[3]);
    tc_fence_before();                       // the tcgen05.ld above is ordered before the next tile's MMAs
    __syncthreads();                         // [C]
    if (ch == 0 && live) {
      const float4 t = *reinterpret_cast<const float4*>(&part[s * MAXO]);
      const float r[MAXO] = {po[0] + t.x + b3s[0], po[1] + t.y + b3s[1], po[2] + t.z + b3s[2], po[3] + t.w + b3s[3]};
      float* dst = p.out[g] + (size_t)(m0 + s) * o;
#pragma unroll
      for (int j = 0; j < MAXO; ++j)
        if (j < o) dst[j] = r[j];
    }
    // `part` is rewritten only after the next tile's barriers [A] and [B]
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) { tc_fence_after(); tmem_dealloc<256>(tmem); }
}

// ------------------------------------------------------------------------------------------------ backward
struct BwdP {
  const float* X; int ldx; int M, D, G, nTiles;
  const float* W2; const float* W3[MAXG]; int o[MAXG];
  const float* H1t; const float* H2t;
  const float* dOut[MAXG];
  const float* vh_v[MAXG]; const float* vh_ov[MAXG]; const float* vh_R[MAXG]; const double* vh_branch[MAXG];
  float vh_scale[MAXG]; float vh_clip; float vh_Bt;
  float* ws2;        // [G][nCta][H*H]   dW2 partials
  float* wsr;        // [G][nCta][RS]    dW1 | db1 | db2 | dW3 | db3 partials
  int RS;
};

// byte offset of element (s, c) of the fp32 staging tile S [128][64] (16-byte chunks XOR-swizzled by the row)
__device__ __forceinline__ uint32_t stage_off(int s, int c) { return (uint32_t)(s * 256 + ((((c >> 2) ^ (s & 7)) << 4) | ((c & 3) << 2))); }

template <int CW>
__device__ __forceinline__ void tmem_ld_cw(uint32_t taddr, uint32_t (&v)[CW]) {
  if constexpr (CW == 32) tmem_ld32_nowait(taddr, v); else tmem_ld16_nowait(taddr, v);
  tmem_ld_wait();
}
// v[CW] = CW consecutive columns (c0 .. c0+CW-1) of row s -> raw and lo K-major images (k-block c0/32)
template <int CW>
__device__ __forceinline__ void store_row_images_cw(uint32_t raw, uint32_t lo, int s, int c0, const float (&v)[CW]) {
  const uint32_t row = (uint32_t)((c0 >> 5) * 16384 + s * 128), x = (uint32_t)(s & 7), cb = (uint32_t)((c0 & 31) >> 2);
#pragma unroll
  for (int j = 0; j < CW / 4; ++j) {
    const uint32_t off = row + (((cb + j) ^ x) << 4);
    sts128(raw + off, v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
    sts128(lo + off, lo_of(v[4 * j]), lo_of(v[4 * j + 1]), lo_of(v[4 * j + 2]), lo_of(v[4 * j + 3]));
  }
}
// v[CW] = elements (row r0+c, column s) of a transposed image with 64-row k-blocks (block = s/32); r0 % 8 == 0
template <int CW>
__device__ __forceinline__ void store_col_images_cw(uint32_t raw, uint32_t lo_delta, int r0, int s, const float (&v)[CW]) {
  const uint32_t l = (uint32_t)(s & 31);
  const uint32_t base = raw + (uint32_t)((s >> 5) * 8192 + r0 * 128) + ((l & 3) << 2) + ((l >> 2) << 4);
#pragma unroll
  for (int c = 0; c < CW; ++c) {
    const uint32_t a = (base ^ (uint32_t)((c & 7) << 4)) + (uint32_t)(c * 128);
    sts32(a, v[c]);
    sts32(a + lo_delta, lo_of(v[c]));
  }
}

// Backward kernel: 128 x (64 / CW) compute threads -- thread = (sample s, CW hidden columns).  The shipped configuration is
// CW = 32, MMAW = false (8 warps, 255 registers, warp 0 issues the MMAs after the publishing barrier): 97 us at C2.
// The other instantiations are measured alternatives kept behind PPX_MLP_TC_CW=16 / PPX_MLP_TC_MMAW=1
// (profiles/mlp_tc_r01d.md): 16 compute warps with 16 columns each (105 us: the kernel is not bound by warps in flight),
// and a dedicated MMA-issue warp that waits on "operands ready" mbarriers (a tcgen05.mma stalls its issuing thread for
// about its own duration -- 48 cycles at M=128,N=64 -- but 9 or 17 warps per CTA put 3 or 5 warps on one of the four
// register files: 168 / 96 registers, spills, 130-155 us).
template <int DP, int CW, bool MMAW>
__global__ void __launch_bounds__(128 * (64 / CW) + (MMAW ? 32 : 0), 1) mlp3_tc_bwd_kernel(BwdP p) {
  constexpr int NCQ = H / CW, NTC = TM * NCQ, NSG = NTC / H, SPG = TM / NSG;   // column groups, compute threads, sample groups
  constexpr int XPT = (TM * DP) / NTC;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem = (smem_u32(smem_raw) + 1023u) & ~1023u;   // 32-bit shared-window addresses from here on
  const uint32_t W_raw = smem;               // B of GEMM 2: B[n = i][k = j] = W2[i][j]: 2 k-blocks x [64][128 B]
  const uint32_t W_lo = smem + 16384;
  const uint32_t V_raw = smem + 32768;       // A of GEMM 1: H1^T [i][s]: 4 k-blocks x [64][128 B]
  const uint32_t V_lo = smem + 65536;
  const uint32_t U_raw = smem + 98304;       // phase 1: dP2 [s][j] (A of GEMM 2, 2 k-blocks x [128][128 B]);
  const uint32_t U_lo = smem + 131072;       // phase 2: dP2^T [j][s] (B of GEMM 1, 4 k-blocks x [64][128 B])
  const uint32_t S = smem + 163840;          // fp32 staging [128][64]: H2, then dP1
  const uint32_t Xs = smem + 196608;         // [TM][DP] fp32
  __shared__ __align__(16) float W3s[MAXO * H];          // [j][c]
  __shared__ __align__(16) float dOs[TM * MAXO];
  __shared__ __align__(8) uint64_t bars[4];
  __shared__ uint32_t tmem_slot;

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int g = blockIdx.y, o = p.o[g], D = p.D;
  const uint32_t barG2 = smem_u32(&bars[0]), barG1 = smem_u32(&bars[1]);     // MMA completion (tcgen05.commit)
  const uint32_t opsG2 = smem_u32(&bars[2]), opsG1 = smem_u32(&bars[3]);     // operands ready (one arrive per compute warp)
  auto bar_compute = [] { asm volatile("bar.sync 1, %0;" ::"n"(NTC) : "memory"); };

  if (tid == 0) {
    mbar_init(barG2, 1); mbar_init(barG1, 1); mbar_init(opsG2, NTC / 32); mbar_init(opsG1, NTC / 32);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 0) tmem_alloc<128>(&tmem_slot);
  if (tid < NTC) {
    float w[H * H / NTC];
#pragma unroll
    for (int r = 0; r < H * H / NTC; ++r) w[r] = __ldg(p.W2 + (size_t)g * H * H + tid + r * NTC);
#pragma unroll
    for (int r = 0; r < H * H / NTC; ++r) {
      const int e = tid + r * NTC, i = e >> 6, j = e & 63;
      const uint32_t off = (uint32_t)((j >> 5) * 8192) + sw128_off(i, j & 31);
      sts32(W_raw + off, w[r]);
      sts32(W_lo + off, lo_of(w[r]));
    }
    for (int e = tid; e < MAXO * H; e += NTC) {
      const int j = e >> 6, c = e & 63;
      W3s[e] = j < o ? __ldg(p.W3[g] + c * o + j) : 0.f;
    }
  }
  fence_async_smem();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = tmem_slot;

  if (MMAW && warp == NTC / 32) {
    // ------------------------------------------------ MMA warp ------------------------------------------------
    int it = 0;
    for (int tile = blockIdx.x; tile < p.nTiles; tile += gridDim.x, ++it) {
      const uint32_t ph = (uint32_t)(it & 1);
      mbar_wait(opsG2, ph);                   // dP2 images written (and the previous GEMM-2 accumulator read)
      tc_fence_after();
      if (elect_one()) {
        issue_3xtf32<16384, 8192, 8>(tmem, U_raw, U_lo, W_raw, W_lo);
        umma_commit(barG2);
      }
      __syncwarp();
      mbar_wait(opsG1, ph);                   // H1^T and dP2^T images written, previous dW2 accumulator drained
      tc_fence_after();
      if (elect_one()) {
        issue_3xtf32<8192, 8192, 16, 64>(tmem + 64, V_raw, V_lo, U_raw, U_lo);
        umma_commit(barG1);
      }
      __syncwarp();
    }
  } else {
    // ------------------------------------------------ compute warps ------------------------------------------------
    const int q = warp & 3, cq = warp >> 2, s = q * 32 + lane, c0 = cq * CW;
    const int tc = tid & 63, sg = tid >> 6;   // thin-reduction mapping: column tc, samples sg*SPG .. +SPG-1
    const uint32_t taddr = tmem + ((uint32_t)(q * 32) << 16) + (uint32_t)c0;
    // this thread's image writes -> visible to the tensor core; then either one arrive per warp for the MMA warp, or
    // (no MMA warp) a barrier after which warp 0 issues the GEMM itself
    auto ops_ready = [&](uint32_t bar, int which) {
      fence_async_smem();
      tc_fence_before();
      if constexpr (MMAW) {
        __syncwarp();
        if (lane == 0) mbar_arrive(bar);
      } else {
        bar_compute();
        if (warp == 0) {
          tc_fence_after();
          if (elect_one()) {
            if (which == 2) { issue_3xtf32<16384, 8192, 8>(tmem, U_raw, U_lo, W_raw, W_lo); umma_commit(barG2); }
            else { issue_3xtf32<8192, 8192, 16, 64>(tmem + 64, V_raw, V_lo, U_raw, U_lo); umma_commit(barG1); }
          }
          __syncwarp();
        }
      }
    };

    float dW2acc[CW];                         // lanes < 16: dW2[i = q*16+lane][c0 .. c0+CW-1]
    float a_dW1[DP], a_db1 = 0.f, a_db2 = 0.f, a_dW3[MAXO] = {0.f, 0.f, 0.f, 0.f}, a_db3 = 0.f;
#pragma unroll
    for (int c = 0; c < CW; ++c) dW2acc[c] = 0.f;
#pragma unroll
    for (int k = 0; k < DP; ++k) a_dW1[k] = 0.f;

    float h1[CW], h2[CW], xpre[XPT];
    float4 dpre = make_float4(0.f, 0.f, 0.f, 0.f);
      auto prefetch = [&](int tile) {
      const int m0 = tile * TM;
      const float4* h1t = reinterpret_cast<const float4*>(p.H1t + ((size_t)(g * p.nTiles + tile) * H + c0) * TM) + s;
      const float4* h2t = reinterpret_cast<const float4*>(p.H2t + ((size_t)(g * p.nTiles + tile) * H + c0) * TM) + s;
#pragma unroll
      for (int j = 0; j < CW / 4; ++j) {
        const float4 a = ld_stream4(h1t + j * TM), b = ld_stream4(h2t + j * TM);
        h1[4 * j] = a.x; h1[4 * j + 1] = a.y; h1[4 * j + 2] = a.z; h1[4 * j + 3] = a.w;
        h2[4 * j] = b.x; h2[4 * j + 1] = b.y; h2[4 * j + 2] = b.z; h2[4 * j + 3] = b.w;
      }
#pragma unroll
      for (int r = 0; r < XPT; ++r) {                        // Xs element e = tid + r*NTC: row e / DP, column e % DP
        const int e = tid + r * NTC, row = e / DP, k = e % DP;
        xpre[r] = (m0 + row < p.M && k < D) ? __ldg(p.X + (size_t)(m0 + row) * p.ldx + k) : 0.f;
      }
      {                                                      // output gradient of this thread's row s (every column group loads it: dP2 then needs no barrier)
        const int b = m0 + s;
        float d[MAXO] = {0.f, 0.f, 0.f, 0.f};
        if (b < p.M) {
          if (p.vh_v[g] != nullptr) {                        // o == 1 (checked on the host); same formula as mlp_fused.cu
            const float w1 = (float)p.vh_branch[g][0], w2 = (float)p.vh_branch[g][1], clip = p.vh_clip;
            const float v = ld_stream(p.vh_v[g] + b), ov = ld_stream(p.vh_ov[g] + b), R = ld_stream(p.vh_R[g] + b);
            const float dd = v - ov;
            const float vc = ov + fminf(fmaxf(dd, -clip), clip);
            const float pass = (dd >= -clip && dd <= clip) ? 1.f : 0.f;
            const float gv = w1 * (-2.f * (R - v)) + w2 * (-2.f * (R - vc)) * pass;
            d[0] = p.vh_scale[g] * gv / p.vh_Bt;
          } else {
#pragma unroll
            for (int j = 0; j < MAXO; ++j)
              if (j < o) d[j] = ld_stream(p.dOut[g] + (size_t)b * o + j);
          }
        }
        dpre = make_float4(d[0], d[1], d[2], d[3]);
      }
    };

    int it = 0;
    if ((int)blockIdx.x < p.nTiles) prefetch(blockIdx.x);
    for (int tile = blockIdx.x; tile < p.nTiles; tile += gridDim.x, ++it) {
      const uint32_t ph = (uint32_t)(it & 1);
      // ---- T1: publish X, dOut and H2 (staging tile S) ----
#pragma unroll
      for (int r = 0; r < XPT; ++r) sts32(Xs + (uint32_t)(tid + r * NTC) * 4, xpre[r]);
      if (c0 == 0) *reinterpret_cast<float4*>(&dOs[s * MAXO]) = dpre;
#pragma unroll
      for (int j = 0; j < CW / 4; ++j)
        sts128(S + stage_off(s, c0 + 4 * j), h2[4 * j], h2[4 * j + 1], h2[4 * j + 2], h2[4 * j + 3]);
      // (no barrier: T2 works from registers; X / dOut / H2 are published to the thin reductions by [B2])
      // ---- T2: dP2 = (dOut W3^T)(1 - H2^2) -> K-major images (phase 1 of U) -> GEMM 2 ----
      float dp2[CW];
      {
        const float dj[MAXO] = {dpre.x, dpre.y, dpre.z, dpre.w};
#pragma unroll
        for (int c = 0; c < CW; c += 4) {
          float4 a = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
          for (int j = 0; j < MAXO; ++j)
            if (j < o) {                      // CTA-uniform
              const float4 w = *reinterpret_cast<const float4*>(&W3s[j * H + c0 + c]);
              a.x = fmaf(dj[j], w.x, a.x); a.y = fmaf(dj[j], w.y, a.y); a.z = fmaf(dj[j], w.z, a.z); a.w = fmaf(dj[j], w.w, a.w);
            }
          dp2[c] = a.x * (1.f - h2[c] * h2[c]); dp2[c + 1] = a.y * (1.f - h2[c + 1] * h2[c + 1]);
          dp2[c + 2] = a.z * (1.f - h2[c + 2] * h2[c + 2]); dp2[c + 3] = a.w * (1.f - h2[c + 3] * h2[c + 3]);
        }
      }
      if (it > 0) {                           // GEMM 1 of the previous tile has finished reading U and V
        mbar_wait(barG1, ph ^ 1);
        tc_fence_after();
        {                                     // ... and its dW2 accumulator is drained (UMMA M = 64: row i sits in lane i%16 of quarter i/16)
          uint32_t z[CW];
          tmem_ld_cw<CW>(taddr + 64, z);
#pragma unroll
          for (int c = 0; c < CW; ++c) dW2acc[c] += __uint_as_float(z[c]);
        }
      }
      store_row_images_cw<CW>(U_raw, U_lo, s, c0, dp2);
      ops_ready(opsG2, 2);
      if constexpr (MMAW) bar_compute();      // [B2] X / dOut / H2 published to the thin reductions
      // ---- T3 (under GEMM 2): H1^T images; dW3 / db3 sums over this thread's SPG samples ----
      store_col_images_cw<CW>(V_raw, 32768u, c0, s, h1);
      {
        float t3[MAXO] = {0.f, 0.f, 0.f, 0.f};
        // element (ss = sg*SPG + r, tc): the row swizzle (ss & 7) == (r & 7) is an XOR of the base with a constant
        const uint32_t sS = S + (uint32_t)(sg * SPG * 256) + (uint32_t)(((tc >> 2) << 4) | ((tc & 3) << 2));
#pragma unroll
        for (int r = 0; r < SPG; ++r) {
          const float hv = lds32((sS ^ (uint32_t)((r & 7) << 4)) + (uint32_t)(r * 256));
          const float4 d = *reinterpret_cast<const float4*>(&dOs[(sg * SPG + r) * MAXO]);
          t3[0] = fmaf(hv, d.x, t3[0]); t3[1] = fmaf(hv, d.y, t3[1]); t3[2] = fmaf(hv, d.z, t3[2]); t3[3] = fmaf(hv, d.w, t3[3]);
        }
#pragma unroll
        for (int j = 0; j < MAXO; ++j) a_dW3[j] += t3[j];
        if (tc < MAXO) {                      // db3[j = tc]: one column of dOut
          float tb = 0.f;
#pragma unroll
          for (int r = 0; r < SPG; ++r) tb += dOs[(sg * SPG + r) * MAXO + tc];
          a_db3 += tb;
        }
      }
      bar_compute();                          // [B3] every read of S (H2) done before dP1 overwrites it
      // ---- T4: dP1 = (dP2 W2^T)(1 - H1^2); transposed dP2 images (phase 2 of U) -> GEMM 1 ----
      mbar_wait(barG2, ph);
      tc_fence_after();
      {
        uint32_t z[CW];
        tmem_ld_cw<CW>(taddr, z);
#pragma unroll
        for (int j = 0; j < CW / 4; ++j) {
          float4 v;
          v.x = __uint_as_float(z[4 * j]) * (1.f - h1[4 * j] * h1[4 * j]);
          v.y = __uint_as_float(z[4 * j + 1]) * (1.f - h1[4 * j + 1] * h1[4 * j + 1]);
          v.z = __uint_as_float(z[4 * j + 2]) * (1.f - h1[4 * j + 2] * h1[4 * j + 2]);
          v.w = __uint_as_float(z[4 * j + 3]) * (1.f - h1[4 * j + 3] * h1[4 * j + 3]);
          sts128(S + stage_off(s, c0 + 4 * j), v.x, v.y, v.z, v.w);
        }
      }
      store_col_images_cw<CW>(U_raw, 32768u, c0, s, dp2);   // GEMM 2 has finished reading the phase-1 images
      ops_ready(opsG1, 1);
      if constexpr (MMAW) bar_compute();      // [B4] dP1 (S) and the dP2^T image published to the thin reductions
      // ---- T5 (under GEMM 1): next tile's loads in flight; dW1 / db1 / db2 sums ----
      if (tile + (int)gridDim.x < p.nTiles) prefetch(tile + gridDim.x);
      {
        float t1[DP], tb = 0.f, t2 = 0.f;
#pragma unroll
        for (int k = 0; k < DP; ++k) t1[k] = 0.f;
        const uint32_t sS = S + (uint32_t)(sg * SPG * 256) + (uint32_t)(((tc >> 2) << 4) | ((tc & 3) << 2));
        const uint32_t sX = Xs + (uint32_t)(sg * SPG * DP * 4);
#pragma unroll
        for (int r = 0; r < SPG; ++r) {
          const float dv = lds32((sS ^ (uint32_t)((r & 7) << 4)) + (uint32_t)(r * 256));
          tb += dv;
#pragma unroll
          for (int k = 0; k < DP; k += 4) {
            const float4 x = lds128(sX + (uint32_t)((r * DP + k) * 4));
            t1[k] = fmaf(dv, x.x, t1[k]); t1[k + 1] = fmaf(dv, x.y, t1[k + 1]);
            t1[k + 2] = fmaf(dv, x.z, t1[k + 2]); t1[k + 3] = fmaf(dv, x.w, t1[k + 3]);
          }
        }
        // db2[tc] += sum over this group's samples of dP2: row tc of the transposed raw image, SPG consecutive samples
        const uint32_t uR = U_raw + (uint32_t)(((sg * SPG) >> 5) * 8192 + tc * 128);
        const uint32_t m0 = (uint32_t)(((sg * SPG) & 31) >> 2), x7 = (uint32_t)(tc & 7);
#pragma unroll
        for (int m = 0; m < SPG / 4; ++m) {
          const float4 v = lds128(uR + (((m0 + m) ^ x7) << 4));
          t2 += (v.x + v.y) + (v.z + v.w);
        }
#pragma unroll
        for (int k = 0; k < DP; ++k) a_dW1[k] += t1[k];
        a_db1 += tb;
        a_db2 += t2;
      }
      bar_compute();                          // [B5] S, Xs, dOs free for the next tile
    }
    // ---- the last tile's dW2 contribution ----
    if (it > 0) {
      mbar_wait(barG1, (uint32_t)((it - 1) & 1));
      tc_fence_after();
      {
        uint32_t z[CW];
        tmem_ld_cw<CW>(taddr + 64, z);
#pragma unroll
        for (int c = 0; c < CW; ++c) dW2acc[c] += __uint_as_float(z[c]);
      }
    }
    // ---- one partial per CTA: dW2 straight from registers; the thin sums of the sample groups combined in order ----
    float* w2 = p.ws2 + (size_t)(g * gridDim.x + blockIdx.x) * H * H;
    if (lane < 16) {
#pragma unroll
      for (int c = 0; c < CW; c += 4)
        *reinterpret_cast<float4*>(&w2[(q * 16 + lane) * H + c0 + c]) = make_float4(dW2acc[c], dW2acc[c + 1], dW2acc[c + 2], dW2acc[c + 3]);
    }
    constexpr int NQ = DP + 3 + MAXO;         // per (column, group): dW1[DP] | db1 | db2 | dW3[4] | db3 (column j holds db3[j])
    static_assert(NSG * NQ * H * 4 <= 98304, "reduction scratch must fit U + S");
    const uint32_t red = U_raw;               // [NSG groups][NQ][64] fp32 over U (and S for DP = 32)
    {
      const uint32_t r = red + (uint32_t)(sg * NQ * H + tc) * 4;
#pragma unroll
      for (int k = 0; k < DP; ++k) sts32(r + k * H * 4, a_dW1[k]);
      sts32(r + DP * H * 4, a_db1); sts32(r + (DP + 1) * H * 4, a_db2);
#pragma unroll
      for (int j = 0; j < MAXO; ++j) sts32(r + (DP + 2 + j) * H * 4, a_dW3[j]);
      sts32(r + (DP + 2 + MAXO) * H * 4, a_db3);
    }
    bar_compute();
    float* wr = p.wsr + ((size_t)g * gridDim.x + blockIdx.x) * p.RS;
    const int offb1 = D * H, offb2 = offb1 + H, offW3 = offb2 + H, offb3 = offW3 + H * o;
    for (int e = tid; e < NQ * H; e += NTC) {
      const int n = e >> 6, c = e & 63;
      const uint32_t a = red + (uint32_t)e * 4;
      float v = lds32(a);
#pragma unroll
      for (int k = 1; k < NSG; ++k) v += lds32(a + (uint32_t)(k * NQ * H * 4));
      if (n < DP) { if (n < D) wr[n * H + c] = v; }
      else if (n == DP) wr[offb1 + c] = v;
      else if (n == DP + 1) wr[offb2 + c] = v;
      else if (n < DP + 2 + MAXO) { const int j = n - DP - 2; if (j < o) wr[offW3 + c * o + j] = v; }
      else { if (c < o) wr[offb3 + c] = v; }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) { tc_fence_after(); tmem_dealloc<128>(tmem); }
}


// ------------------------------------------------------------------------------------------------ backward, v2
// Round-2 restructure (VERDICT r1 item 1).  v1 above spends ~1900 instructions per thread and tile, most of them on
// (a) the transposed scalar-store images of H1 and dP2 that the weight-gradient GEMM needs, (b) the thin reductions
// dW1 / db1 / db2 / dW3 on the FMA pipe behind CTA barriers, and its MMA-issuing warp is a ~2700-cycle straggler at every
// barrier (a tcgen05.mma blocks its issuing thread for about its own duration).  v2 (operand forms and MMA costs probed
// by tools/umma_probe3.cu / umma_probe4.cu):
//   * GEMM 2 (dP1 = dP2 W2^T) takes its A operand from TENSOR MEMORY: the owning threads write their 32 dP2 columns
//     (raw | lo) with two tcgen05.st -- no shared-memory image, no swizzle arithmetic, and the MMA is faster (32 vs 48
//     cycles at M 128, N 64);
//   * GEMM 1 (dW2 += H1^T dP2, reduction over the samples) reads MN-major SWIZZLE_128B_BASE32B images: a thread's 32
//     columns of a sample ARE 128 contiguous bytes of that layout, so the images are 16-byte vector stores;
//   * dW1, db1 and db2 come off the tensor pipe as well: GEMM 3 = [dP1 | dP2]^T [X | 1] (M = 128: the dP1 image takes
//     the place of the H1 image once GEMM 1 has read it and sits next to the dP2 image; B = a small K-major image of
//     X^T with a ones row, N = DP + 8);
//   * dW3 / db3 (64 x o numbers) are reduced inside each warp with a transposing shuffle network and kept in one
//     register per output across the tiles -- with that the tile loop has NO CTA barrier: a compute warp only meets the
//     MMA warp, through mbarriers;
//   * a dedicated MMA warp (warp 8; its warpgroup gives its registers to the 8 compute warps) issues the three GEMMs
//     of a tile behind "operands ready" mbarriers, so no compute warp ever stalls on an MMA.
namespace v2 {
// shared-memory bytes from the 1024-aligned base; the raw images of V and Q (and their lo images) are adjacent so that
// GEMM 3 reads [V ; Q] as one M = 128 MN-major operand (4 blocks of 32 rows, 16 KB apart)
constexpr uint32_t ACC2 = 0, ACC1 = 64, ACC3 = 128, A_RAW = 192, A_LO = 256;     // tensor-memory columns
constexpr uint32_t W_RAW = 0, W_LO = 16384, V_RAW = 32768, Q_RAW = 65536, LO_DELTA = 65536, XE_OFF = 163840;
constexpr int REGS_MMA = 24;
template <int CW> struct Cfg {
  static constexpr int NCQ = H / CW;                // column groups
  static constexpr int NTC = TM * NCQ;              // compute threads: thread = (sample s, CW hidden columns)
  static constexpr int NTH = NTC + 128;             // + the MMA warpgroup (its first warp issues; the others only lend registers)
  // setmaxnreg moves registers through the CTA's pool only: what the compute warps take (inc) must have been released by
  // the MMA warpgroup (dec) -- asking for more spins forever in USETMAXREG.TRY_ALLOC (measured: a hung box).
  static constexpr int REGS_LAUNCH = (65536 / NTH) / 8 * 8;           // what ptxas gives every thread at launch (168 / 96)
  static constexpr int REGS = CW == 32 ? 240 : 112;
  static_assert(NTC * (REGS - REGS_LAUNCH) <= 128 * (REGS_LAUNCH - REGS_MMA), "setmaxnreg.inc would exceed what setmaxnreg.dec releases");
  static_assert(REGS % 8 == 0 && REGS <= 255 && REGS_MMA % 8 == 0 && REGS_MMA >= 24, "setmaxnreg operands");
};
}  // namespace v2

template <int N>
__device__ __forceinline__ void tmem_ld_n(uint32_t taddr, uint32_t (&v)[N]) {
  if constexpr (N == 32) tmem_ld32_nowait(taddr, v); else tmem_ld16_nowait(taddr, v);
  tmem_ld_wait();
}
template <int N>
__device__ __forceinline__ void tmem_st_n(uint32_t taddr, const uint32_t (&v)[N]) {
  if constexpr (N == 32) tmem_st32(taddr, v); else tmem_st16(taddr, v);
}
// v[CW] = columns c0 .. c0+CW-1 of row s -> MN-major BASE32B images (raw at `img`, lo at `img + lo_delta`); img = image base.
// The kernel is bound by the shared-memory data pipe (tensor-core operand fetch + these stores: ncu r02d 82 % busy), so the
// stores must be conflict-free: the 32-byte-chunk swizzle only separates 4 of the 8 rows of a store phase -- rows s and
// s + 4 would hit the same 16 bytes -- so lanes with bit 2 of s set write the two 16-byte halves of every 32-byte chunk
// in the opposite order (4 selects per store instead of a 2-way bank conflict).
template <int CW>
__device__ __forceinline__ void store_mn_images(uint32_t img, uint32_t lo_delta, int s, int c0, const float (&v)[CW]) {
  // bits [5,7) of the block base are zero: the 32-byte-chunk swizzle is an XOR with (s & 3) << 5
  const uint32_t row = (img + (uint32_t)((c0 >> 5) * 16384 + s * 128)) | (uint32_t)((s & 3) << 5);
  const bool swp = (s & 4) != 0;
  const uint32_t hx = swp ? 16u : 0u;
  const int j0 = (c0 & 31) >> 2;                    // first 16-byte chunk of this thread inside the 128-byte row (even)
#pragma unroll
  for (int jj = 0; jj < CW / 4; ++jj) {
    const int j = j0 + jj, jo = jj ^ 1;             // this instruction's chunk for swp == 0; the lane's other chunk of the pair
    const uint32_t a = ((row ^ (uint32_t)((j >> 1) << 5)) + (uint32_t)((j & 1) << 4)) ^ hx;
    const float x0 = swp ? v[4 * jo] : v[4 * jj], x1 = swp ? v[4 * jo + 1] : v[4 * jj + 1];
    const float x2 = swp ? v[4 * jo + 2] : v[4 * jj + 2], x3 = swp ? v[4 * jo + 3] : v[4 * jj + 3];
    sts128(a, x0, x1, x2, x3);
    sts128(a + lo_delta, lo_of(x0), lo_of(x1), lo_of(x2), lo_of(x3));
  }
}
// every lane holds v[0..CW-1]; afterwards column k's sum over the 32 lanes sits in lane k (CW = 32) or in lanes 2k and
// 2k+1 (CW = 16).  Fixed shuffle network -> deterministic.
template <int CW>
__device__ __forceinline__ float warp_transpose_sum(float (&v)[CW], int lane) {
  constexpr int L0 = 16;
#pragma unroll
  for (int off = L0, n = CW / 2; n >= 1; off >>= 1, n >>= 1) {
    const bool up = (lane & off) != 0;
#pragma unroll
    for (int k = 0; k < n; ++k) {
      const float keep = up ? v[k + n] : v[k], send = up ? v[k] : v[k + n];
      v[k] = keep + __shfl_xor_sync(0xffffffffu, send, off);
    }
  }
  if constexpr (CW == 16) v[0] += __shfl_xor_sync(0xffffffffu, v[0], 1);
  return v[0];
}

template <int DP, int CW>
__global__ void __launch_bounds__(v2::Cfg<CW>::NTH, 1) mlp3_tc_bwd2_kernel(BwdP p) {
  using namespace v2;
  using C = Cfg<CW>;
  constexpr int NTC = C::NTC, NTH = C::NTH, NCW = NTC / 32;
  constexpr int NX = DP + 8;                        // rows of the thin B operand: X^T (DP rows) | ones | 7 zero rows
  constexpr uint32_t XE_KB = NX * 128;              // bytes of one 32-sample k-block of that image
  constexpr uint32_t XE_BYTES = 4 * XE_KB;          // one image (raw or lo)
  constexpr int XPT = (TM * DP) / NTC;
  static_assert((TM * DP) % NTC == 0, "X tile must divide over the compute threads");
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t W_raw = smem + W_RAW, W_lo = smem + W_LO;          // B of GEMM 2: B[n = i][k = j] = W2[i][j], K-major
  const uint32_t V_raw = smem + V_RAW;                               // MN-major [2 blocks][128 s][128 B]: H1, then dP1
  const uint32_t Q_raw = smem + Q_RAW;                               // MN-major: dP2
  const uint32_t Xe_raw = smem + XE_OFF, Xe_lo = Xe_raw + XE_BYTES;  // K-major [4 k-blocks][NX rows][128 B]
  __shared__ __align__(16) float W3s[MAXO * H];                      // [j][c]
  __shared__ __align__(16) float red3[4][MAXO + 2][H];               // end of kernel: per-sample-quarter dW3 / db3 / db2 partials
  __shared__ __align__(8) uint64_t bars[6];
  __shared__ uint32_t tmem_slot;

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int g = blockIdx.y, o = p.o[g], D = p.D;
  const uint32_t barG2 = smem_u32(&bars[0]), barG1 = smem_u32(&bars[1]), barG3 = smem_u32(&bars[2]);   // tcgen05.commit
  const uint32_t opsG2 = smem_u32(&bars[3]), opsG1 = smem_u32(&bars[4]), opsG3 = smem_u32(&bars[5]);   // one arrive per compute warp
  auto bar_compute = [] { asm volatile("bar.sync 1, %0;" ::"n"(NTC) : "memory"); };
  const int nT = ((int)blockIdx.x < p.nTiles) ? (p.nTiles - 1 - (int)blockIdx.x) / (int)gridDim.x + 1 : 0;   // tiles of this CTA

  if (tid == 0) {
    mbar_init(barG2, 1); mbar_init(barG1, 1); mbar_init(barG3, 1);
    mbar_init(opsG2, NCW); mbar_init(opsG1, NCW); mbar_init(opsG3, NCW);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 0) tmem_alloc<512>(&tmem_slot);
  {                                                 // W2 -> K-major images; loads batched ahead of the stores
    constexpr int WPT = (H * H + NTH - 1) / NTH;
    float w[WPT];
#pragma unroll
    for (int r = 0; r < WPT; ++r) { const int e = tid + r * NTH; w[r] = e < H * H ? __ldg(p.W2 + (size_t)g * H * H + e) : 0.f; }
#pragma unroll
    for (int r = 0; r < WPT; ++r) {
      const int e = tid + r * NTH, i = e >> 6, j = e & 63;
      if (e < H * H) {
        const uint32_t off = (uint32_t)((j >> 5) * 8192) + sw128_off(i, j & 31);
        sts32(W_raw + off, w[r]);
        sts32(W_lo + off, lo_of(w[r]));
      }
    }
  }
  for (int e = tid; e < MAXO * H; e += NTH) {
    const int j = e >> 6, c = e & 63;
    W3s[e] = j < o ? __ldg(p.W3[g] + c * o + j) : 0.f;
  }
  for (uint32_t e = tid; e < 2 * XE_BYTES / 4; e += NTH) sts32(Xe_raw + e * 4, 0.f);
  __syncthreads();
  if (tid < TM) sts32(Xe_raw + (uint32_t)(tid >> 5) * XE_KB + sw128_off(DP, tid & 31), 1.f);      // the ones row (its lo part is zero)
  fence_async_smem();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = tmem_slot;

  // Software pipeline over the tiles t0, t1, ... of this CTA (phases of tile t):
  //   A(t)  dP2 -> tensor memory                    -> GEMM 2(t) = dP1pre        [needs GEMM 2(t-1) read out]
  //   B(t)  H1 image (V), X^T image                 -> GEMM 1(t) = dW2           [needs GEMM 3(t-1) done: it read V and X^T]
  //   D(t)  dP1 image (into V), dP2(t+1) image (Q)  -> GEMM 3(t) = dW1 | db1     [needs GEMM 2(t) and GEMM 1(t) done]
  // One loop iteration runs B(t), dP1(t), A(t+1) + the in-warp sums of tile t+1, D(t); the tensor pipe runs
  // GEMM 1(t), GEMM 2(t+1), GEMM 3(t) -- GEMM 2(t+1) fills the gap while the compute warps write the dP1 image.  The only
  // serial resource is the V image: B(t) -> GEMM 1(t) -> D(t) -> GEMM 3(t) -> B(t+1).
  if (warp >= NCW) {
    // ------------------------------------------------ MMA warpgroup ------------------------------------------------
    setmaxnreg_dec<REGS_MMA>();
    if (warp == NCW) {
      // (loops deliberately not unrolled: an MMA occupies its issuer for 23-32 cycles anyway, and the unrolled form keeps
      // ~100 precomputed descriptors alive -- spills at the 24 registers this warpgroup keeps)
      const uint64_t dwr = make_desc(W_raw), dwl = make_desc(W_lo);
      const uint64_t dvr = make_desc_mn32(V_raw, 16384, 512), dvl = make_desc_mn32(V_raw + LO_DELTA, 16384, 512);
      const uint64_t dqr = make_desc_mn32(Q_raw, 16384, 512), dql = make_desc_mn32(Q_raw + LO_DELTA, 16384, 512);
      const uint64_t dxr = make_desc(Xe_raw), dxl = make_desc(Xe_lo);
      constexpr uint32_t id2 = make_idesc_full(128, 64, 0, 0), id1 = make_idesc_full(64, 64, 1, 1), id3 = make_idesc_full(64, NX, 1, 0);
      const bool leader = elect_one();
      auto gemm2 = [&](int it) {                    // dP1pre [128 x 64] = dP2 (tensor memory) . W2^T; small terms first
        mbar_wait(opsG2, (uint32_t)(it & 1));
        tc_fence_after();
        if (leader) {
#pragma unroll 1
          for (int ks = 0; ks < 8; ++ks) {
            const uint64_t ob = (uint64_t)(((ks >> 2) * 8192 + (ks & 3) * 32) >> 4);
            umma_tf32_ts(tmem + ACC2, tmem + A_LO + ks * 8, dwr + ob, id2, ks ? 1u : 0u);
            umma_tf32_ts(tmem + ACC2, tmem + A_RAW + ks * 8, dwl + ob, id2, 1u);
          }
#pragma unroll 1
          for (int ks = 0; ks < 8; ++ks) {
            const uint64_t ob = (uint64_t)(((ks >> 2) * 8192 + (ks & 3) * 32) >> 4);
            umma_tf32_ts(tmem + ACC2, tmem + A_RAW + ks * 8, dwr + ob, id2, 1u);
          }
          umma_commit(barG2);
        }
        __syncwarp();
      };
      if (nT > 0) gemm2(0);
      for (int it = 0; it < nT; ++it) {
        const uint32_t ph = (uint32_t)(it & 1);
        // GEMM 1: dW2 [64 x 64] = H1^T dP2 over the 128 samples (both operands MN-major)
        mbar_wait(opsG1, ph);
        tc_fence_after();
        if (leader) {
#pragma unroll 1
          for (int ks = 0; ks < 16; ++ks) {
            const uint64_t oo = (uint64_t)(ks * 64);
            umma_tf32(tmem + ACC1, dvl + oo, dqr + oo, id1, ks ? 1u : 0u);
            umma_tf32(tmem + ACC1, dvr + oo, dql + oo, id1, 1u);
          }
#pragma unroll 1
          for (int ks = 0; ks < 16; ++ks) {
            const uint64_t oo = (uint64_t)(ks * 64);
            umma_tf32(tmem + ACC1, dvr + oo, dqr + oo, id1, 1u);
          }
          umma_commit(barG1);
        }
        __syncwarp();
        if (it + 1 < nT) gemm2(it + 1);
        // GEMM 3: [dW1^T | db1] [64 x NX] = dP1^T [X | 1] over the 128 samples (the dP1 image sits where H1 was)
        mbar_wait(opsG3, ph);
        tc_fence_after();
        if (leader) {
#pragma unroll 1
          for (int ks = 0; ks < 16; ++ks) {
            const uint64_t oa = (uint64_t)(ks * 64), ob = (uint64_t)(((ks >> 2) * XE_KB + (ks & 3) * 32) >> 4);
            umma_tf32(tmem + ACC3, dvl + oa, dxr + ob, id3, ks ? 1u : 0u);
            umma_tf32(tmem + ACC3, dvr + oa, dxl + ob, id3, 1u);
          }
#pragma unroll 1
          for (int ks = 0; ks < 16; ++ks) {
            const uint64_t oa = (uint64_t)(ks * 64), ob = (uint64_t)(((ks >> 2) * XE_KB + (ks & 3) * 32) >> 4);
            umma_tf32(tmem + ACC3, dvr + oa, dxr + ob, id3, 1u);
          }
          umma_commit(barG3);
        }
        __syncwarp();
      }
    }
  } else {
    // ------------------------------------------------ compute warps ------------------------------------------------
    setmaxnreg_inc<C::REGS>();
    const int q = warp & 3, cq = warp >> 2, s = q * 32 + lane, c0 = cq * CW;
    const uint32_t tlane = tmem + ((uint32_t)(q * 32) << 16);
    auto arrive = [&](uint32_t bar) {         // this warp's operand writes -> visible to the tensor core; one arrive per warp
      fence_async_smem();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(bar);
    };

    float dW2acc[CW];                         // lanes < 16: dW2[i = q*16+lane][c0 .. c0+CW-1]
    float acc3[NX];                           // cq == 0, lanes < 16: dW1[n][i = q*16+lane] (n < DP), db1[i] (n == DP)
    float a_dW3[MAXO] = {0.f, 0.f, 0.f, 0.f}; // dW3[column of this lane][j] over this warp's samples (see warp_transpose_sum)
    float a_db3 = 0.f, a_db2 = 0.f;           // lane j < o: db3[j]; db2[column of this lane]; over this warp's samples
#pragma unroll
    for (int c = 0; c < CW; ++c) dW2acc[c] = 0.f;
#pragma unroll
    for (int n = 0; n < NX; ++n) acc3[n] = 0.f;

    float h1[CW], h2[CW], xpre[XPT];
    float4 dpre = make_float4(0.f, 0.f, 0.f, 0.f);
    // prefetches are unconditional (the tile index is clamped): a conditional load makes the compiler merge old and new
    // values with register moves at the loop edge, and those moves wait for the loads
    auto prefetch_hd = [&](int tile_) {       // H2 and the output gradient of the tile
      const int tile = min(tile_, p.nTiles - 1);
      const float4* h2t = reinterpret_cast<const float4*>(p.H2t + ((size_t)(g * p.nTiles + tile) * H + c0) * TM) + s;
#pragma unroll
      for (int j = 0; j < CW / 4; ++j) {
        const float4 b = ld_stream4(h2t + j * TM);
        h2[4 * j] = b.x; h2[4 * j + 1] = b.y; h2[4 * j + 2] = b.z; h2[4 * j + 3] = b.w;
      }
      const int b = tile * TM + s;
      float d[MAXO] = {0.f, 0.f, 0.f, 0.f};
      if (b < p.M) {
        if (p.vh_v[g] != nullptr) {           // o == 1 (checked on the host); same formula as mlp_fused.cu
          const float w1 = (float)p.vh_branch[g][0], w2 = (float)p.vh_branch[g][1], clip = p.vh_clip;
          const float v = ld_stream(p.vh_v[g] + b), ov = ld_stream(p.vh_ov[g] + b), R = ld_stream(p.vh_R[g] + b);
          const float dd = v - ov;
          const float vc = ov + fminf(fmaxf(dd, -clip), clip);
          const float pass = (dd >= -clip && dd <= clip) ? 1.f : 0.f;
          const float gv = w1 * (-2.f * (R - v)) + w2 * (-2.f * (R - vc)) * pass;
          d[0] = p.vh_scale[g] * gv / p.vh_Bt;
        } else {
#pragma unroll
          for (int j = 0; j < MAXO; ++j)
            if (j < o) d[j] = ld_stream(p.dOut[g] + (size_t)b * o + j);
        }
      }
      dpre = make_float4(d[0], d[1], d[2], d[3]);
    };
    auto prefetch_x = [&](int tile_) {        // this thread's share of the tile's X rows
      const int m0 = min(tile_, p.nTiles - 1) * TM;
#pragma unroll
      for (int r = 0; r < XPT; ++r) {
        const int e = tid + r * NTC, row = e / DP, k = e % DP;
        xpre[r] = (m0 + row < p.M && k < D) ? __ldg(p.X + (size_t)(m0 + row) * p.ldx + k) : 0.f;
      }
    };
    auto prefetch_b = [&](int tile_) {        // H1 of the tile
      const int tile = min(tile_, p.nTiles - 1);
      const float4* h1t = reinterpret_cast<const float4*>(p.H1t + ((size_t)(g * p.nTiles + tile) * H + c0) * TM) + s;
#pragma unroll
      for (int j = 0; j < CW / 4; ++j) {
        const float4 a = ld_stream4(h1t + j * TM);
        h1[4 * j] = a.x; h1[4 * j + 1] = a.y; h1[4 * j + 2] = a.z; h1[4 * j + 3] = a.w;
      }
    };
    // A(t): dP2 = (dOut W3^T)(1 - H2^2) -> tensor memory (A operand of GEMM 2), from the prefetched h2 / dpre
    auto phase_a = [&](float (&dp2)[CW]) {
      const float dj[MAXO] = {dpre.x, dpre.y, dpre.z, dpre.w};
#pragma unroll
      for (int c = 0; c < CW; c += 4) {
        float4 a = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
        for (int j = 0; j < MAXO; ++j)
          if (j < o) {                        // CTA-uniform
            const float4 w = *reinterpret_cast<const float4*>(&W3s[j * H + c0 + c]);
            a.x = fmaf(dj[j], w.x, a.x); a.y = fmaf(dj[j], w.y, a.y); a.z = fmaf(dj[j], w.z, a.z); a.w = fmaf(dj[j], w.w, a.w);
          }
        dp2[c] = a.x * (1.f - h2[c] * h2[c]); dp2[c + 1] = a.y * (1.f - h2[c + 1] * h2[c + 1]);
        dp2[c + 2] = a.z * (1.f - h2[c + 2] * h2[c + 2]); dp2[c + 3] = a.w * (1.f - h2[c + 3] * h2[c + 3]);
      }
#pragma unroll
      for (int hh = 0; hh < CW; hh += 16) {    // 16 columns at a time: fewer live registers than one 32-wide store
        uint32_t u[16];
#pragma unroll
        for (int c = 0; c < 16; ++c) u[c] = __float_as_uint(dp2[hh + c]);
        tmem_st16(tlane + A_RAW + c0 + hh, u);
#pragma unroll
        for (int c = 0; c < 16; ++c) u[c] = __float_as_uint(lo_of(dp2[hh + c]));
        tmem_st16(tlane + A_LO + c0 + hh, u);
      }
      tmem_st_wait();
    };
    // in-warp sums of the tile whose h2 / dpre / dp2 are in registers: dW3, db3, db2 over this warp's 32 samples
    auto phase_c = [&](const float (&dp2)[CW]) {
      const float dj[MAXO] = {dpre.x, dpre.y, dpre.z, dpre.w};
#pragma unroll
      for (int j = 0; j < MAXO; ++j)
        if (j < o) {                          // CTA-uniform
          float v[CW];
#pragma unroll
          for (int c = 0; c < CW; ++c) v[c] = h2[c] * dj[j];
          a_dW3[j] += warp_transpose_sum<CW>(v, lane);
          const float t = warp_sum(dj[j]);
          if (lane == j) a_db3 += t;
        }
      float v[CW];
#pragma unroll
      for (int c = 0; c < CW; ++c) v[c] = dp2[c];
      a_db2 += warp_transpose_sum<CW>(v, lane);
    };

    if (nT > 0) {
      // ---- prologue: A(t0), its in-warp sums, its dP2 image ----
      const int t0 = blockIdx.x;
      prefetch_hd(t0);
      prefetch_x(t0);
      prefetch_b(t0);
      {
        float dp2[CW];
        phase_a(dp2);
        arrive(opsG2);
        store_mn_images<CW>(Q_raw, LO_DELTA, s, c0, dp2);
        phase_c(dp2);
      }
      prefetch_hd(t0 + (int)gridDim.x);
      for (int it = 0; it < nT; ++it) {
        const uint32_t ph = (uint32_t)(it & 1);
        const int t1 = (int)blockIdx.x + (it + 1) * (int)gridDim.x;      // next tile of this CTA (clamped by the prefetches)
        const bool has_next = it + 1 < nT;
        // ---- B(t): previous GEMM 3 out; H1 image + X^T image -> GEMM 1(t) ----
        if (it > 0) {
          mbar_wait(barG3, ph ^ 1);
          tc_fence_after();
          if (cq == 0) {
#pragma unroll
            for (int n0 = 0; n0 < NX; n0 += 8) {
              uint32_t y[8];
              tmem_ld8_nowait(tlane + ACC3 + n0, y);
              tmem_ld_wait();
#pragma unroll
              for (int n = 0; n < 8; ++n) acc3[n0 + n] += __uint_as_float(y[n]);
            }
          }
        }
        store_mn_images<CW>(V_raw, LO_DELTA, s, c0, h1);
#pragma unroll
        for (int r = 0; r < XPT; ++r) {
          const int e = tid + r * NTC, row = e / DP, k = e % DP;
          const uint32_t off = (uint32_t)(row >> 5) * XE_KB + sw128_off(k, row & 31);
          sts32(Xe_raw + off, xpre[r]);
          sts32(Xe_lo + off, lo_of(xpre[r]));
        }
        arrive(opsG1);                        // (the dP2 image of this tile was written in the previous iteration / the prologue)
        prefetch_x(t1);
        // ---- dP1(t) = (dP2 W2^T)(1 - H1^2) into registers; GEMM 2's accumulator and operand columns are then free ----
        mbar_wait(barG2, ph);
        tc_fence_after();
        float dp1[CW];
        {
          uint32_t z[CW];
          tmem_ld_n<CW>(tlane + ACC2 + c0, z);
#pragma unroll
          for (int c = 0; c < CW; ++c) dp1[c] = __uint_as_float(z[c]) * (1.f - h1[c] * h1[c]);
        }
        prefetch_b(t1);                       // H1 registers are free
        // ---- A(t+1) + its in-warp sums (under GEMM 1(t)) ----
        float dp2n[CW];
        if (has_next) {
          phase_a(dp2n);
          arrive(opsG2);
          phase_c(dp2n);
        }
        prefetch_hd(t1 + (int)gridDim.x);
        // ---- D(t): GEMM 1(t) has read V and Q: dW2 out, dP1 image where H1 was -> GEMM 3(t); dP2(t+1) image ----
        mbar_wait(barG1, ph);
        tc_fence_after();
        {
          uint32_t z[CW];
          tmem_ld_n<CW>(tlane + ACC1 + c0, z);
#pragma unroll
          for (int c = 0; c < CW; ++c) dW2acc[c] += __uint_as_float(z[c]);
        }
        store_mn_images<CW>(V_raw, LO_DELTA, s, c0, dp1);
        arrive(opsG3);
        if (has_next) store_mn_images<CW>(Q_raw, LO_DELTA, s, c0, dp2n);
      }
      mbar_wait(barG3, (uint32_t)((nT - 1) & 1));               // the last tile's GEMM 3
      tc_fence_after();
      if (cq == 0) {
#pragma unroll
        for (int n0 = 0; n0 < NX; n0 += 8) {
          uint32_t y[8];
          tmem_ld8_nowait(tlane + ACC3 + n0, y);
          tmem_ld_wait();
#pragma unroll
          for (int n = 0; n < 8; ++n) acc3[n0 + n] += __uint_as_float(y[n]);
        }
      }
    }
    // ---- one partial per CTA ----
    float* w2 = p.ws2 + (size_t)(g * gridDim.x + blockIdx.x) * H * H;
    float* wr = p.wsr + ((size_t)g * gridDim.x + blockIdx.x) * p.RS;
    const int offb1 = D * H, offb2 = offb1 + H, offW3 = offb2 + H, offb3 = offW3 + H * o;
    if (lane < 16) {
      const int i = q * 16 + lane;
#pragma unroll
      for (int c = 0; c < CW; c += 4)
        *reinterpret_cast<float4*>(&w2[i * H + c0 + c]) = make_float4(dW2acc[c], dW2acc[c + 1], dW2acc[c + 2], dW2acc[c + 3]);
      if (cq == 0) {
#pragma unroll
        for (int n = 0; n < DP; ++n)
          if (n < D) wr[n * H + i] = acc3[n];
        wr[offb1 + i] = acc3[DP];
      }
    }
    {                                         // this warp's dW3 / db2 / db3 partials: column of lane l is c0 + l (CW = 32) or c0 + l/2
      const bool own = CW == 32 || (lane & 1) == 0;
      const int c = c0 + (CW == 32 ? lane : (lane >> 1));
      if (own) {
#pragma unroll
        for (int j = 0; j < MAXO; ++j) red3[q][j][c] = a_dW3[j];
        red3[q][MAXO + 1][c] = a_db2;
      }
      if (cq == 0 && lane < MAXO) red3[q][MAXO][lane] = a_db3;
    }
    bar_compute();
    for (int e = tid; e < (MAXO + 2) * H; e += NTC) {     // combine the four sample quarters in a fixed order
      const int n = e >> 6, c = e & 63;
      const float v = (red3[0][n][c] + red3[1][n][c]) + (red3[2][n][c] + red3[3][n][c]);
      if (n < MAXO) { if (n < o) wr[offW3 + c * o + n] = v; }
      else if (n == MAXO) { if (c < o) wr[offb3 + c] = v; }
      else wr[offb2 + c] = v;
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) { tc_fence_after(); tmem_dealloc<512>(tmem); }
}

inline bool shape_ok(int D, int Hh, int G, const int* outs) {
  if (Hh != H || D < 1 || D > MAXD || G < 1 || G > MAXG) return false;
  for (int g = 0; g < G; ++g)
    if (outs[g] < 1 || outs[g] > MAXO) return false;
  return true;
}
inline int dp_of(int D) { return D <= 8 ? 8 : (D <= 16 ? 16 : 32); }
inline int n_tiles(int M) { return (M + TM - 1) / TM; }
inline int rest_size(int D, int o) { return D * H + 2 * H + H * o + o; }
inline int omax_of(int G, const int* outs) { int m = 0; for (int g = 0; g < G; ++g) m = std::max(m, outs[g]); return m; }
constexpr size_t kFwdSmem = 98304 + 1024;
inline size_t bwd_smem(int DP) { return 196608 + (size_t)TM * DP * 4 + 1024; }
inline int fwd_grid(int M, int G) { return std::max(1, std::min(n_tiles(M), 2 * sm_count() / G)); }
inline int bwd_grid(int M, int G) { return std::max(1, std::min(n_tiles(M), sm_count() / G)); }

template <int DP>
int launch_fwd(const FwdP& p, dim3 grid, cudaStream_t st) {
  static bool configured = false;
  if (!configured) {
    PPX_CUDA(cudaFuncSetAttribute(mlp3_tc_fwd_kernel<DP>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kFwdSmem));
    configured = true;
  }
  mlp3_tc_fwd_kernel<DP><<<grid, NT, kFwdSmem, st>>>(p);
  return after_launch("mlp3_tc_fwd");
}
constexpr size_t kFwd2Smem = 49152 + 1024;
template <int DP>
int launch_fwd2(const FwdP& p, dim3 grid, cudaStream_t st) {
  static bool configured = false;
  if (!configured) {
    PPX_CUDA(cudaFuncSetAttribute(mlp3_tc_fwd2_kernel<DP>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kFwd2Smem));
    configured = true;
  }
  mlp3_tc_fwd2_kernel<DP><<<grid, NT, kFwd2Smem, st>>>(p);
  return after_launch("mlp3_tc_fwd2");
}
template <int DP, int CW, bool MMAW>
int launch_bwd(const BwdP& p, dim3 grid, cudaStream_t st) {
  static bool configured = false;
  if (!configured) {
    PPX_CUDA(cudaFuncSetAttribute(mlp3_tc_bwd_kernel<DP, CW, MMAW>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bwd_smem(DP)));
    configured = true;
  }
  mlp3_tc_bwd_kernel<DP, CW, MMAW><<<grid, TM * (H / CW) + (MMAW ? 32 : 0), bwd_smem(DP), st>>>(p);
  return after_launch("mlp3_tc_bwd");
}

template <int DP, int CW>
int launch_bwd2(const BwdP& p, dim3 grid, cudaStream_t st) {
  constexpr size_t smem = v2::XE_OFF + 2 * 4 * (size_t)(DP + 8) * 128 + 1024;
  static bool configured = false;
  if (!configured) {
    PPX_CUDA(cudaFuncSetAttribute(mlp3_tc_bwd2_kernel<DP, CW>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    configured = true;
  }
  mlp3_tc_bwd2_kernel<DP, CW><<<grid, v2::Cfg<CW>::NTH, smem, st>>>(p);
  return after_launch("mlp3_tc_bwd2");
}

}  // namespace mt
}  // namespace ppx

using namespace ppx;

extern "C" int ppx_mlp3_tc_supported(int D, int H, int G, const int* outs) {
  return (outs && mt::shape_ok(D, H, G, outs)) ? 1 : 0;
}

extern "C" int64_t ppx_mlp3_tc_act_elems(int M, int H, int G) {
  if (H != mt::H || M < 0 || G < 1) return -1;
  return (int64_t)G * mt::n_tiles(M) * mt::H * mt::TM;
}

extern "C" int ppx_mlp3_tc_fwd(const float* X, int ldx, int M, int D, int H, int G, const int* outs, const float* W1,
                               const float* b1, const float* W2, const float* b2, const float* const* W3,
                               const float* const* b3, float* H1t, float* H2t, float* const* out, void* stream) {
  PPX_REQUIRE(X && outs && W1 && b1 && W2 && b2 && W3 && b3 && H1t && H2t && out, "mlp3_tc_fwd: null pointer");
  PPX_REQUIRE(mt::shape_ok(D, H, G, outs), "mlp3_tc_fwd: unsupported shape D=%d H=%d G=%d", D, H, G);
  PPX_REQUIRE(M >= 0 && ldx >= D, "mlp3_tc_fwd: M=%d ldx=%d", M, ldx);
  if (M == 0) return PPX_OK;
  mt::FwdP p{};
  p.X = X; p.ldx = ldx; p.M = M; p.D = D; p.G = G; p.nTiles = mt::n_tiles(M);
  p.W1 = W1; p.b1 = b1; p.W2 = W2; p.b2 = b2; p.H1t = H1t; p.H2t = H2t;
  for (int g = 0; g < G; ++g) { p.W3[g] = W3[g]; p.b3[g] = b3[g]; p.o[g] = outs[g]; p.out[g] = out[g]; }
  dim3 grid((unsigned)mt::fwd_grid(M, G), (unsigned)G);
  cudaStream_t st = (cudaStream_t)stream;
  // D <= 16: layer 1 on the tensor pipe, A operands in TMEM (v2); 16 < D <= 32: the round-1 kernel
  if (D <= 16) return mt::dp_of(D) == 8 ? mt::launch_fwd2<8>(p, grid, st) : mt::launch_fwd2<16>(p, grid, st);
  return mt::launch_fwd<32>(p, grid, st);
}

extern "C" int64_t ppx_mlp3_tc_bwd_workspace(int M, int D, int H, int G, const int* outs) {
  if (!outs || !mt::shape_ok(D, H, G, outs)) return -1;
  const int n = mt::bwd_grid(M, G), RS = mt::round4(mt::rest_size(D, mt::omax_of(G, outs)));
  return (int64_t)G * n * ((int64_t)mt::H * mt::H + RS);
}

static std::atomic<void*> g_bwd_probe{nullptr};
extern "C" int ppx_mlp3_tc_bwd_probe(void* cuda_event) {
  g_bwd_probe.store(cuda_event);
  return PPX_OK;
}

extern "C" int ppx_mlp3_tc_bwd(const float* X, int ldx, int M, int D, int H, int G, const int* outs, const float* W2,
                               const float* const* W3, const float* H1t, const float* H2t, const float* const* dOut,
                               const ppx_value_head* vh, float clip_range, int64_t B_total, float* dW1, float* db1,
                               float* dW2, float* db2, float* const* dW3, float* const* db3, float* workspace,
                               double* sumsq_partials, int64_t* step_dev, const ppx_fused_adam* adam,
                               void* stream) {
  PPX_REQUIRE(X && outs && W2 && W3 && H1t && H2t && dOut && dW1 && db1 && dW2 && db2 && dW3 && db3 && workspace, "mlp3_tc_bwd: null pointer");
  PPX_REQUIRE(mt::shape_ok(D, H, G, outs), "mlp3_tc_bwd: unsupported shape D=%d H=%d G=%d", D, H, G);
  PPX_REQUIRE(M >= 1 && ldx >= D, "mlp3_tc_bwd: M=%d ldx=%d", M, ldx);
  PPX_REQUIRE(!adam || sumsq_partials, "mlp3_tc_bwd: the fused optimiser tail needs sumsq_partials");
  const int n = mt::bwd_grid(M, G), RS = mt::round4(mt::rest_size(D, mt::omax_of(G, outs)));
  mt::BwdP p{};
  p.X = X; p.ldx = ldx; p.M = M; p.D = D; p.G = G; p.nTiles = mt::n_tiles(M); p.W2 = W2; p.H1t = H1t; p.H2t = H2t;
  p.ws2 = workspace; p.wsr = workspace + (size_t)G * n * mt::H * mt::H; p.RS = RS;
  p.vh_clip = clip_range; p.vh_Bt = (float)(B_total > 0 ? B_total : M);
  for (int g = 0; g < G; ++g) {
    p.W3[g] = W3[g]; p.o[g] = outs[g]; p.dOut[g] = dOut[g];
    if (vh && vh[g].values) {
      PPX_REQUIRE(outs[g] == 1 && vh[g].old_values && vh[g].returns && vh[g].branch, "mlp3_tc_bwd: value head %d needs o=1 and all inputs", g);
      p.vh_v[g] = vh[g].values; p.vh_ov[g] = vh[g].old_values; p.vh_R[g] = vh[g].returns; p.vh_branch[g] = vh[g].branch;
      p.vh_scale[g] = vh[g].scale;
    } else {
      PPX_REQUIRE(dOut[g], "mlp3_tc_bwd: dOut[%d] is null", g);
    }
  }
  dim3 grid((unsigned)n, (unsigned)G);
  cudaStream_t st = (cudaStream_t)stream;
  int rc;
  if (D <= 16) {            // v2: A of GEMM 2 from tensor memory, MN-major images, dW1 / db1 on the tensor pipe
    rc = mt::dp_of(D) == 8 ? mt::launch_bwd2<8, 32>(p, grid, st) : mt::launch_bwd2<16, 32>(p, grid, st);
  } else {                  // 16 < D <= 32: the round-1 kernel (its operand images do not fit next to a 40-row X^T image)
    rc = mt::launch_bwd<32, 32, false>(p, grid, st);
  }
  if (rc) return rc;
  if (void* ev = g_bwd_probe.exchange(nullptr)) PPX_CUDA(cudaEventRecord((cudaEvent_t)ev, st));   // measurement hook, see ppx.h
  return mf::mlp3_reduce_launch(H, D, G, outs, p.ws2, p.wsr, n, RS, dW1, db1, dW2, db2, dW3, db3, sumsq_partials,
                                (sumsq_partials && !adam) ? step_dev : nullptr, adam, st);
}
