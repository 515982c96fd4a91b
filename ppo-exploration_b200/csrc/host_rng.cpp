// Host-side, bit-exact replay of numpy's legacy shuffle:  np.random.permutation(n)  (buffer.py:239).
//
// The reference draws one permutation per epoch from the GLOBAL legacy RandomState (MT19937).  To keep
// "bit-exact shuffle indices" without paying numpy's generic shuffle loop (7-18 ms per 512k on the
// host, which would bound the whole learner pass), this restates numpy's algorithm in C:
//   RandomState.permutation(n): arr = arange(n, int64); shuffle(arr)
//   shuffle (1-d fast path):    for i = n-1 .. 1:  j = random_interval(i);  swap(arr[i], arr[j])
//   random_interval(max):       mask = next_pow2(max+1)-1;  do v = next_uint32() & mask while v > max
//                               (64-bit draws when max > 0xffffffff)
//   next_uint32:                MT19937 genrand with the standard tempering
// The caller passes numpy's own state (np.random.get_state(): key[624], pos) and writes the advanced
// state back with np.random.set_state, so interleaved numpy calls (e.g. RND's randn()) stay in sequence.
// The learner's shuffle only draws here -- the partner sequence (RNG-bound; AVX-512 block rejection with compress-store
// when the CPU has it) -- and applies the swaps on the device (shuffle_dev.cu); ppx_np_permutation does both on the host.
// Compiled by g++ (not nvcc): it uses target attributes / immintrin.
#include <stdlib.h>
#include <immintrin.h>
#include "common.cuh"

namespace {
constexpr int MT_N = 624, MT_M = 397;
constexpr uint32_t MATRIX_A = 0x9908b0dfu, UPPER = 0x80000000u, LOWER = 0x7fffffffu;

bool has_avx512() {
  static const bool ok = __builtin_cpu_supports("avx512f") && __builtin_cpu_supports("avx512bw") &&
                         __builtin_cpu_supports("avx512vl") && __builtin_cpu_supports("avx512dq");
  return ok;
}

inline uint32_t twist(uint32_t a, uint32_t b, uint32_t far) {
  const uint32_t y = (a & UPPER) | (b & LOWER);
  return far ^ (y >> 1) ^ ((y & 1u) ? MATRIX_A : 0u);
}

void gen_block_base(uint32_t* k, uint32_t* __restrict__ o) {
  int i;
  for (i = 0; i < MT_N - MT_M; i++) k[i] = twist(k[i], k[i + 1], k[i + MT_M]);
  for (; i < MT_N - 1; i++) k[i] = twist(k[i], k[i + 1], k[i + (MT_M - MT_N)]);
  k[MT_N - 1] = twist(k[MT_N - 1], k[0], k[MT_M - 1]);
  for (i = 0; i < MT_N; ++i) {
    uint32_t y = k[i];
    y ^= (y >> 11);
    y ^= (y << 7) & 0x9d2c5680u;
    y ^= (y << 15) & 0xefc60000u;
    y ^= (y >> 18);
    o[i] = y;
  }
}

// 16 state words per step.  The recurrence k[i] = f(k[i], k[i+1], k[i+397 mod 624]) reads ahead by one word and by
// 397 (or back by 227), so a 16-wide step never reads a word the same step writes; the two scalar remainders sit
// where the far operand wraps.  Bit-identical to gen_block_base (checked by the numpy replay test).
#define PPX_MT_STEP16(i, src)                                                                      \
  {                                                                                                \
    const __m512i a = _mm512_loadu_si512((const void*)(k + (i)));                                  \
    const __m512i b = _mm512_loadu_si512((const void*)(k + (i) + 1));                              \
    const __m512i y = _mm512_or_si512(_mm512_and_si512(a, up), _mm512_and_si512(b, lw));           \
    const __mmask16 odd = _mm512_test_epi32_mask(y, one);                                          \
    __m512i r = _mm512_xor_si512(_mm512_loadu_si512((const void*)(k + (src))), _mm512_srli_epi32(y, 1)); \
    r = _mm512_mask_xor_epi32(r, odd, r, ma);                                                      \
    _mm512_storeu_si512((void*)(k + (i)), r);                                                      \
  }

__attribute__((target("avx512f,avx512bw,avx512vl,avx512dq")))
void gen_block_avx512(uint32_t* k, uint32_t* __restrict__ o) {
  const __m512i up = _mm512_set1_epi32((int)UPPER), lw = _mm512_set1_epi32((int)LOWER);
  const __m512i ma = _mm512_set1_epi32((int)MATRIX_A), one = _mm512_set1_epi32(1);
  int i = 0;
  for (; i + 16 <= MT_N - MT_M; i += 16) PPX_MT_STEP16(i, i + MT_M)
  for (; i < MT_N - MT_M; i++) k[i] = twist(k[i], k[i + 1], k[i + MT_M]);
  for (; i + 16 <= MT_N - 1; i += 16) PPX_MT_STEP16(i, i + (MT_M - MT_N))
  for (; i < MT_N - 1; i++) k[i] = twist(k[i], k[i + 1], k[i + (MT_M - MT_N)]);
  k[MT_N - 1] = twist(k[MT_N - 1], k[0], k[MT_M - 1]);
  const __m512i c1 = _mm512_set1_epi32((int)0x9d2c5680u), c2 = _mm512_set1_epi32((int)0xefc60000u);
  static_assert(MT_N % 16 == 0, "tempering runs in whole vectors");
  for (int j = 0; j < MT_N; j += 16) {
    __m512i v = _mm512_loadu_si512((const void*)(k + j));
    v = _mm512_xor_si512(v, _mm512_srli_epi32(v, 11));
    v = _mm512_xor_si512(v, _mm512_and_si512(_mm512_slli_epi32(v, 7), c1));
    v = _mm512_xor_si512(v, _mm512_and_si512(_mm512_slli_epi32(v, 15), c2));
    v = _mm512_xor_si512(v, _mm512_srli_epi32(v, 18));
    _mm512_storeu_si512((void*)(o + j), v);
  }
}

// MT19937 with block generation: the 624-word state update and the tempering run over whole blocks (16 words per
// step with AVX-512, else straight auto-vectorised loops), extraction is a buffered load.  Same output sequence as
// numpy's word-at-a-time mt19937_next.
struct Mt {
  uint32_t* key;
  int pos;
  alignas(64) uint32_t out[MT_N];
  Mt(uint32_t* k, int p) : key(k), pos(p) {
    for (int i = p; i < MT_N; ++i) {               // the unread tail of the CURRENT key block
      uint32_t y = k[i];
      y ^= (y >> 11);
      y ^= (y << 7) & 0x9d2c5680u;
      y ^= (y << 15) & 0xefc60000u;
      y ^= (y >> 18);
      out[i] = y;
    }
  }
  inline void gen() {
    if (has_avx512()) gen_block_avx512(key, out);
    else gen_block_base(key, out);
    pos = 0;
  }
  inline uint32_t next32() {
    if (pos == MT_N) gen();
    return out[pos++];
  }
  inline uint64_t next64() {                       // numpy: (uint64)next32() << 32 | next32()
    const uint64_t hi = next32();
    return (hi << 32) | next32();
  }
};

inline uint64_t random_interval(Mt& mt, uint64_t max) {
  if (max == 0) return 0;
  uint64_t mask = max, value;
  mask |= mask >> 1; mask |= mask >> 2; mask |= mask >> 4; mask |= mask >> 8; mask |= mask >> 16; mask |= mask >> 32;
  if (max <= 0xffffffffull) {
    while ((value = (mt.next32() & mask)) > max) {}
  } else {
    while ((value = (mt.next64() & mask)) > max) {}
  }
  return value;
}
}  // namespace

// Branch-free form of the rejection loop for 32-bit bounds: every draw is stored, the position only
// advances when the draw is accepted.  Identical draw sequence, no data-dependent branch to mispredict.
static inline void draw_partners(Mt& mt, int64_t n, int64_t* j_out) {
  int64_t i = n - 1;
  for (; i >= 1 && (uint64_t)i > 0xffffffffull; --i) j_out[i] = (int64_t)random_interval(mt, (uint64_t)i);
  while (i >= 1) {
    const uint32_t mask = 0xffffffffu >> __builtin_clz((uint32_t)i);
    const uint32_t v = mt.next32() & mask;
    j_out[i] = (int64_t)v;
    i -= (int64_t)(v <= (uint32_t)i);
  }
}

// 32-bit variant of draw_partners for n <= 2^31: the mask only changes when i crosses a power of two, so the
// inner loop runs with a constant mask straight over the tempered block (no per-draw clz, no call per word),
// and the partner list is int32.  Same draw sequence.
static inline void draw_partners32(Mt& mt, int64_t n, int32_t* j_out) {
  int64_t i = n - 1;
  while (i >= 1) {
    const uint32_t mask = 0xffffffffu >> __builtin_clz((uint32_t)i);
    const int64_t lo = (int64_t)(mask >> 1) + 1;            // positions [lo, mask] share this mask
    while (i >= lo) {
      if (mt.pos == MT_N) mt.gen();
      const uint32_t* __restrict__ o = mt.out;
      int p = mt.pos;
      while (p < MT_N && i >= lo) {
        const uint32_t v = o[p++] & mask;
        j_out[i] = (int32_t)v;
        i -= (int64_t)(v <= (uint32_t)i);
      }
      mt.pos = p;
    }
  }
}

// the swap partners j_i for i = n-1 .. 1 (j_out[i] = partner of position i; j_out[0] unused): the scalar reference
// of the acceptance-order draw loop below
extern "C" int ppx_np_shuffle_draws32(uint32_t* key624_host, int* pos_host, int64_t n, int32_t* j_out_host) {
  PPX_REQUIRE(key624_host && pos_host && j_out_host && n >= 0 && n <= 0x7fffffffll, "np_shuffle_draws32: bad arguments");
  PPX_REQUIRE(*pos_host >= 0 && *pos_host <= MT_N, "np_shuffle_draws32: MT19937 pos=%d out of range", *pos_host);
  Mt mt(key624_host, *pos_host);
  draw_partners32(mt, n, j_out_host);
  *pos_host = mt.pos;
  return PPX_OK;
}

// arange(n) with the swaps applied
static void np_shuffle_apply(const int64_t* j_host, int64_t n, int64_t* out_host) {
  for (int64_t i = 0; i < n; ++i) out_host[i] = i;
  for (int64_t i = n - 1; i >= 1; --i) {
    const int64_t j = j_host[i];
    const int64_t t = out_host[j];
    out_host[j] = out_host[i];
    out_host[i] = t;
  }
}

// draws and swaps back to back, on the host
extern "C" int ppx_np_permutation(uint32_t* key624_host, int* pos_host, int64_t n, int64_t* out_host) {
  PPX_REQUIRE(key624_host && pos_host && out_host && n >= 0, "np_permutation: bad arguments");
  PPX_REQUIRE(*pos_host >= 0 && *pos_host <= MT_N, "np_permutation: MT19937 pos=%d out of range", *pos_host);
  Mt mt(key624_host, *pos_host);
  int64_t* j = (int64_t*)malloc((size_t)(n > 0 ? n : 1) * sizeof(int64_t));
  if (!j) return ppx::fail(PPX_ERR_ARG, "np_permutation: out of host memory");
  draw_partners(mt, n, j);
  *pos_host = mt.pos;
  np_shuffle_apply(j, n, out_host);
  free(j);
  return PPX_OK;
}

// ------------------------------------------------------------------------------------------------
// The learner's draw loop: the accepted partners in ACCEPTANCE order (acc[r] is the partner of position i = n-1-r).
// ------------------------------------------------------------------------------------------------
namespace {
#define PPX_DRAW_SCALAR_STEP()                                   \
  {                                                              \
    const uint32_t v = o[p++] & mask;                            \
    acc[r] = (int32_t)v;                                         \
    const int64_t ok = (int64_t)(v <= (uint32_t)i);              \
    r += ok;                                                     \
    i -= ok;                                                     \
  }

void draw_acc_base(Mt& mt, int64_t n, int32_t* acc) {
  int64_t i = n - 1, r = 0;
  while (i >= 1) {
    const uint32_t mask = 0xffffffffu >> __builtin_clz((uint32_t)i);
    const int64_t lo = (int64_t)(mask >> 1) + 1;
    while (i >= lo) {
      if (mt.pos == MT_N) mt.gen();
      const uint32_t* __restrict__ o = mt.out;
      int p = mt.pos;
      while (p < MT_N && i >= lo) PPX_DRAW_SCALAR_STEP()
      mt.pos = p;
    }
  }
}

// 64 (then 16) draws per step: with i the position at the start of the step, a draw v is certainly accepted if
// v <= i - (W-1) (at most W-1 accepts precede it inside the step) and certainly rejected if v > i; a step holding a draw
// in between (probability ~ W^2 / 2^k for a k-bit mask) falls to the next narrower path.  Accepted draws are packed with
// a register compress and a full-width store: the lanes past the packed ones land on entries a later step rewrites
// (r + 16 <= n - 1 because the vector paths stop 16 positions above the end of the mask's range).
__attribute__((target("avx512f,avx512bw,avx512vl,avx512dq,popcnt")))
void draw_acc_avx512(Mt& mt, int64_t n, int32_t* acc) {
  int64_t i = n - 1, r = 0;
  while (i >= 1) {
    const uint32_t mask = 0xffffffffu >> __builtin_clz((uint32_t)i);
    const int64_t lo = (int64_t)(mask >> 1) + 1;
    const __m512i maskv = _mm512_set1_epi32((int)mask);
    while (i >= lo) {
      if (mt.pos == MT_N) mt.gen();
      const uint32_t* __restrict__ o = mt.out;
      int p = mt.pos;
      while (p + 64 <= MT_N && i - 64 >= lo) {
        const uint32_t ii = (uint32_t)i;
        const __m512i top = _mm512_set1_epi32((int)ii), safe = _mm512_set1_epi32((int)(ii - 63u));
        const __m512i v0 = _mm512_and_si512(_mm512_loadu_si512((const void*)(o + p)), maskv);
        const __m512i v1 = _mm512_and_si512(_mm512_loadu_si512((const void*)(o + p + 16)), maskv);
        const __m512i v2 = _mm512_and_si512(_mm512_loadu_si512((const void*)(o + p + 32)), maskv);
        const __m512i v3 = _mm512_and_si512(_mm512_loadu_si512((const void*)(o + p + 48)), maskv);
        const __mmask16 a0 = _mm512_cmple_epu32_mask(v0, top), a1 = _mm512_cmple_epu32_mask(v1, top);
        const __mmask16 a2 = _mm512_cmple_epu32_mask(v2, top), a3 = _mm512_cmple_epu32_mask(v3, top);
        const __mmask16 s0 = _mm512_cmple_epu32_mask(v0, safe), s1 = _mm512_cmple_epu32_mask(v1, safe);
        const __mmask16 s2 = _mm512_cmple_epu32_mask(v2, safe), s3 = _mm512_cmple_epu32_mask(v3, safe);
        if (((a0 ^ s0) | (a1 ^ s1) | (a2 ^ s2) | (a3 ^ s3)) != 0) break;            // ambiguous: 16-wide path below
        const int64_t c0 = __builtin_popcount((unsigned)a0), c1 = __builtin_popcount((unsigned)a1);
        const int64_t c2 = __builtin_popcount((unsigned)a2), c3 = __builtin_popcount((unsigned)a3);
        _mm512_storeu_si512((void*)(acc + r), _mm512_maskz_compress_epi32(a0, v0));
        _mm512_storeu_si512((void*)(acc + r + c0), _mm512_maskz_compress_epi32(a1, v1));
        _mm512_storeu_si512((void*)(acc + r + c0 + c1), _mm512_maskz_compress_epi32(a2, v2));
        _mm512_storeu_si512((void*)(acc + r + c0 + c1 + c2), _mm512_maskz_compress_epi32(a3, v3));
        const int64_t c = c0 + c1 + c2 + c3;
        r += c;
        i -= c;
        p += 64;
      }
      for (int blk = 0; blk < 4 && p + 16 <= MT_N && i - 16 >= lo; ++blk) {          // <= one 64-step's worth, then retry wide
        const __m512i v = _mm512_and_si512(_mm512_loadu_si512((const void*)(o + p)), maskv);
        const uint32_t ii = (uint32_t)i;
        const __mmask16 sure = _mm512_cmple_epu32_mask(v, _mm512_set1_epi32((int)(ii - 15u)));
        const __mmask16 maybe = _mm512_cmple_epu32_mask(v, _mm512_set1_epi32((int)ii));
        if (sure == maybe) {
          _mm512_storeu_si512((void*)(acc + r), _mm512_maskz_compress_epi32(sure, v));
          const int64_t c = (int64_t)__builtin_popcount((unsigned)sure);
          r += c;
          i -= c;
          p += 16;
        } else {
          for (int q = 0; q < 16; ++q) PPX_DRAW_SCALAR_STEP()
        }
      }
      while (p < MT_N && i >= lo && (p + 16 > MT_N || i - 16 < lo)) PPX_DRAW_SCALAR_STEP()
      mt.pos = p;
    }
  }
}
}  // namespace

extern "C" int ppx_np_shuffle_draws32_stream(uint32_t* key624_host, int* pos_host, int64_t n, int32_t* acc_host) {
  PPX_REQUIRE(key624_host && pos_host && acc_host && n >= 0 && n <= 0x7fffffffll, "np_shuffle_draws32_stream: bad arguments");
  PPX_REQUIRE(*pos_host >= 0 && *pos_host <= MT_N, "np_shuffle_draws32_stream: MT19937 pos=%d out of range", *pos_host);
  Mt mt(key624_host, *pos_host);
  if (has_avx512()) draw_acc_avx512(mt, n, acc_host);
  else draw_acc_base(mt, n, acc_host);
  *pos_host = mt.pos;
  return PPX_OK;
}
