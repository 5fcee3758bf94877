// Pure arithmetic of the end-of-step reductions (tail.cuh, post_kernel.cuh, compact_kernel), host and
// device: the CPU tests compile this header on its own and check it against exact references.
//
// Exact order-independent sums of fp32 values.  A finite fp32 value q is m * 2^e with m a 24-bit integer
// and e in [-149, 104], so q is the integer m << (e + 149) in units of 2^-149.  The accumulator holds that
// integer as XS_WORDS signed 64-bit words; word k carries multiples of 2^(32k - 149).  One addend touches
// two adjacent words, each with a magnitude below 2^32, so 2^31 addends cannot overflow a word, and the
// carries are resolved once, when the sum is read (xs_to_double).  Integer additions commute: the per-slab
// (xs_pieces) and per-launch sums are fire-and-forget atomics and the result does not depend on their order.  Words
// 0..8 receive addends, word 9 only carries: the range reaches past 2^171, above 2^31 * FLT_MAX.
// NaN and +-Inf are not summed; they set flags (FX_*), which decide the result on their own.
#pragma once
#include <stdint.h>
#ifndef __CUDA_ARCH__
#include <string.h>
#endif

#ifdef __CUDACC__
#define GFB_HD __host__ __device__ __forceinline__
#else
#define GFB_HD inline
#endif

namespace gfb {

constexpr int XS_WORDS = 10;
constexpr int XS_E0 = -149;  // word k carries multiples of 2^(32k + XS_E0)
constexpr uint32_t FX_NAN = 1u, FX_POS_INF = 2u, FX_NEG_INF = 4u;

GFB_HD uint32_t xs_bits(float q) {
#ifdef __CUDA_ARCH__
  return __float_as_uint(q);
#else
  uint32_t u;
  memcpy(&u, &q, sizeof u);
  return u;
#endif
}

GFB_HD double xs_double_from_bits(long long b) {
#ifdef __CUDA_ARCH__
  return __longlong_as_double(b);
#else
  double d;
  memcpy(&d, &b, sizeof d);
  return d;
#endif
}
GFB_HD double xs_pow2(int e) { return xs_double_from_bits((long long)(e + 1023) << 52); }  // (-1022 <= e <= 1023)

// q -> its increments of words k (lo) and k + 1 (hi), both of magnitude below 2^32; returns k, or -1 for
// +-0 and for NaN / +-Inf, which set `flags` instead
GFB_HD int xs_split(float q, long long& lo, long long& hi, uint32_t& flags) {
  const uint32_t u = xs_bits(q);
  const uint32_t ef = (u >> 23) & 0xffu;
  uint32_t m = u & 0x7fffffu;
  lo = hi = 0;
  if (ef == 0xffu) {
    flags |= m ? FX_NAN : ((u >> 31) ? FX_NEG_INF : FX_POS_INF);
    return -1;
  }
  if (ef == 0u && m == 0u) return -1;
  int s = 0;  // q = m * 2^(s + XS_E0); a denormal has e = -149, s = 0
  if (ef) {
    m |= 0x800000u;
    s = (int)ef - 1;
  }
  const unsigned long long v = (unsigned long long)m << (s & 31);
  lo = (long long)(v & 0xffffffffull);
  hi = (long long)(v >> 32);
  if (u >> 31) {
    lo = -lo;
    hi = -hi;
  }
  return s >> 5;
}

// A slab sums a word's increments as two signed 32-bit counters of 16-bit pieces (units 1 and 2^16):
// native shared atomics.  |piece| < 2^16, so 2^15 addends per slab cannot overflow a counter.
GFB_HD void xs_pieces(long long v, int& p0, int& p1) {
  const long long a = v < 0 ? -v : v;
  p0 = (int)(a & 0xffff);
  p1 = (int)(a >> 16);
  if (v < 0) {
    p0 = -p0;
    p1 = -p1;
  }
}
GFB_HD long long xs_join(int c0, int c1) { return (long long)c0 + (long long)c1 * 65536; }

// words 0..XS_WORDS-2 into [0, 2^32), the carries (and the sign) into the last word
GFB_HD void xs_normalize(long long* w) {
  for (int k = 0; k < XS_WORDS - 1; ++k) {
    const long long c = w[k] >> 32;  // (arithmetic shift: floor division by 2^32)
    w[k] &= 0xffffffffll;
    w[k + 1] += c;
  }
}

// the accumulated sum as a double (NaN / +-Inf from the flags): NaN if any addend was NaN or both
// infinities were added, else the infinity that was added, else the exact sum rounded to double (the
// words are summed from the top, all of one sign: within 2 ulp of double).  A zero sum is +0.
GFB_HD double xs_to_double(const long long* acc, uint32_t flags) {
  if ((flags & FX_NAN) || ((flags & FX_POS_INF) && (flags & FX_NEG_INF))) return xs_double_from_bits(0x7ff8000000000000ll);
  if (flags & FX_POS_INF) return xs_double_from_bits(0x7ff0000000000000ll);
  if (flags & FX_NEG_INF) return xs_double_from_bits((long long)0xfff0000000000000ull);
  long long w[XS_WORDS];
  for (int k = 0; k < XS_WORDS; ++k) w[k] = acc[k];
  xs_normalize(w);
  const bool neg = w[XS_WORDS - 1] < 0;
  if (neg) {  // the magnitude, in the same normal form
    for (int k = 0; k < XS_WORDS; ++k) w[k] = -w[k];
    xs_normalize(w);
  }
  double d = 0.0;
  for (int k = XS_WORDS - 1; k >= 0; --k) d += (double)w[k] * xs_pow2(32 * k + XS_E0);
  return neg ? -d : d;
}

// logged mean of the sum over n > 0 values: the sum itself when it is NaN or past the fp32 range (an fp32
// sum of the same values overflows too), else sum / n rounded to fp32
GFB_HD float xs_mean(double sum, double n) {
  const float s = (float)sum;
  if (s != s || s > 3.4028234663852886e38f || s < -3.4028234663852886e38f) return s;
  return (float)(sum / n);
}

// ---------------------------------------------------------------------------------------------
// compact_kernel's launch geometry: at most CMP_MAX_BLOCKS blocks, each a multiple of CMP_THREADS words
// (the 16-byte loads of the words before a block's range), and only blocks whose range starts inside the
// n_words mask words: together they cover [0, n_words) exactly.
// ---------------------------------------------------------------------------------------------
constexpr int CMP_THREADS = 256;
constexpr int CMP_MAX_BLOCKS = 128;
struct CompactGeometry {
  int n_blocks, words_per_block;
};
GFB_HD CompactGeometry compact_geometry(int n_words) {
  const int want = (n_words + CMP_THREADS - 1) / CMP_THREADS;
  const int n0 = want < 1 ? 1 : (want > CMP_MAX_BLOCKS ? CMP_MAX_BLOCKS : want);
  int per = ((n_words + n0 - 1) / n0 + CMP_THREADS - 1) / CMP_THREADS * CMP_THREADS;
  if (per < CMP_THREADS) per = CMP_THREADS;
  const int n_blocks = (n_words + per - 1) / per;
  return CompactGeometry{n_blocks < 1 ? 1 : n_blocks, per};
}

}  // namespace gfb
