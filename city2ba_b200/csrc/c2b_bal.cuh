// c2b_bal.cuh — BAL files (src/baproblem.rs:709-764) encoded on the device.
//
// Text.  Every f64 is printed the way Rust's `{}` prints it: the shortest decimal significand that parses back to
// the same double (among the shortest, the one closest to the exact binary value; an exact tie goes to the even
// digit), written positionally, never with an exponent; NaN is "NaN", infinities "inf" / "-inf", -0.0 is "-0".
// The significand comes from Ryu (Adams, "Ryu: fast float-to-string conversion", PLDI 2018), restated here:
// the rounding interval [v - ulp/2, v + ulp/2] (a quarter ulp below powers of two) is scaled to a decimal
// exponent with 128-bit fixed-point multipliers by 5^q or 5^-q, digits are removed while the shortened interval
// still contains a number, and the last removed digit rounds.  It is exact: the paper proves that 125-bit
// multipliers (c2b_bal_tables.h, generated with exact integers) give floor(m * 10^-q * 2^e2) without error for
// every f64, and the trailing-zero flags track the cases where the product is an exact integer.
// Lines: a length pass (one length per line), an exclusive scan (c2b_sort.cuh), a write pass that puts each
// line's bytes at its offset.  The driver (c2b_api.cu, bal_write) runs them over windows of lines and cuts
// chunks of at most a byte budget at line ends found in the scan.
//
// Binary.  Every item is an 8-byte big-endian word and the byte offset of camera c's count word is
// 24 + 8c + 24 offsets[c]; each thread writes one word, found by a binary search over that closed form.
#pragma once
#include "c2b_bal_tables.h"
#include "c2b_common.cuh"

namespace c2b {

constexpr int BAL_THREADS = 256;

// one problem on the device
struct BalView {
  const double *vecs;  // C x 9 camera vectors (to_vec, computed on the host: c2b_camera_to_vec)
  const double *pts;   // P x 3
  const uint64_t *off; // C + 1
  const uint32_t *idx; // O
  const double *uv;    // O x 2
  uint64_t C, P, O;
};

// ---- shortest round-trip digits (Ryu) ------------------------------------------------------------------
__device__ __forceinline__ uint32_t bal_pow5bits(int32_t e) { return (uint32_t)(((e * 1217359) >> 19) + 1); }
__device__ __forceinline__ uint32_t bal_log10pow2(int32_t e) { return (uint32_t)((e * 78913) >> 18); }
__device__ __forceinline__ uint32_t bal_log10pow5(int32_t e) { return (uint32_t)((e * 732923) >> 20); }

__device__ __forceinline__ uint32_t bal_pow5_factor(uint64_t v) {
  uint32_t n = 0;
  while (v % 5 == 0) {
    v /= 5;
    ++n;
  }
  return n;
}

// (m * mul) >> j for a 128-bit mul = {lo, hi} and 64 <= j < 128
__device__ __forceinline__ uint64_t bal_mul_shift(uint64_t m, const uint64_t *mul, int32_t j) {
  const uint64_t hi0 = __umul64hi(m, mul[0]);
  const uint64_t lo2 = m * mul[1], hi2 = __umul64hi(m, mul[1]);
  const uint64_t lo = lo2 + hi0;
  const uint64_t hi = hi2 + (lo < hi0);
  const int s = j - 64;
  return s == 0 ? lo : (hi << (64 - s)) | (lo >> s);
}

// finite, nonzero x = m * 10^e with the fewest digits (trailing zeros of m removed)
__device__ __forceinline__ void bal_shortest(uint64_t bits, uint64_t &out_m, int32_t &out_e) {
  const uint64_t ieee_m = bits & ((1ull << 52) - 1);
  const uint32_t ieee_e = (uint32_t)((bits >> 52) & 0x7ff);
  int32_t e2;
  uint64_t m2;
  if (ieee_e == 0) {
    e2 = 1 - 1023 - 52 - 2;
    m2 = ieee_m;
  } else {
    e2 = (int32_t)ieee_e - 1023 - 52 - 2;
    m2 = (1ull << 52) | ieee_m;
  }
  const bool accept_bounds = (m2 & 1) == 0;  // round-half-even parsing accepts the interval's ends
  const uint64_t mv = 4 * m2;
  const uint32_t mm_shift = ieee_m != 0 || ieee_e <= 1;  // 0: the lower neighbour is a quarter ulp away
  uint64_t vr, vp, vm;
  int32_t e10;
  bool vm_tz = false, vr_tz = false;
  if (e2 >= 0) {
    const uint32_t q = bal_log10pow2(e2) - (e2 > 3);
    e10 = (int32_t)q;
    const int32_t k = BAL_POW5_INV_BITCOUNT + (int32_t)bal_pow5bits((int32_t)q) - 1;
    const int32_t i = -e2 + (int32_t)q + k;
    const uint64_t *mul = BAL_POW5_INV_SPLIT[q];
    vr = bal_mul_shift(4 * m2, mul, i);
    vp = bal_mul_shift(4 * m2 + 2, mul, i);
    vm = bal_mul_shift(4 * m2 - 1 - mm_shift, mul, i);
    if (q <= 21) {
      // at most one of mp, mv, mm is a multiple of 5
      if (mv % 5 == 0)
        vr_tz = bal_pow5_factor(mv) >= q;
      else if (accept_bounds)
        vm_tz = bal_pow5_factor(mv - 1 - mm_shift) >= q;
      else
        vp -= bal_pow5_factor(mv + 2) >= q;
    }
  } else {
    const uint32_t q = bal_log10pow5(-e2) - (-e2 > 1);
    e10 = (int32_t)q + e2;
    const int32_t i = -e2 - (int32_t)q;
    const int32_t k = (int32_t)bal_pow5bits(i) - BAL_POW5_BITCOUNT;
    const int32_t j = (int32_t)q - k;
    const uint64_t *mul = BAL_POW5_SPLIT[i];
    vr = bal_mul_shift(4 * m2, mul, j);
    vp = bal_mul_shift(4 * m2 + 2, mul, j);
    vm = bal_mul_shift(4 * m2 - 1 - mm_shift, mul, j);
    if (q <= 1) {
      // mv = 4 m2 has two trailing zero bits; mm has one iff mm_shift == 1; mp = mv + 2 has one
      vr_tz = true;
      if (accept_bounds)
        vm_tz = mm_shift == 1;
      else
        --vp;
    } else if (q < 63) {
      vr_tz = (mv & ((1ull << q) - 1)) == 0;  // the product has q trailing zeros iff mv has q trailing zero bits
    }
  }
  int32_t removed = 0;
  uint64_t output;
  if (vm_tz || vr_tz) {
    // rare general case: track whether everything removed so far was zero
    uint32_t last = 0;
    while (vp / 10 > vm / 10) {
      vm_tz &= vm % 10 == 0;
      vr_tz &= last == 0;
      last = (uint32_t)(vr % 10);
      vr /= 10;
      vp /= 10;
      vm /= 10;
      ++removed;
    }
    if (vm_tz) {
      while (vm % 10 == 0) {
        vr_tz &= last == 0;
        last = (uint32_t)(vr % 10);
        vr /= 10;
        vp /= 10;
        vm /= 10;
        ++removed;
      }
    }
    if (vr_tz && last == 5 && vr % 2 == 0) last = 4;  // exactly ...50...0: round half to even
    output = vr + ((vr == vm && (!accept_bounds || !vm_tz)) || last >= 5);
  } else {
    bool round_up = false;
    if (vp / 100 > vm / 100) {
      round_up = vr % 100 >= 50;
      vr /= 100;
      vp /= 100;
      vm /= 100;
      removed += 2;
    }
    while (vp / 10 > vm / 10) {
      round_up = vr % 10 >= 5;
      vr /= 10;
      vp /= 10;
      vm /= 10;
      ++removed;
    }
    output = vr + (vr == vm || round_up);
  }
  int32_t e = e10 + removed;
  while (output % 10 == 0) {
    output /= 10;
    ++e;
  }
  out_m = output;
  out_e = e;
}

__device__ __forceinline__ int bal_ndigits(uint64_t v) {
  int n = 1;
  while (v >= 10) {
    v /= 10;
    ++n;
  }
  return n;
}

// ---- text sinks: the length pass counts, the write pass stores ---------------------------------------------
template <bool W>
struct BalSink {
  char *p;
  uint32_t n;
  __device__ __forceinline__ void put(char c) {
    if (W) p[n] = c;
    ++n;
  }
  __device__ __forceinline__ void zeros(int k) {
    if (W)
      for (int j = 0; j < k; ++j) p[n + j] = '0';
    n += (uint32_t)k;
  }
  // the nd digits of v (nd = bal_ndigits(v)); a '.' after the first `point` digits when 0 < point < nd
  __device__ __forceinline__ void digits(uint64_t v, int nd, int point) {
    const int dot = (point > 0 && point < nd) ? 1 : 0;
    if (W) {
      for (int j = nd - 1; j >= 0; --j) {
        p[n + j + (dot && j >= point)] = (char)('0' + v % 10);
        v /= 10;
      }
      if (dot) p[n + point] = '.';
    }
    n += (uint32_t)(nd + dot);
  }
  __device__ __forceinline__ void u64(uint64_t v) { digits(v, bal_ndigits(v), 0); }
  __device__ __forceinline__ void f64(double x) {
    const uint64_t bits = (uint64_t)__double_as_longlong(x);
    const bool neg = bits >> 63;
    const uint32_t ieee_e = (uint32_t)((bits >> 52) & 0x7ff);
    const uint64_t ieee_m = bits & ((1ull << 52) - 1);
    if (ieee_e == 0x7ff) {
      if (ieee_m) {
        put('N');
        put('a');
        put('N');
      } else {
        if (neg) put('-');
        put('i');
        put('n');
        put('f');
      }
      return;
    }
    if (neg) put('-');
    if (ieee_e == 0 && ieee_m == 0) {
      put('0');
      return;
    }
    uint64_t m;
    int32_t e;
    bal_shortest(bits, m, e);
    const int nd = bal_ndigits(m);
    if (e >= 0) {
      digits(m, nd, 0);
      zeros(e);
    } else if (nd + e > 0) {
      digits(m, nd, nd + e);
    } else {
      put('0');
      put('.');
      zeros(-(nd + e));
      digits(m, nd, 0);
    }
  }
};

// line L of the text file: the header, O observation lines, C camera lines, P point lines
template <bool W>
__device__ __forceinline__ uint32_t bal_text_line(const BalView &v, uint64_t L, char *out) {
  BalSink<W> s{out, 0};
  if (L == 0) {
    s.u64(v.C);
    s.put(' ');
    s.u64(v.P);
    s.put(' ');
    s.u64(v.O);
  } else if (L <= v.O) {
    const uint64_t o = L - 1;
    uint64_t lo = 0, hi = v.C;  // the camera c with off[c] <= o < off[c + 1]
    while (hi - lo > 1) {
      const uint64_t mid = (lo + hi) >> 1;
      if (v.off[mid] <= o)
        lo = mid;
      else
        hi = mid;
    }
    s.u64(lo);
    s.put(' ');
    s.u64(v.idx[o]);
    s.put(' ');
    s.f64(v.uv[2 * o]);
    s.put(' ');
    s.f64(v.uv[2 * o + 1]);
  } else if (L <= v.O + v.C) {
    const double *x = v.vecs + 9 * (L - 1 - v.O);
    for (int k = 0; k < 9; ++k) {
      if (k) s.put(' ');
      s.f64(x[k]);
    }
  } else {
    const double *x = v.pts + 3 * (L - 1 - v.O - v.C);
    s.f64(x[0]);
    s.put(' ');
    s.f64(x[1]);
    s.put(' ');
    s.f64(x[2]);
  }
  s.put('\n');
  return s.n;
}

// lens[i] = length of line first + i, i < n
__global__ void __launch_bounds__(BAL_THREADS) k_bal_text_len(BalView v, uint64_t first, uint32_t n,
                                                              uint32_t *__restrict__ lens) {
  const uint32_t i = blockIdx.x * BAL_THREADS + threadIdx.x;
  if (i < n) lens[i] = bal_text_line<false>(v, first + i, nullptr);
}

// The chunk: the most lines of the window (at least one) whose bytes fit `budget`.  start = exclusive scan of the
// window's n line lengths, total = their sum.  res[0] = lines, res[1] = bytes.
__global__ void k_bal_text_cut(const uint32_t *__restrict__ start, const uint32_t *__restrict__ total, uint32_t n,
                               uint32_t budget, uint32_t *res) {
  uint32_t lo = 1, hi = n;  // end of line k-1 = start[k] (k < n) or total: the largest k with end <= budget
  while (lo < hi) {
    const uint32_t mid = lo + (hi - lo + 1) / 2;
    const uint32_t end = mid < n ? start[mid] : *total;
    if (end <= budget)
      lo = mid;
    else
      hi = mid - 1;
  }
  res[0] = lo;
  res[1] = lo < n ? start[lo] : *total;
}

__global__ void __launch_bounds__(BAL_THREADS) k_bal_text_write(BalView v, uint64_t first, uint32_t n,
                                                                const uint32_t *__restrict__ start,
                                                                char *__restrict__ out) {
  const uint32_t i = blockIdx.x * BAL_THREADS + threadIdx.x;
  if (i < n) bal_text_line<true>(v, first + i, out + start[i]);
}

__device__ __forceinline__ uint64_t bal_bswap64(uint64_t x) {
  return ((uint64_t)__byte_perm((uint32_t)x, 0, 0x0123) << 32) | __byte_perm((uint32_t)(x >> 32), 0, 0x0123);
}

// words [w0, w0 + n) of the binary file
__global__ void __launch_bounds__(BAL_THREADS) k_bal_binary(BalView v, uint64_t w0, uint64_t n,
                                                            uint64_t *__restrict__ out) {
  const uint64_t t = (uint64_t)blockIdx.x * BAL_THREADS + threadIdx.x;
  if (t >= n) return;
  const uint64_t w = w0 + t;
  const uint64_t obs_words = v.C + 3 * v.O;  // count word + 3 words per observation
  uint64_t word;
  if (w < 3) {
    word = w == 0 ? v.C : w == 1 ? v.P : v.O;
  } else if (w < 3 + obs_words) {
    const uint64_t r = w - 3;  // camera c's block starts at word c + 3 off[c]
    uint64_t lo = 0, hi = v.C;
    while (hi - lo > 1) {
      const uint64_t mid = (lo + hi) >> 1;
      if (mid + 3 * v.off[mid] <= r)
        lo = mid;
      else
        hi = mid;
    }
    const uint64_t d = r - (lo + 3 * v.off[lo]);
    if (d == 0) {
      word = v.off[lo + 1] - v.off[lo];
    } else {
      const uint64_t o = v.off[lo] + (d - 1) / 3;
      const uint32_t f = (uint32_t)((d - 1) % 3);
      word = f == 0 ? (uint64_t)v.idx[o] : (uint64_t)__double_as_longlong(v.uv[2 * o + f - 1]);
    }
  } else if (w < 3 + obs_words + 9 * v.C) {
    word = (uint64_t)__double_as_longlong(v.vecs[w - 3 - obs_words]);
  } else {
    word = (uint64_t)__double_as_longlong(v.pts[w - 3 - obs_words - 9 * v.C]);
  }
  out[t] = bal_bswap64(word);
}

}  // namespace c2b
