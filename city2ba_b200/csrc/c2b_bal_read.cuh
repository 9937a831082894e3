// c2b_bal_read.cuh — BAL files (src/baproblem.rs:580-706) parsed on the device.
//
// Text.  A chunk of the file (complete tokens only: the driver cuts it after its last whitespace byte) is in device
// memory.  k_bal_tok_flags packs one token-start flag per byte into ballot words and counts them; an exclusive scan
// of the counts (c2b_sort.cuh) gives every word the ordinal of its first token within the chunk, and the chunk's
// first ordinal is a device counter that k_bal_tok_advance moves on.  The layout after the header is fixed, so the
// ordinal alone says what a token is (an observation's field, a camera component, a point coordinate), and
// k_bal_parse_text stores every token in place.
//
// Numbers: Eisel-Lemire (Lemire, "Number Parsing at a Gigabyte per Second", 2021).  The first 19 significant digits
// form w, the token's decimal exponent q; w * 5^q is formed with a truncated 128-bit power of five
// (c2b_bal_tables.h, BAL_POW5_128), which is always enough for an exact w (Mushtak and Lemire, "Fast number parsing
// without fallback", 2023).  With more digits the value lies in [w, w + 1) * 10^q: when both ends round to the same
// double that is the answer, otherwise the token goes to the host (std::from_chars) through a side buffer.
//
// Binary.  One thread per big-endian word; the camera of an observation word is found by a binary search over the
// closed form of the camera blocks' starts (c + 3 offsets[c] words after the header), the inverse of k_bal_binary.
#pragma once
#include "c2b_bal_tables.h"
#include "c2b_common.cuh"

namespace c2b {

constexpr int BALR_THREADS = 256;

__host__ __device__ __forceinline__ bool bal_ws(char c) {
  return c == ' ' || c == '\t' || c == '\n' || c == '\v' || c == '\f' || c == '\r';
}

// nom's digit1 as a u64: false for an empty token, a non-digit or an overflow
__host__ __device__ __forceinline__ bool bal_parse_index(const char *s, uint32_t len, uint64_t &v) {
  if (len == 0) return false;
  v = 0;
  for (uint32_t i = 0; i < len; ++i) {
    const uint32_t d = (uint32_t)(unsigned char)s[i] - '0';
    if (d > 9) return false;
    if (v > (0xffffffffffffffffull - d) / 10) return false;
    v = v * 10 + d;
  }
  return true;
}

// Eisel-Lemire for w != 0: the bits of the nearest double to w * 10^q (fast_float's compute_float, restated)
__device__ __forceinline__ uint64_t bal_el_bits(int64_t q, uint64_t w) {
  if (q < BAL_Q_MIN) return 0;
  if (q > BAL_Q_MAX) return 0x7ff0000000000000ull;
  const int lz = __clzll((long long)w);
  w <<= lz;
  const uint64_t *p5 = BAL_POW5_128[q - BAL_Q_MIN];  // {low, high}
  uint64_t lo = w * p5[1], hi = __umul64hi(w, p5[1]);
  constexpr uint64_t mask = 0xffffffffffffffffull >> 55;  // 52 + 3 bits of precision are needed
  if ((hi & mask) == mask) {
    const uint64_t hi2 = __umul64hi(w, p5[0]);
    lo += hi2;
    hi += lo < hi2;
  }
  const int upper = (int)(hi >> 63);
  const int shift = upper + 64 - 52 - 3;
  uint64_t m = hi >> shift;
  int32_t p2 = (int32_t)(((152170 + 65536) * (int32_t)q) >> 16) + 63 + upper - lz + 1023;
  if (p2 <= 0) {  // subnormal (an exact halfway case cannot occur here)
    if (-p2 + 1 >= 64) return 0;
    m >>= -p2 + 1;
    m += m & 1;
    m >>= 1;
    return m;  // a carry into bit 52 is the smallest normal: the same bits
  }
  // round half to even: only an exact product (low word <= 1) in the range of q where that can happen
  if (lo <= 1 && q >= -4 && q <= 23 && (m & 3) == 1 && (m << shift) == hi) m &= ~1ull;
  m += m & 1;
  m >>= 1;
  if (m >= (2ull << 52)) {
    m = 1ull << 52;
    ++p2;
  }
  m &= ~(1ull << 52);
  if (p2 >= 0x7ff) return 0x7ff0000000000000ull;
  return ((uint64_t)p2 << 52) | m;
}

enum { BAL_NUM_OK = 0, BAL_NUM_BAD = 1, BAL_NUM_SLOW = 2 };

// Rust's f64::from_str grammar; BAL_NUM_SLOW: w and w + 1 round differently (more than 19 significant digits),
// *near_inf then says whether the two candidates are the largest finite double and infinity
__device__ __forceinline__ int bal_parse_f64(const char *s, uint32_t len, uint64_t &bits, bool &near_inf) {
  uint32_t i = 0;
  const bool neg = len > 0 && s[0] == '-';
  if (len > 0 && (s[0] == '-' || s[0] == '+')) i = 1;
  if (i == len) return BAL_NUM_BAD;
  const uint64_t sign = neg ? 0x8000000000000000ull : 0;
  const char c0 = s[i] | 0x20;
  if (c0 == 'i' || c0 == 'n') {
    const char *word = c0 == 'n' ? "nan" : "infinity";
    const uint32_t rest = len - i;
    if (!(rest == 3 || (c0 == 'i' && rest == 8))) return BAL_NUM_BAD;
    for (uint32_t k = 0; k < rest; ++k)
      if ((s[i + k] | 0x20) != word[k]) return BAL_NUM_BAD;
    bits = sign | (c0 == 'n' ? 0x7ff8000000000000ull : 0x7ff0000000000000ull);
    return BAL_NUM_OK;
  }
  uint64_t w = 0;
  int nd = 0;                // significant digits in w
  int64_t q = 0;             // decimal exponent of w
  bool truncated = false;    // a nonzero digit did not fit in w
  bool any = false;
  for (; i < len; ++i) {
    const uint32_t d = (uint32_t)(unsigned char)s[i] - '0';
    if (d > 9) break;
    any = true;
    if (nd < 19) {
      if (w || d) {
        w = w * 10 + d;
        ++nd;
      }
    } else {
      ++q;
      truncated |= d != 0;
    }
  }
  if (i < len && s[i] == '.') {
    for (++i; i < len; ++i) {
      const uint32_t d = (uint32_t)(unsigned char)s[i] - '0';
      if (d > 9) break;
      any = true;
      if (nd < 19) {
        --q;
        if (w || d) {
          w = w * 10 + d;
          ++nd;
        }
      } else {
        truncated |= d != 0;
      }
    }
  }
  if (!any) return BAL_NUM_BAD;
  if (i < len && (s[i] | 0x20) == 'e') {
    ++i;
    bool eneg = false;
    if (i < len && (s[i] == '-' || s[i] == '+')) eneg = s[i++] == '-';
    if (i == len) return BAL_NUM_BAD;
    int64_t e = 0;
    for (; i < len; ++i) {
      const uint32_t d = (uint32_t)(unsigned char)s[i] - '0';
      if (d > 9) return BAL_NUM_BAD;
      if (e < 100000000000ll) e = e * 10 + d;  // saturates far outside every exponent that matters
    }
    q += eneg ? -e : e;
  }
  if (i != len) return BAL_NUM_BAD;
  if (w == 0) {
    bits = sign;
    return BAL_NUM_OK;
  }
  const uint64_t a = bal_el_bits(q, w);
  if (truncated) {
    const uint64_t b = bal_el_bits(q, w + 1);
    if (a != b) {
      near_inf = b == 0x7ff0000000000000ull;
      return BAL_NUM_SLOW;
    }
  }
  bits = sign | a;
  return BAL_NUM_OK;
}

// a token the device leaves to the host: its ordinal and where it lies in the chunk; len bit 31: near infinity
struct BalSlow {
  uint64_t ordinal;
  uint32_t pos, len;
};

struct BalTextArgs {
  const char *buf;           // the chunk
  uint32_t n;                // its bytes
  const uint32_t *words;     // token-start ballot words
  const uint32_t *first;     // exclusive scan of their popcounts
  const uint64_t *base;      // ordinal of the chunk's first token
  uint64_t file_off;         // file offset of buf[0]
  uint64_t C, P, O;
  uint32_t *cam_of;          // O: camera of each observation, file order
  uint32_t *idx;             // O: point of each observation, file order
  double *uv;                // 2 O, file order
  double *vecs;              // 9 C
  double *pts;               // 3 P
  unsigned long long *err;   // [0] first malformed token, [1] first index out of range (file offsets)
  BalSlow *slow;
  uint32_t *n_slow;
};

// the f64 a number token of ordinal t is stored in (t past the header and before the end of the points, and not an
// observation's index)
__device__ __forceinline__ double *bal_num_slot(uint64_t t, uint64_t C, uint64_t O, double *uv, double *vecs,
                                                double *pts) {
  const uint64_t r = t - 3;
  if (r < 4 * O) return uv + 2 * (r / 4) + (r % 4) - 2;
  if (r - 4 * O < 9 * C) return vecs + (r - 4 * O);
  return pts + (r - 4 * O - 9 * C);
}

// words[w] = token-start flags of bytes [32 w, 32 w + 32), counts[w] = their number.  Byte 0 starts a token when it
// is not whitespace: a chunk begins after a whitespace byte or at the start of the file.
__global__ void __launch_bounds__(BALR_THREADS) k_bal_tok_flags(const char *__restrict__ buf, uint32_t n,
                                                                uint32_t *__restrict__ words,
                                                                uint32_t *__restrict__ counts) {
  const uint32_t i = blockIdx.x * BALR_THREADS + threadIdx.x;
  bool start = false;
  if (i < n) start = !bal_ws(buf[i]) && (i == 0 || bal_ws(buf[i - 1]));
  const uint32_t b = __ballot_sync(0xffffffffu, start);
  if ((threadIdx.x & 31) == 0 && i < n) {
    words[i >> 5] = b;
    counts[i >> 5] = __popc(b);
  }
}

// one thread per ballot word: every token that starts in its 32 bytes
__global__ void __launch_bounds__(BALR_THREADS) k_bal_parse_text(BalTextArgs a, uint32_t n_words) {
  const uint32_t wi = blockIdx.x * BALR_THREADS + threadIdx.x;
  if (wi >= n_words) return;
  uint32_t bits = a.words[wi];
  uint64_t t = *a.base + a.first[wi];
  const uint64_t need = 3 + 4 * a.O + 9 * a.C + 3 * a.P;
  for (; bits; bits &= bits - 1, ++t) {
    if (t < 3 || t >= need) continue;  // the header is the host's; tokens after the points are ignored
    const uint32_t pos = wi * 32 + (uint32_t)__ffs((int)bits) - 1;
    uint32_t end = pos + 1;
    while (end < a.n && !bal_ws(a.buf[end])) ++end;
    const char *s = a.buf + pos;
    const uint32_t len = end - pos;
    const uint64_t r = t - 3;
    if (r < 4 * a.O && (r & 3) < 2) {
      uint64_t v;
      if (!bal_parse_index(s, len, v)) {
        atomicMin(a.err, (unsigned long long)(a.file_off + pos));
      } else if ((r & 3) == 0) {
        if (v >= a.C) atomicMin(a.err + 1, (unsigned long long)(a.file_off + pos));
        else a.cam_of[r / 4] = (uint32_t)v;
      } else {
        if (v >= a.P) atomicMin(a.err + 1, (unsigned long long)(a.file_off + pos));
        else a.idx[r / 4] = (uint32_t)v;
      }
      continue;
    }
    uint64_t x = 0;
    bool near_inf = false;
    const int st = bal_parse_f64(s, len, x, near_inf);
    if (st == BAL_NUM_OK) {
      *bal_num_slot(t, a.C, a.O, a.uv, a.vecs, a.pts) = __longlong_as_double((long long)x);
    } else if (st == BAL_NUM_SLOW) {
      const uint32_t k = atomicAdd(a.n_slow, 1u);  // the buffer holds every token of a chunk of >= 20 bytes each
      a.slow[k] = BalSlow{t, pos, len | (near_inf ? 0x80000000u : 0u)};
    } else {
      atomicMin(a.err, (unsigned long long)(a.file_off + pos));
    }
  }
}

// the chunk's token count onto the running ordinal
__global__ void k_bal_tok_advance(uint64_t *base, const uint32_t *total) { *base += *total; }

// values of the tokens the host converted: (ordinal, bits) pairs
__global__ void __launch_bounds__(BALR_THREADS) k_bal_scatter_slow(const uint64_t *__restrict__ pairs, uint64_t n,
                                                                   uint64_t C, uint64_t O, double *uv, double *vecs,
                                                                   double *pts) {
  const uint64_t i = (uint64_t)blockIdx.x * BALR_THREADS + threadIdx.x;
  if (i < n) *bal_num_slot(pairs[2 * i], C, O, uv, vecs, pts) = __longlong_as_double((long long)pairs[2 * i + 1]);
}

// cnt[c] += observations of camera c; *unordered = 1 when some observation's camera is below its predecessor's
__global__ void __launch_bounds__(BALR_THREADS) k_bal_cam_count(const uint32_t *__restrict__ cam_of, uint64_t O,
                                                                uint32_t *__restrict__ cnt, uint32_t *unordered) {
  const uint64_t o = (uint64_t)blockIdx.x * BALR_THREADS + threadIdx.x;
  if (o >= O) return;
  const uint32_t c = cam_of[o];
  atomicAdd(cnt + c, 1u);
  if (o && c < cam_of[o - 1]) *unordered = 1;
}

// offsets[c] = first[c] (exclusive scan of the counts), offsets[C] = O
__global__ void __launch_bounds__(BALR_THREADS) k_bal_offsets(const uint32_t *__restrict__ first, uint64_t C,
                                                              uint64_t O, uint64_t *__restrict__ offsets) {
  const uint64_t c = (uint64_t)blockIdx.x * BALR_THREADS + threadIdx.x;
  if (c < C) offsets[c] = first[c];
  if (c == C) offsets[C] = O;
}

// keys = camera, vals = file ordinal: the input of the stable regrouping sort
__global__ void __launch_bounds__(BALR_THREADS) k_bal_regroup_keys(const uint32_t *__restrict__ cam_of, uint64_t O,
                                                                   uint64_t *__restrict__ keys,
                                                                   uint32_t *__restrict__ vals) {
  const uint64_t o = (uint64_t)blockIdx.x * BALR_THREADS + threadIdx.x;
  if (o >= O) return;
  keys[o] = cam_of[o];
  vals[o] = (uint32_t)o;
}

__global__ void __launch_bounds__(BALR_THREADS) k_bal_regroup_gather(const uint32_t *__restrict__ order, uint64_t O,
                                                                     const uint32_t *__restrict__ idx_in,
                                                                     const double2 *__restrict__ uv_in,
                                                                     uint32_t *__restrict__ idx_out,
                                                                     double2 *__restrict__ uv_out) {
  const uint64_t o = (uint64_t)blockIdx.x * BALR_THREADS + threadIdx.x;
  if (o >= O) return;
  const uint32_t s = order[o];
  idx_out[o] = idx_in[s];
  uv_out[o] = uv_in[s];
}

struct BalBinArgs {
  const uint64_t *buf;     // the chunk: words [w0, w0 + n)
  uint64_t w0, n;
  const uint64_t *off;     // CSR offsets of the cameras [0, c_known) whose count words have been read
  uint64_t c_known;
  uint64_t C, P, O;
  uint32_t *idx;
  double *uv, *vecs, *pts;
  unsigned long long *err;  // [1]: first point index out of range (file offset)
};

__device__ __forceinline__ uint64_t balr_bswap64(uint64_t x) {
  return ((uint64_t)__byte_perm((uint32_t)x, 0, 0x0123) << 32) | __byte_perm((uint32_t)(x >> 32), 0, 0x0123);
}

__global__ void __launch_bounds__(BALR_THREADS) k_bal_parse_binary(BalBinArgs a) {
  const uint64_t t = (uint64_t)blockIdx.x * BALR_THREADS + threadIdx.x;
  if (t >= a.n) return;
  const uint64_t w = a.w0 + t;
  const uint64_t word = balr_bswap64(a.buf[t]);
  const uint64_t obs_words = a.C + 3 * a.O;
  if (w < 3) return;
  if (w < 3 + obs_words) {
    if (a.c_known == 0) return;
    const uint64_t r = w - 3;
    uint64_t lo = 0, hi = a.c_known;  // the last camera whose block starts at or before r
    while (hi - lo > 1) {
      const uint64_t mid = (lo + hi) >> 1;
      if (mid + 3 * a.off[mid] <= r)
        lo = mid;
      else
        hi = mid;
    }
    const uint64_t d = r - (lo + 3 * a.off[lo]);
    if (d == 0) return;  // the count word: checked by the host
    const uint64_t o = a.off[lo] + (d - 1) / 3;
    const uint32_t f = (uint32_t)((d - 1) % 3);
    if (f == 0) {
      if (word >= a.P) atomicMin(a.err + 1, (unsigned long long)(8 * w));
      else a.idx[o] = (uint32_t)word;
    } else {
      a.uv[2 * o + f - 1] = __longlong_as_double((long long)word);
    }
  } else if (w < 3 + obs_words + 9 * a.C) {
    a.vecs[w - 3 - obs_words] = __longlong_as_double((long long)word);
  } else if (w < 3 + obs_words + 9 * a.C + 3 * a.P) {
    a.pts[w - 3 - obs_words - 9 * a.C] = __longlong_as_double((long long)word);
  }
}

}  // namespace c2b
