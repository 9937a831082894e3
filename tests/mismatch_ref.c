/* tests/mismatch_ref.c — the test suite's sequential restatement of the GPU rule of add_incorrect_correspondences
 * (src/noise.rs:180-226; city2ba_b200/csrc/c2b_mismatch.cuh states the rule).  Built by tests/test_oracle_mismatch.py
 * with -ffp-contract=off, so every distance, quotient and product is the same IEEE operation as the device's
 * round-to-nearest intrinsics.
 *
 * Per camera of more than one observation, per observation i in order: selected iff
 * u = ((w0 | w1 << 32) >> 11) 2^-53 <= chance, (w0..w3) = Philox4x32-10(key seed, counter (i lo, i hi, 6, 0));
 * d_j = sqrt(dx dx + dy dy); a non-finite one is NegativeWeight, maxd == 0 AllWeightsZero;
 * q_j = floor((maxd - d_j) / maxd 2^32); j = the first index whose prefix sum of q exceeds mulhi64(w2 | w3 << 32, sum q).
 * The swaps are applied after every pick is known, so point_idx is unchanged on an error.  Returns 0, or 1
 * (AllWeightsZero) / 2 (NegativeWeight) with *err_obs = the first failing observation.  picks (O entries or NULL):
 * the partner of each selected observation, -1 for the others. */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>

enum { ST_MISMATCH = 6 };

void mm_philox4x32_10(const uint32_t ctr[4], const uint32_t key[2], uint32_t out[4]) {
  uint32_t c0 = ctr[0], c1 = ctr[1], c2 = ctr[2], c3 = ctr[3], k0 = key[0], k1 = key[1];
  for (int r = 0; r < 10; ++r) {
    uint64_t p0 = (uint64_t)0xD2511F53u * c0, p1 = (uint64_t)0xCD9E8D57u * c2;
    uint32_t n0 = (uint32_t)(p1 >> 32) ^ c1 ^ k0, n2 = (uint32_t)(p0 >> 32) ^ c3 ^ k1;
    c0 = n0;
    c1 = (uint32_t)p1;
    c2 = n2;
    c3 = (uint32_t)p0;
    k0 += 0x9E3779B9u;
    k1 += 0xBB67AE85u;
  }
  out[0] = c0;
  out[1] = c1;
  out[2] = c2;
  out[3] = c3;
}

static uint64_t mulhi64(uint64_t a, uint64_t b) { return (uint64_t)(((unsigned __int128)a * b) >> 64); }

static uint64_t weight(const double *p, const double *q, double maxd) {
  double dx = p[0] - q[0], dy = p[1] - q[1];
  double d = sqrt(dx * dx + dy * dy);
  return (uint64_t)((maxd - d) / maxd * 4294967296.0);
}

int mm_add_incorrect_correspondences(const uint64_t *offsets, uint64_t C, uint32_t *point_idx, const double *uv,
                                     double chance, uint64_t seed, uint64_t *n_selected, uint64_t *n_swapped,
                                     int64_t *picks, uint64_t *err_obs) {
  uint64_t O = offsets[C], ns = 0, nw = 0;
  uint64_t *swap_i = malloc((O ? O : 1) * sizeof *swap_i), *swap_j = malloc((O ? O : 1) * sizeof *swap_j);
  int rc = 0;
  if (picks)
    for (uint64_t o = 0; o < O; ++o) picks[o] = -1;
  for (uint64_t c = 0; c < C && !rc; ++c) {
    uint64_t a = offsets[c], b = offsets[c + 1];
    if (b - a <= 1) continue;
    for (uint64_t i = a; i < b; ++i) {
      uint32_t ctr[4] = {(uint32_t)i, (uint32_t)(i >> 32), ST_MISMATCH, 0}, key[2] = {(uint32_t)seed,
                                                                                      (uint32_t)(seed >> 32)}, w[4];
      mm_philox4x32_10(ctr, key, w);
      double u = (double)((((uint64_t)w[1] << 32) | w[0]) >> 11) * 0x1p-53;
      if (!(u <= chance)) continue;
      double m2 = 0.0;
      int finite = 1;
      for (uint64_t j = a; j < b; ++j) {
        double dx = uv[2 * i] - uv[2 * j], dy = uv[2 * i + 1] - uv[2 * j + 1];
        double s2 = dx * dx + dy * dy;
        if (!isfinite(s2))
          finite = 0;
        else if (s2 > m2)
          m2 = s2;
      }
      if (!finite || m2 == 0.0) {
        rc = finite ? 1 : 2;
        *err_obs = i;
        break;
      }
      double maxd = sqrt(m2);
      uint64_t T = 0, acc = 0, j;
      for (uint64_t k = a; k < b; ++k) T += weight(uv + 2 * i, uv + 2 * k, maxd);
      uint64_t t = mulhi64((uint64_t)w[2] | (uint64_t)w[3] << 32, T);
      for (j = a; j < b; ++j) {
        acc += weight(uv + 2 * i, uv + 2 * j, maxd);
        if (acc > t) break;
      }
      if (picks) picks[i] = (int64_t)j;
      swap_i[ns] = i;
      swap_j[ns] = j;
      ++ns;
      nw += j != i;
    }
  }
  if (!rc) {
    for (uint64_t k = 0; k < ns; ++k) {
      uint32_t t = point_idx[swap_i[k]];
      point_idx[swap_i[k]] = point_idx[swap_j[k]];
      point_idx[swap_j[k]] = t;
    }
    *n_selected = ns;
    *n_swapped = nw;
  }
  free(swap_i);
  free(swap_j);
  return rc;
}
