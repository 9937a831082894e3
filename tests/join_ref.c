/* tests/join_ref.c — the test suite's sequential restatement of the GPU rule of join_landmarks (src/noise.rs:323-378;
 * city2ba_b200/csrc/c2b_join.cuh states the rule).  Built by tests/test_oracle_join.py with -ffp-contract=off, so every
 * difference, square and sum is the same IEEE operation as the device's round-to-nearest intrinsics.
 *
 * (w0..w3) = Philox4x32-10(key seed, counter (o lo, o hi, 7, 0)) for every observation o; key_o = w0 | w1 << 32,
 * r_o = w2 | w3 << 32.  n = floor(join_percent P) (0 for a negative or NaN join_percent); the min(n, O) smallest pairs
 * (key_o, o) are selected (by sorting).  m = min(11, P); the neighbour list of a point q is the m smallest pairs
 * (d2(p_q, p_k), k) over all points, d2 = (dx dx + dy dy) + dz dz, by brute force; a selected observation takes
 * list[1 + mulhi64(r_o, m - 1)] of the point it sees.  With at least one selection: P < 2 returns 1 (No neighbors?!),
 * a point with a coordinate that is not finite returns 2 with *bad_point = the lowest one; point_idx is unchanged
 * then. */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>

enum { ST_JOIN = 7, JN_K = 11 };

void jn_philox4x32_10(const uint32_t ctr[4], const uint32_t key[2], uint32_t out[4]) {
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

static void draws(uint64_t seed, uint64_t o, uint64_t *key, uint64_t *r) {
  uint32_t ctr[4] = {(uint32_t)o, (uint32_t)(o >> 32), ST_JOIN, 0}, k[2] = {(uint32_t)seed, (uint32_t)(seed >> 32)}, w[4];
  jn_philox4x32_10(ctr, k, w);
  *key = (uint64_t)w[0] | (uint64_t)w[1] << 32;
  *r = (uint64_t)w[2] | (uint64_t)w[3] << 32;
}

uint64_t jn_count(double join_percent, uint64_t P, uint64_t O) {
  double nf = join_percent * (double)P;
  uint64_t n = nf >= 18446744073709551616.0 ? ~0ull : nf >= 1.0 ? (uint64_t)nf : 0;
  return n < O ? n : O;
}

static double dist2(const double *p, const double *q) {
  double dx = p[0] - q[0], dy = p[1] - q[1], dz = p[2] - q[2];
  return (dx * dx + dy * dy) + dz * dz;
}

/* the m = min(11, P) smallest (d2, k) of point q, ascending: indices into nb[], distances into d2 (may be NULL) */
uint64_t jn_neighbours(const double *pts, uint64_t P, uint64_t q, uint32_t *nb, double *d2) {
  double bd[JN_K];
  uint32_t bk[JN_K];
  uint64_t m = P < JN_K ? P : JN_K, n = 0;
  for (uint64_t k = 0; k < P; ++k) {
    double d = dist2(pts + 3 * q, pts + 3 * k);
    if (n == m && !(d < bd[m - 1])) continue;  /* equal d: the larger index k loses */
    uint64_t t = n < m ? n++ : m - 1;
    while (t > 0 && d < bd[t - 1]) {
      bd[t] = bd[t - 1];
      bk[t] = bk[t - 1];
      --t;
    }
    bd[t] = d;
    bk[t] = (uint32_t)k;
  }
  for (uint64_t j = 0; j < m; ++j) {
    nb[j] = bk[j];
    if (d2) d2[j] = bd[j];
  }
  return m;
}

typedef struct {
  uint64_t key, o;
} pair_t;

static int cmp_pair(const void *a, const void *b) {
  const pair_t *x = a, *y = b;
  if (x->key != y->key) return x->key < y->key ? -1 : 1;
  return x->o < y->o ? -1 : x->o > y->o;
}

/* selected (O entries or NULL): 1 for the selected observations, else 0 */
int jn_join_landmarks(const double *pts, uint64_t P, uint32_t *point_idx, uint64_t O, double join_percent,
                      uint64_t seed, uint64_t *n_selected, uint64_t *n_changed, uint8_t *selected,
                      uint64_t *bad_point) {
  uint64_t k = jn_count(join_percent, P, O), nc = 0;
  if (selected)
    for (uint64_t o = 0; o < O; ++o) selected[o] = 0;
  *n_selected = *n_changed = 0;
  if (k == 0) return 0;
  if (P < 2) return 1;
  for (uint64_t i = 0; i < P; ++i)
    if (!isfinite(pts[3 * i]) || !isfinite(pts[3 * i + 1]) || !isfinite(pts[3 * i + 2])) {
      *bad_point = i;
      return 2;
    }
  pair_t *v = malloc(O * sizeof *v);
  uint32_t *pick = malloc(k * sizeof *pick);
  for (uint64_t o = 0; o < O; ++o) {
    uint64_t r;
    v[o].o = o;
    draws(seed, o, &v[o].key, &r);
  }
  qsort(v, O, sizeof *v, cmp_pair);
  for (uint64_t s = 0; s < k; ++s) {
    uint64_t key, r, o = v[s].o;
    uint32_t nb[JN_K];
    draws(seed, o, &key, &r);
    uint64_t m = jn_neighbours(pts, P, point_idx[o], nb, NULL);
    pick[s] = nb[1 + mulhi64(r, m - 1)];
  }
  for (uint64_t s = 0; s < k; ++s) {
    uint64_t o = v[s].o;
    nc += pick[s] != point_idx[o];
    point_idx[o] = pick[s];
    if (selected) selected[o] = 1;
  }
  *n_selected = k;
  *n_changed = nc;
  free(v);
  free(pick);
  return 0;
}
