/* align_brute.c -- test reference for the alignment entry points (awry_align_*): for every hit, the awry_alignment the
 * header promises, computed without the library's search.  Query and text bytes are mapped to symbols through the same
 * table as exact search (`lut`, filled from the oracle's awo_ascii_to_index: $0 A1 C2 G3 N4 T5); both strands: the
 * query of v = 2q + 1 is rc(q), complemented symbol by symbol and reversed.
 *
 * Hamming: the window text[s .. s+L) compared symbol by symbol.
 * Edit distance: the suffix-distance table F[i][j] = the least cost of aligning Q[i .. L) against text[s+j .. s+j+l) for
 * any l (the end is free), over the window text[s .. s+m), m = min(n - s, L + k), then a walk from (0, 0) that takes, at
 * each cell, the first of =, X, I, D whose successor keeps the cost: F[i][j] = cost(op) + F[next].  That walk gives
 * the lexicographically smallest optimal op string; it does not assume that a match is always optimal.  Only the cells
 * with |i - j| <= k + 1 are filled (the others count as more than k): the walk visits cells with |i - j| <= c <= k (c =
 * its cost so far) and an optimal path from such a cell never leaves |i - j| <= k, so every value the walk compares is
 * exact.  An alignment of cost <= k uses at most L + k text symbols, so the window loses none.
 *
 * out: 44 bytes per hit, the layout of awry_alignment, every unused byte 0.  A query that is empty, holds '$' or '#' or
 * has L <= k, a hit with seq_idx >= n_seqs or s >= n, and a hit over k get "no alignment": distance k + 1, no ops. */
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#define AB_MAXK 3

static const char AB_LETTER[6] = {'$', 'A', 'C', 'G', 'N', 'T'};
static const uint8_t AB_COMP[6] = {0, 5, 3, 2, 4, 1};

static void put32(uint8_t *p, uint32_t v) {
  for (int b = 0; b < 4; b++) p[b] = (uint8_t)(v >> (8 * b));
}

/* one op (0-based t) of the record */
static void put_op(uint8_t *out, int t, uint32_t qpos, uint32_t tpos, char op, uint8_t qs, uint8_t ts) {
  uint8_t *o = out + 8 + 12 * t;
  put32(o, qpos);
  put32(o + 4, tpos);
  o[8] = (uint8_t)op;
  o[9] = op == 'D' ? 0 : (uint8_t)AB_LETTER[qs];
  o[10] = op == 'I' ? 0 : (uint8_t)AB_LETTER[ts];
}

/* the record of query sym[0 .. len) at text start s (tsym = the whole text, n symbols); returns the distance */
static uint32_t align_one(const uint8_t *tsym, uint64_t n, uint64_t s, const uint8_t *sym, uint64_t len, uint32_t metric,
                          uint32_t k, uint8_t *out) {
  memset(out, 0, 44);
  out[4] = (uint8_t)(k + 1);
  if (s >= n || len <= k) return k + 1;
  if (metric == 0) {
    if (s + len > n) return k + 1;
    uint32_t d = 0;
    for (uint64_t i = 0; i < len; i++) {
      if (sym[i] == tsym[s + i]) continue;
      if (d == k) { /* over k: drop the ops written so far */
        memset(out, 0, 44);
        out[4] = (uint8_t)(k + 1);
        return k + 1;
      }
      put_op(out, (int)d, (uint32_t)i, (uint32_t)i, 'X', sym[i], tsym[s + i]);
      d++;
    }
    put32(out, (uint32_t)len);
    out[4] = out[5] = (uint8_t)d;
    return d;
  }
  const uint64_t m = (n - s < len + k) ? n - s : len + k;
  const int64_t W = 2 * (int64_t)k + 3, big = 1 << 20; /* band slot b = j - i + k + 1 */
  int32_t *F = (int32_t *)malloc((len + 1) * W * sizeof(int32_t));
#define AB_F(i, j) (((int64_t)(j) - (int64_t)(i) < -(int64_t)k - 1 || (int64_t)(j) - (int64_t)(i) > (int64_t)k + 1 || (uint64_t)(j) > m) \
                        ? big : F[(uint64_t)(i) * W + (uint64_t)((int64_t)(j) - (int64_t)(i) + (int64_t)k + 1)])
  for (int64_t i = (int64_t)len; i >= 0; i--) {
    for (int64_t b = W - 1; b >= 0; b--) {
      const int64_t j = i + b - (int64_t)k - 1;
      int32_t v = big;
      if (j >= 0 && (uint64_t)j <= m) {
        if ((uint64_t)i == len) {
          v = 0; /* the end is free */
        } else {
          if ((uint64_t)j < m) {
            const int32_t dg = AB_F(i + 1, j + 1) + (sym[i] != tsym[s + (uint64_t)j]);
            const int32_t dl = AB_F(i, j + 1) + 1;
            v = dg < v ? dg : v;
            v = dl < v ? dl : v;
          }
          const int32_t in = AB_F(i + 1, j) + 1;
          v = in < v ? in : v;
        }
      }
      F[i * W + b] = v;
    }
  }
  const int32_t d = AB_F(0, 0);
  if (d > (int32_t)k) {
    free(F);
    return k + 1;
  }
  uint64_t i = 0, j = 0;
  int t = 0;
  while (i < len) {
    const int32_t f = AB_F(i, j);
    if (j < m && sym[i] == tsym[s + j] && AB_F(i + 1, j + 1) == f) { /* = */
      i++, j++;
    } else if (j < m && sym[i] != tsym[s + j] && AB_F(i + 1, j + 1) + 1 == f) {
      put_op(out, t++, (uint32_t)i, (uint32_t)j, 'X', sym[i], tsym[s + j]);
      i++, j++;
    } else if (AB_F(i + 1, j) + 1 == f) {
      put_op(out, t++, (uint32_t)i, (uint32_t)j, 'I', sym[i], 0);
      i++;
    } else {
      put_op(out, t++, (uint32_t)i, (uint32_t)j, 'D', 0, tsym[s + j]);
      j++;
    }
  }
#undef AB_F
  free(F);
  put32(out, (uint32_t)j);
  out[4] = out[5] = (uint8_t)d;
  return (uint32_t)d;
}

/* every hit of a locate call: hit_off (nv + 1, nv = nq << strands), hits (seq_idx, local_pos) pairs -> out */
int64_t align_brute(const uint8_t *lut, const uint8_t *text, uint64_t n, const uint64_t *seq_starts, uint64_t n_seqs,
                    const uint8_t *qbytes, const uint64_t *qoff, uint64_t nq, uint32_t metric, uint32_t strands, uint32_t k,
                    const uint64_t *hit_off, const uint64_t *hits, uint8_t *out) {
  if (k > AB_MAXK || strands > 1 || metric > 1) return -1;
  uint8_t *tsym = (uint8_t *)malloc(n ? n : 1);
  for (uint64_t i = 0; i < n; i++) tsym[i] = lut[text[i]];
  const int64_t nv = (int64_t)(nq << strands);
#pragma omp parallel for schedule(dynamic, 1)
  for (int64_t v = 0; v < nv; v++) {
    const uint64_t q = (uint64_t)v >> strands, len = qoff[q + 1] - qoff[q];
    uint8_t *sym = (uint8_t *)malloc(len ? len : 1);
    int refused = len == 0;
    for (uint64_t i = 0; i < len; i++) {
      const uint8_t c = qbytes[qoff[q] + i];
      refused |= c == '$' || c == '#';
      sym[i] = lut[c];
    }
    if (strands && (v & 1))
      for (uint64_t i = 0; i < len; i++) sym[i] = AB_COMP[lut[qbytes[qoff[q] + len - 1 - i]]];
    for (uint64_t h = hit_off[v]; h < hit_off[v + 1]; h++) {
      const uint64_t seq = hits[2 * h], local = hits[2 * h + 1];
      const uint64_t s = (!refused && seq < n_seqs) ? seq_starts[seq] + local : n;
      align_one(tsym, n, s, sym, refused ? 0 : len, metric, k, out + 44 * h);
    }
    free(sym);
  }
  free(tsym);
  return (int64_t)hit_off[nv];
}

/* one query against one start, for the CPU test of this reference against exhaustive enumeration; returns the distance */
uint32_t align_brute_one(const uint8_t *lut, const uint8_t *text, uint64_t n, uint64_t s, const uint8_t *q, uint64_t len,
                         uint32_t metric, uint32_t k, uint8_t *out) {
  uint8_t *tsym = (uint8_t *)malloc(n ? n : 1), *sym = (uint8_t *)malloc(len ? len : 1);
  for (uint64_t i = 0; i < n; i++) tsym[i] = lut[text[i]];
  for (uint64_t i = 0; i < len; i++) sym[i] = lut[q[i]];
  const uint32_t d = align_one(tsym, n, s, sym, len, metric, k, out);
  free(tsym);
  free(sym);
  return d;
}
