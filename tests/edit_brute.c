/* edit_brute.c -- test reference for the edit-distance search entry points (awry_*_edit): for every query and every
 * start s, 0 <= s < n, of the text the index holds, a DP of the query against text[s .. min(n, s+L+k)) with the start
 * fixed at s and the end free gives d(s) = min over l of ed(query, text[s .. s+l)).  Query and text bytes are mapped
 * to symbols through the same table as exact search (`lut`, filled from the oracle's awo_ascii_to_index).  Only the
 * cells with |i - j| <= k are kept (the others exceed k: a cell is at least |i - j|), and a start is dropped once a
 * whole row exceeds k.  No pieces, no index.  tests/test_gpu_edit.py compiles it into a temporary directory.
 *
 * counts[q * (k+1) + d] = starts of query q at distance d; hit_off (nq + 1) = CSR offsets of the starts at distance
 * <= k; with hit_pos != NULL their positions (ascending) and distances are written too. */
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#define EB_MAXK 3
#define EB_W (2 * EB_MAXK + 1)

/* d(s) of query sym[0 .. len) at text start s, or k + 1 when it exceeds k */
static uint32_t edit_at(const uint8_t *tsym, uint64_t n, uint64_t s, const uint8_t *sym, uint64_t len, uint32_t k) {
  const int64_t big = k + 1;
  const uint64_t m = (n - s < len + k) ? n - s : len + k; /* text symbols the alignment may use */
  /* row i, band slot b = j - i + k (j = text symbols consumed, 0 .. m) */
  int64_t prev[EB_W], cur[EB_W];
  for (int b = 0; b < EB_W; b++) {
    const int64_t j = b - (int64_t)k;
    prev[b] = (b <= 2 * (int)k && j >= 0 && (uint64_t)j <= m) ? (j < big ? j : big) : big; /* row 0: D[0][j] = j */
  }
  for (uint64_t i = 1; i <= len; i++) {
    int64_t row_min = big;
    for (int b = 0; b <= 2 * (int)k; b++) {
      const int64_t j = (int64_t)i + b - (int64_t)k;
      int64_t v = big;
      if (j >= 0 && (uint64_t)j <= m) {
        if (j == 0) {
          v = (int64_t)i;                                                     /* D[i][0] = i */
        } else {
          v = prev[b] + (tsym[s + (uint64_t)j - 1] != sym[i - 1]);            /* diagonal */
          if (b + 1 <= 2 * (int)k && prev[b + 1] + 1 < v) v = prev[b + 1] + 1; /* query symbol against nothing */
          if (b > 0 && cur[b - 1] + 1 < v) v = cur[b - 1] + 1;                 /* text symbol against nothing */
        }
        if (v > big) v = big;
      }
      cur[b] = v;
      if (v < row_min) row_min = v;
    }
    if (row_min > (int64_t)k) return k + 1;
    memcpy(prev, cur, sizeof cur);
  }
  int64_t best = big;
  for (int b = 0; b <= 2 * (int)k; b++) {
    const int64_t j = (int64_t)len + b - (int64_t)k;
    if (j >= 0 && (uint64_t)j <= m && prev[b] < best) best = prev[b];
  }
  return (uint32_t)best;
}

int64_t edit_brute(const uint8_t *lut, const uint8_t *text, uint64_t n, const uint8_t *qbytes, const uint64_t *qoff,
                   uint64_t nq, uint32_t k, uint64_t *counts, uint64_t *hit_off, uint64_t *hit_pos, uint8_t *hit_d) {
  if (k > EB_MAXK) return -1;
  memset(counts, 0, nq * (k + 1) * sizeof(uint64_t));
  uint64_t *per = hit_off + 1;
  uint8_t *tsym = (uint8_t *)malloc(n ? n : 1);
  for (uint64_t i = 0; i < n; i++) tsym[i] = lut[text[i]];
#pragma omp parallel for schedule(dynamic, 1)
  for (int64_t qi = 0; qi < (int64_t)nq; qi++) {
    const uint64_t q = (uint64_t)qi, len = qoff[q + 1] - qoff[q];
    uint8_t sym[8192];
    if (len > sizeof sym) continue;
    for (uint64_t i = 0; i < len; i++) sym[i] = lut[qbytes[qoff[q] + i]];
    uint64_t found = 0, at = hit_pos ? hit_off[q] : 0;
    for (uint64_t s = 0; s < n; s++) {
      const uint32_t d = edit_at(tsym, n, s, sym, len, k);
      if (d > k) continue;
      counts[q * (k + 1) + d]++;
      if (hit_pos) {
        hit_pos[at] = s;
        hit_d[at] = (uint8_t)d;
        at++;
      }
      found++;
    }
    if (!hit_pos) per[q] = found;
  }
  free(tsym);
  if (!hit_pos) {
    hit_off[0] = 0;
    for (uint64_t q = 0; q < nq; q++) hit_off[q + 1] += hit_off[q];
  }
  return (int64_t)hit_off[nq];
}

/* d(s) for one query and one start, for the CPU test of this reference against a plain DP */
uint32_t edit_brute_one(const uint8_t *lut, const uint8_t *text, uint64_t n, uint64_t s, const uint8_t *q, uint64_t len,
                        uint32_t k) {
  uint8_t *tsym = (uint8_t *)malloc(n ? n : 1), sym[8192];
  for (uint64_t i = 0; i < n; i++) tsym[i] = lut[text[i]];
  for (uint64_t i = 0; i < len && i < sizeof sym; i++) sym[i] = lut[q[i]];
  const uint32_t d = edit_at(tsym, n, s, sym, len, k);
  free(tsym);
  return d;
}
