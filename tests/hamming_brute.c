/* hamming_brute.c -- test reference for the Hamming search entry points (awry_*_hamming): a plain scan over every
 * window text[s .. s+L), 0 <= s <= n - L, of the text the index holds, query and text bytes mapped to symbols through
 * the same table as exact search (`lut`, filled from the oracle's awo_ascii_to_index), stopping a window once its
 * distance exceeds k.  tests/test_gpu_hamming.py compiles it into a temporary directory.
 *
 * counts[q * (k+1) + d] = windows of query q at distance d; hit_off (nq + 1) = CSR offsets of the windows at
 * distance <= k; with hit_pos != NULL their start positions (ascending) and distances are written too. */
#include <stdint.h>
#include <string.h>

int64_t hamming_brute(const uint8_t *lut, const uint8_t *text, uint64_t n, const uint8_t *qbytes, const uint64_t *qoff,
                      uint64_t nq, uint32_t k, uint64_t *counts, uint64_t *hit_off, uint64_t *hit_pos, uint8_t *hit_d) {
  memset(counts, 0, nq * (k + 1) * sizeof(uint64_t));
  uint64_t *per = hit_off + 1;
#pragma omp parallel for schedule(dynamic, 4)
  for (int64_t qi = 0; qi < (int64_t)nq; qi++) {
    const uint64_t q = (uint64_t)qi, len = qoff[q + 1] - qoff[q];
    uint8_t sym[8192];
    if (len > sizeof sym) continue;
    for (uint64_t i = 0; i < len; i++) sym[i] = lut[qbytes[qoff[q] + i]];
    uint64_t found = 0, at = hit_pos ? hit_off[q] : 0;
    for (uint64_t s = 0; len <= n && s <= n - len; s++) {
      uint32_t d = 0;
      for (uint64_t i = 0; i < len && d <= k; i++) d += lut[text[s + i]] != sym[i];
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
  if (!hit_pos) {
    hit_off[0] = 0;
    for (uint64_t q = 0; q < nq; q++) hit_off[q + 1] += hit_off[q];
  }
  return (int64_t)hit_off[nq];
}
