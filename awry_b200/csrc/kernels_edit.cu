// kernels_edit.cu -- edit-distance search (<= k substitutions, insertions and deletions) on a nucleotide index that
// holds the unsampled suffix array and the reversed text (awry_*_edit, include/awry_b200.h).  It shares the Hamming
// pipeline up to the candidates (kernels_hamming.cu): the read is cut into k + 1 pieces, piece j = bytes [a_j,
// a_{j+1}), every exact occurrence of piece j at text position p is a candidate, s0 = p - a_j.  Only the
// verification differs: a start whose best alignment keeps piece j intact lies in [s0 - k, s0 + k], so a candidate
// names 2k + 1 starts, and each gets its distance d(s) from one banded DP (DESIGN.md §1d).
#include "kernels_common.cuh"

namespace awry {

// whether search-order symbols [y, y + m) of the read equal reversed-text symbols [x, x + m)
__device__ __forceinline__ bool piece_at(const IndexView& ix, const uint32_t* rq, uint32_t y, int64_t x, uint32_t m) {
  for (uint32_t u = 0; u < m; u += 8) {
    const uint32_t have = m - u;
    const uint32_t mask = have >= 8 ? 0xffffffffu : (1u << (4 * have)) - 1u;
    if ((read8(rq, y + u) ^ rtext8(ix, x + u)) & mask) return false;
  }
  return true;
}

// ---- verification: one thread per candidate.  Search order: the read reversed (R, its packed words) against the
// reversed text, where the original start s is the END of the alignment (rtext index bwt_len - 1 - s) and the
// original end is free (row 0 is all zero, Sellers).  Cell (i, δ) = R[0 .. i) against rtext[.. rb + i + δ),
// rb = bwt_len - s0 - L, for the 4k + 1 diagonals δ = -2k .. 2k: an alignment of cost <= k that ends on a diagonal
// in [-k, k] never leaves them.  Row L, diagonal δ is d(s0 - δ).  Cells hold min(distance, k + 1).
// Start s (d(s) <= k) is reported by its OWNER only: the smallest (j', p') over exact occurrences of piece j' at
// p' with |p' - a_j' - s| <= k -- such an occurrence exists and is a candidate whose range contains s, so every
// start comes out once.  Count: counts[q (k+1) + d] += 1.  Place: the candidate takes popc(acc) consecutive slots
// keys[hit_off[q] + acc[q] ..] (acc[q] += popc) and writes its accepted starts' keys there.  Place-best: the same for
// the accepted starts within the bound of a.best[q].
template <int K, int MODE>
__global__ void __launch_bounds__(256) edit_verify_kernel(IndexView ix, HammingSlice a) {
  constexpr int P = K + 1, W = 4 * K + 1, B = 2 * K;  // pieces, band width, diagonal offset of δ = 0
  constexpr uint64_t ONES = 0x1111111111111111ull >> (4 * (16 - W));  // one bit per band nibble
  const uint64_t stride = gridDim.x * uint64_t(blockDim.x);
  const int64_t n_text = int64_t(ix.bwt_len) - 1;
  for (uint64_t i = blockIdx.x * uint64_t(blockDim.x) + threadIdx.x; i < a.n; i += stride) {
    const uint32_t g = a.map[i];
    AWRY_CHK(g < a.npieces);
    const uint32_t q = g / P, j = g - q * P;
    const uint64_t o0 = a.qoff[q], o1 = a.qoff[q + 1];
    const uint32_t len = checked_len(o0, o1, ByteRange{a.b_lo, a.b_hi});  // 0: refused by the prepass (the call fails)
    const uint2 r = a.sp_cnt[g];
    uint64_t p;
    if (r.y == CNT_AT_TEXT_POS) {  // finished in the text by the search kernel: the piece's one occurrence
      p = r.x;
    } else {
      const uint64_t row = uint64_t(r.x) + (a.c0 + i - a.hoff[g]);
      AWRY_CHK(row < ix.n_full_sa);
      p = __ldg(ix.full_sa + row);
    }
    const int64_t s0 = int64_t(p) - int64_t(uint64_t(j) * len / P);
    uint32_t acc = 0;  // bit k + δ: start s0 - δ accepted
    uint32_t dist[2 * K + 1] = {};
    if (len > uint32_t(K) && s0 + K >= 0 && s0 - K <= n_text - 1) {
      const uint64_t w0 = 4 * (q + (o0 >> 6));
      AWRY_CHK(w0 >= a.qw_lo && w0 - a.qw_lo + (len + 7) / 8 / 2 + 8 < a.qw_n);
      const uint32_t* const rq = reinterpret_cast<const uint32_t*>(a.qwords + w0);
      const int64_t rb = int64_t(ix.bwt_len) - s0 - int64_t(len);
      // band text of row i: nibble w = rtext[rb + i - 1 + w - B]; rows shift it down one nibble and bring in the top
      uint64_t win = 0;
      if (W > 1) {
        const uint64_t t2 = uint64_t(rtext8(ix, rb - B)) | (uint64_t(rtext8(ix, rb - B + 8)) << 32);
        win = (t2 & ((1ull << (4 * (W - 1))) - 1ull)) << 4;
      }
      int64_t tx = rb + B;  // reversed-text index of the next top nibble
      uint32_t tw = 0, qw = 0;
      uint32_t D[W];
#pragma unroll
      for (int w = 0; w < W; w++) D[w] = 0;
      bool alive = true;
      for (uint32_t row = 0; row < len && alive; row++) {
        if ((row & 7) == 0) {
          qw = __ldg(rq + (row >> 3));
          tw = rtext8(ix, tx);
          tx += 8;
          if (row) {  // every 8 rows: stop once the whole band exceeds k (a row's minimum never decreases)
            uint32_t mn = D[0];
#pragma unroll
            for (int w = 1; w < W; w++) mn = min(mn, D[w]);
            alive = mn <= uint32_t(K);
          }
        }
        win = (win >> 4) | (uint64_t(tw & 15u) << (4 * (W - 1)));
        tw >>= 4;
        const uint64_t x = win ^ (uint64_t(qw & 15u) * ONES);
        qw >>= 4;
        const uint64_t mm = (x | (x >> 1) | (x >> 2) | (x >> 3)) & ONES;  // bit 4w: the cell's symbols differ
        uint32_t nd[W];
#pragma unroll
        for (int w = 0; w < W; w++) {
          const uint32_t diag = D[w] + uint32_t((mm >> (4 * w)) & 1u);
          nd[w] = w + 1 < W ? min(diag, D[w + 1] + 1u) : diag;  // (w + 1: one read symbol more, same text)
        }
#pragma unroll
        for (int w = 1; w < W; w++) nd[w] = min(nd[w], nd[w - 1] + 1u);  // one text symbol more, same read
#pragma unroll
        for (int w = 0; w < W; w++) D[w] = min(nd[w], uint32_t(K + 1));
      }
      if (alive) {
#pragma unroll
        for (int t = 0; t <= 2 * K; t++) {  // t = k + δ
          const int64_t s = s0 - (t - K);
          dist[t] = D[t + K];
          if (dist[t] <= uint32_t(K) && s >= 0 && s <= n_text - 1) acc |= 1u << t;
        }
      }
      if (acc) {
        // ownership: occ[j'] bit o + B = piece j' occurs exactly at p' = s0 + a_j' + o, o = -2k .. 2k (j' < j), or at
        // p' = p + o, o = -2k .. -1 (j' = j); start s0 - δ is covered by o in [-δ - k, -δ + k]
        uint32_t smaller = 0;  // bit k + δ: start s0 - δ is covered by a smaller (j', p')
        for (uint32_t jj = 0; jj <= j && smaller != (1u << (2 * K + 1)) - 1u; jj++) {
          const uint32_t aj = uint32_t(uint64_t(jj) * len / P), aj1 = uint32_t(uint64_t(jj + 1) * len / P);
          const uint32_t m = aj1 - aj;
          uint32_t occ = 0;
          const int o_hi = jj < j ? B : -1;
          for (int o = -B; o <= o_hi; o++) {
            const int64_t pp = s0 + int64_t(aj) + o;
            if (pp < 0 || pp + int64_t(m) > n_text) continue;
            if (piece_at(ix, rq, len - aj1, int64_t(ix.bwt_len) - pp - int64_t(m), m)) occ |= 1u << (o + B);
          }
#pragma unroll
          for (int t = 0; t <= 2 * K; t++) {  // δ = t - k: o in [-t, 2k - t], bits [2k - t, 4k - t]
            const uint32_t cover = ((1u << (2 * K + 1)) - 1u) << (2 * K - t);
            if (occ & cover) smaller |= 1u << t;
          }
        }
        acc &= ~smaller;
      }
      if (MODE == VERIFY_PLACE_BEST && acc) {
        const uint8_t b = a.best[q];
#pragma unroll
        for (int t = 0; t <= 2 * K; t++)
          if (!within_map_bound(dist[t], b, K)) acc &= ~(1u << t);
      }
    }
    if (MODE != VERIFY_COUNT) {
      if (acc) {
        uint64_t at = a.hit_off[q] + atomicAdd(reinterpret_cast<unsigned long long*>(a.acc) + q,
                                               (unsigned long long)__popc(acc));
        AWRY_CHK(at + __popc(acc) <= a.hit_off[q + 1]);
#pragma unroll
        for (int t = 0; t <= 2 * K; t++)
          if ((acc >> t) & 1u) a.keys[at++] = (uint64_t(s0 - (t - K)) << 2) | dist[t];
      }
    } else if (acc) {
#pragma unroll
      for (int t = 0; t <= 2 * K; t++)
        if ((acc >> t) & 1u) atomicAdd(reinterpret_cast<unsigned long long*>(a.counts) + (uint64_t(q) * P + dist[t]), 1ull);
    }
  }
}

template <int K>
static void launch_edit_verify_k(const IndexView& ix, const HammingSlice& a, VerifyMode mode, unsigned grid,
                                 cudaStream_t s) {
  if (mode == VERIFY_PLACE)
    edit_verify_kernel<K, VERIFY_PLACE><<<grid, 256, 0, s>>>(ix, a);
  else if (mode == VERIFY_PLACE_BEST)
    edit_verify_kernel<K, VERIFY_PLACE_BEST><<<grid, 256, 0, s>>>(ix, a);
  else
    edit_verify_kernel<K, VERIFY_COUNT><<<grid, 256, 0, s>>>(ix, a);
}

cudaError_t launch_edit_verify(const IndexView& ix, const HammingSlice& a, uint32_t k, VerifyMode mode, int sm_count,
                               cudaStream_t s) {
  if (a.n == 0) return cudaSuccess;
  if (k > 3 || ix.rtext == nullptr || ix.full_sa == nullptr) return cudaErrorInvalidValue;
  const unsigned grid = unsigned(std::max<uint64_t>(1, std::min<uint64_t>(uint64_t(sm_count) * 8, (a.n + 255) / 256)));
  switch (k) {
    case 0: launch_edit_verify_k<0>(ix, a, mode, grid, s); break;
    case 1: launch_edit_verify_k<1>(ix, a, mode, grid, s); break;
    case 2: launch_edit_verify_k<2>(ix, a, mode, grid, s); break;
    default: launch_edit_verify_k<3>(ix, a, mode, grid, s); break;
  }
  COUNT_LAUNCH();
  return cudaGetLastError();
}

// ---- loci (awry_*_edit_loci, DESIGN.md §1g): one thread per hit of hits sorted per query (ascending, distinct starts).
// Hit i of query q = map[i] (range off[q] .. off[q + 1]) is a locus unless (a) a hit within k of it has a smaller
// distance, or (b) its distance is >= 1 and the start just before it is a hit at the same distance.  Positions are
// distinct, so the hits within k of i are among its k neighbours on each side.  Hit i is the key keys[i] = (s << 2) | d.
// Count: counts[q (k+1) + d] += 1 per locus.  Otherwise keep[i] = 1 for a locus, else 0, and keep[n] = 0.
__device__ __forceinline__ void loci_hit(const uint64_t* keys, uint64_t i, uint64_t& s, uint32_t& d) {
  const uint64_t x = keys[i];
  s = x >> 2;
  d = uint32_t(x & 3);
}

__global__ void edit_loci_kernel(const uint64_t* __restrict__ keys, const uint64_t* __restrict__ off,
                                 const uint32_t* __restrict__ map, uint64_t n, uint32_t k, uint64_t* __restrict__ keep,
                                 uint64_t* __restrict__ counts) {
  const uint64_t stride = gridDim.x * uint64_t(blockDim.x);
  for (uint64_t i = blockIdx.x * uint64_t(blockDim.x) + threadIdx.x; i < n; i += stride) {
    const uint32_t q = map[i];
    const uint64_t lo = off[q], hi = off[q + 1];
    AWRY_CHK(lo <= i && i < hi);
    uint64_t s, t;
    uint32_t d, e;
    loci_hit(keys, i, s, d);
    bool locus = true;
    for (uint32_t j = 1; j <= k && i - lo >= j && locus; j++) {
      loci_hit(keys, i - j, t, e);
      AWRY_CHK(t < s);
      if (s - t > k) break;
      locus = e > d || (e == d && (d == 0 || t + 1 != s));
    }
    for (uint32_t j = 1; j <= k && i + j < hi && locus; j++) {
      loci_hit(keys, i + j, t, e);
      AWRY_CHK(t > s);
      if (t - s > k) break;
      locus = e >= d;
    }
    if (counts) {
      if (locus) atomicAdd(reinterpret_cast<unsigned long long*>(counts) + (uint64_t(q) * (k + 1) + d), 1ull);
    } else {
      keep[i] = locus;
      if (i == 0) keep[n] = 0;
    }
  }
}

cudaError_t launch_edit_loci(const uint64_t* d_keys, const uint64_t* d_off, const uint32_t* d_map, uint64_t n, uint32_t k,
                             uint64_t* d_keep, uint64_t* d_counts, cudaStream_t s) {
  if (n == 0) return cudaSuccess;
  const unsigned grid = unsigned(std::min<uint64_t>((n + 255) / 256, 148 * 16));
  edit_loci_kernel<<<grid, 256, 0, s>>>(d_keys, d_off, d_map, n, k, d_keep, d_counts);
  COUNT_LAUNCH();
  return cudaGetLastError();
}

// the CSR of the loci: off[q] = P[off[q]], q = 0 .. nq, P the exclusive scan of the keep flags (in place)
__global__ void edit_loci_offsets_kernel(const uint64_t* __restrict__ P, uint64_t* __restrict__ off, uint64_t nq) {
  const uint64_t stride = gridDim.x * uint64_t(blockDim.x);
  for (uint64_t q = blockIdx.x * uint64_t(blockDim.x) + threadIdx.x; q <= nq; q += stride) off[q] = P[off[q]];
}

cudaError_t launch_edit_loci_offsets(const uint64_t* d_P, uint64_t* d_off, uint64_t nq, cudaStream_t s) {
  const unsigned grid = unsigned(std::min<uint64_t>((nq + 256) / 256, 148 * 16));
  edit_loci_offsets_kernel<<<grid, 256, 0, s>>>(d_P, d_off, nq);
  COUNT_LAUNCH();
  return cudaGetLastError();
}

// hit i is a locus iff P[i + 1] > P[i]; its key goes to slot P[i] of keys_out
__global__ void edit_loci_compact_kernel(const uint64_t* __restrict__ P, uint64_t n, const uint64_t* __restrict__ keys,
                                         uint64_t* __restrict__ keys_out) {
  const uint64_t stride = gridDim.x * uint64_t(blockDim.x);
  for (uint64_t i = blockIdx.x * uint64_t(blockDim.x) + threadIdx.x; i < n; i += stride) {
    const uint64_t o = P[i];
    if (P[i + 1] == o) continue;
    keys_out[o] = keys[i];
  }
}

cudaError_t launch_edit_loci_compact(const uint64_t* d_P, uint64_t n, const uint64_t* d_keys, uint64_t* d_keys_out,
                                     cudaStream_t s) {
  if (n == 0) return cudaSuccess;
  const unsigned grid = unsigned(std::min<uint64_t>((n + 255) / 256, 148 * 16));
  edit_loci_compact_kernel<<<grid, 256, 0, s>>>(d_P, n, d_keys, d_keys_out);
  COUNT_LAUNCH();
  return cudaGetLastError();
}

}  // namespace awry
