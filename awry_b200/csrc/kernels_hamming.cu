// kernels_hamming.cu -- Hamming search (<= k substitutions, no indels) on a nucleotide index that holds the
// unsampled suffix array and the reversed text (awry_*_hamming, include/awry_b200.h).  Pigeonhole scheme: a read
// of length L is cut into k + 1 pieces, piece j = bytes [a_j, a_{j+1}) with a_j = floor(j L / (k + 1)); every
// window within distance k matches one piece exactly.  The pieces are searched with the exact kernels (kernels.cu)
// and every exact occurrence of piece j at text position p names the candidate window s = p - a_j, which the
// kernels here verify against IndexView::rtext.  A window is reported by the smallest j whose piece it matches
// exactly, so each window comes out once without a global deduplication.
#include <cub/device/device_scan.cuh>
#include <cub/device/device_segmented_sort.cuh>
#include <thrust/iterator/counting_iterator.h>
#include <thrust/iterator/transform_iterator.h>

#include "kernels_common.cuh"

namespace awry {

// piece offsets of every query: poff[(k+1) q + j] = qoff[q] + a_j, poff[(k+1) nq] = qoff[nq].  A query with L <= k
// has empty pieces (and every window would match): it is latched like an empty query, as the caller's query
// q >> shift (shift 1: the queries are the virtual ones of both strands, kernels.hpp).  Offsets outside [b_lo,
// b_hi] are left to the read's own prepass (launch_pack), which latches them with the query's index.
__global__ void __launch_bounds__(256)
    hamming_pieces_kernel(const uint64_t* __restrict__ qoff, uint64_t nq, uint32_t k, uint64_t b_lo, uint64_t b_hi,
                          uint32_t shift, uint64_t* __restrict__ poff, unsigned long long* first_bad) {
  const uint64_t stride = gridDim.x * uint64_t(blockDim.x);
  for (uint64_t q = blockIdx.x * uint64_t(blockDim.x) + threadIdx.x; q < nq; q += stride) {
    const uint64_t o0 = qoff[q], o1 = qoff[q + 1];
    const bool valid = !(o0 < b_lo || o1 > b_hi || o1 < o0 || o1 - o0 >= (1ull << 32));
    const uint64_t len = valid ? o1 - o0 : 0;
    if (valid && len <= k) atomicMin(first_bad, bad_query_code(q >> shift, BAD_QUERY));
    for (uint32_t j = 0; j <= k; j++) poff[(k + 1) * q + j] = o0 + j * len / (k + 1);
    if (q + 1 == nq) poff[(k + 1) * nq] = o1;
  }
}

cudaError_t launch_hamming_pieces(const uint64_t* d_qoff, uint64_t nq, uint32_t k, uint64_t b_lo, uint64_t b_hi,
                                  uint32_t shift, uint64_t* d_poff, unsigned long long* d_first_bad, cudaStream_t s) {
  if (nq == 0) return cudaSuccess;
  const unsigned grid = unsigned(std::min<uint64_t>((nq + 255) / 256, 148 * 16));
  hamming_pieces_kernel<<<grid, 256, 0, s>>>(d_qoff, nq, k, b_lo, b_hi, shift, d_poff, d_first_bad);
  COUNT_LAUNCH();
  return cudaGetLastError();
}

// the words of every piece from those of its query, 4 lanes per query (as strand_words_kernel).  Piece j = bytes
// [a_j, a_{j+1}) is the search-order nibble range [L - a_{j+1}, L - a_j) of the query's stream, so its word w is
// one funnel shift of the query's words wi, wi + 1 (wi = (L - a_{j+1} + 16 w) / 16).  What pack_kernel writes for the
// piece's bytes comes out: the same codes (pack_kernel maps every byte the same way wherever the query is cut), the
// nibbles past the piece's last symbol zero, and no word past its last.  A query the prepass refused (or an empty
// one) has no words; its pieces are empty or refused themselves (hamming_pieces_kernel), so none is written.
__global__ void __launch_bounds__(256)
    hamming_piece_words_kernel(const uint64_t* __restrict__ qwords, const uint64_t* __restrict__ qoff, uint64_t nq,
                               ByteRange br, uint32_t k, uint64_t* __restrict__ pwords) {
  const uint32_t sub = threadIdx.x & 3, P = k + 1;
  const uint64_t ngroups = (gridDim.x * uint64_t(blockDim.x)) >> 2;
  for (uint64_t q = (blockIdx.x * uint64_t(blockDim.x) + threadIdx.x) >> 2; q < nq; q += ngroups) {
    const uint64_t o0 = qoff[q];
    const uint32_t len = checked_len(o0, qoff[q + 1], br);
    if (len == 0) continue;
    const uint64_t* const src = qwords + 4 * (q + (o0 >> 6));
    uint32_t a0 = 0;  // a_j
    for (uint32_t j = 0; j < P; j++) {
      const uint32_t a1 = uint32_t(uint64_t(j + 1) * len / P), m = a1 - a0, s0 = len - a1;
      uint64_t* const dst = pwords + 4 * (uint64_t(P) * q + j + ((o0 + a0) >> 6));
      for (uint32_t w = sub; 16 * w < m; w += 4) {
        const uint32_t si = s0 + 16 * w, wi = si >> 4, sh = 4 * (si & 15);
        const uint64_t lo = src[wi], hi = sh && 16 * (wi + 1) < len ? src[wi + 1] : 0ull;
        uint64_t x = sh ? (lo >> sh) | (hi << (64 - sh)) : lo;
        const uint32_t have = m - 16 * w;  // symbols of this word (the rest stay 0)
        if (have < 16) x &= (1ull << (4 * have)) - 1;
        dst[w] = x;
      }
      a0 = a1;
    }
  }
}

cudaError_t launch_hamming_piece_words(const uint64_t* d_qwords, const uint64_t* d_qoff, uint64_t nq, uint64_t b_lo,
                                       uint64_t b_hi, uint32_t k, uint64_t* d_pwords, cudaStream_t s) {
  if (nq == 0) return cudaSuccess;
  const unsigned grid = unsigned(std::min<uint64_t>((nq * 4 + 255) / 256, 148 * 64));
  hamming_piece_words_kernel<<<grid, 256, 0, s>>>(d_qwords, d_qoff, nq, ByteRange{b_lo, b_hi}, k, d_pwords);
  COUNT_LAUNCH();
  return cudaGetLastError();
}

// qcand[i] = hoff[(k+1) i], i = 0 .. nq: the candidates of query i are [qcand[i], qcand[i+1])
__global__ void hamming_query_bounds_kernel(const uint64_t* __restrict__ hoff, uint32_t k, uint64_t nq,
                                            uint64_t* __restrict__ qcand) {
  const uint64_t stride = gridDim.x * uint64_t(blockDim.x);
  for (uint64_t i = blockIdx.x * uint64_t(blockDim.x) + threadIdx.x; i <= nq; i += stride) qcand[i] = hoff[(k + 1) * i];
}

cudaError_t launch_hamming_query_bounds(const uint64_t* d_hoff, uint32_t k, uint64_t nq, uint64_t* d_qcand, cudaStream_t s) {
  const unsigned grid = unsigned(std::min<uint64_t>((nq + 256) / 256, 148 * 16));
  hamming_query_bounds_kernel<<<grid, 256, 0, s>>>(d_hoff, k, nq, d_qcand);
  COUNT_LAUNCH();
  return cudaGetLastError();
}

// candidate -> piece map of the slice [c0, c0 + n): piece g is written where its candidates start (and at 0 when
// they began before the slice), then an inclusive max-scan carries it over the rest.  One thread per piece and one
// scan, so a piece with 10^4 occurrences costs what 10^4 singletons cost.
__global__ void hamming_map_scatter_kernel(const uint64_t* __restrict__ hoff, uint64_t npieces, uint64_t c0, uint64_t n,
                                           uint32_t* __restrict__ map) {
  const uint64_t stride = gridDim.x * uint64_t(blockDim.x);
  for (uint64_t g = blockIdx.x * uint64_t(blockDim.x) + threadIdx.x; g < npieces; g += stride) {
    const uint64_t st = hoff[g], en = hoff[g + 1];
    if (en <= st) continue;
    if (st >= c0 && st < c0 + n)
      map[st - c0] = uint32_t(g);
    else if (st < c0 && en > c0)
      map[0] = uint32_t(g);
  }
}

struct MaxU32 {
  __host__ __device__ uint32_t operator()(uint32_t a, uint32_t b) const { return a > b ? a : b; }
};

cudaError_t launch_hamming_map(const uint64_t* d_hoff, uint64_t npieces, uint64_t c0, uint64_t n, uint32_t* d_map,
                               void* d_temp, size_t& temp_bytes, cudaStream_t s) {
  if (d_temp == nullptr) return cub::DeviceScan::InclusiveScan(nullptr, temp_bytes, d_map, d_map, MaxU32{}, (long long)n, s);
  cudaError_t e = cudaMemsetAsync(d_map, 0, n * 4, s);
  if (e != cudaSuccess) return e;
  const unsigned grid = unsigned(std::max<uint64_t>(1, std::min<uint64_t>((npieces + 255) / 256, 148 * 16)));
  hamming_map_scatter_kernel<<<grid, 256, 0, s>>>(d_hoff, npieces, c0, n, d_map);
  COUNT_LAUNCH();
  if ((e = cudaGetLastError()) != cudaSuccess) return e;
  e = cub::DeviceScan::InclusiveScan(d_temp, temp_bytes, d_map, d_map, MaxU32{}, (long long)n, s);
  COUNT_LAUNCH();
  return e;
}

// ---- verification: 4 lanes per candidate, 8 candidates per warp.  Lane `sub` of a group reads 32-byte sector
// s_first + sub + 4 r of the reversed text in round r (one LDG.256 each, 256 symbols per round), counts the
// mismatches of each piece against the packed read, and the group adds them up; it stops once the total exceeds k.
// The window of search-order symbol j is rtext[rb0 + j] with rb0 = bwt_len - s - L (rtext[i] = text[bwt_len - 1 - i],
// layout.cuh): read and text are two forward streams.  A candidate is accepted iff its distance d <= k and its piece
// j is the smallest one without a mismatch.  Count: counts[q (k+1) + d] += 1.  Locate: keys[i] = (s << 2) | d, or ~0
// (rejected), and acc[q - q0] += 1.  Place: (s << 2) | d goes to keys[hit_off[q] + acc[q]++] (one slot of the range
// the count pass gave q; the order within it is settled by the sort that follows).
template <int K, int MODE>
__global__ void __launch_bounds__(256) hamming_verify_kernel(IndexView ix, HammingSlice a) {
  constexpr uint32_t FULL = 0xffffffffu;
  constexpr int P = K + 1;
  const uint32_t lane = threadIdx.x & 31, sub = lane & 3;
  const uint64_t warp = (blockIdx.x * uint64_t(blockDim.x) + threadIdx.x) >> 5;
  const uint64_t nwarps = (gridDim.x * uint64_t(blockDim.x)) >> 5;
  const uint64_t n_text = uint64_t(ix.bwt_len) - 1;
  for (uint64_t base = warp * 8; base < a.n; base += nwarps * 8) {
    const uint64_t i = base + (lane >> 2);
    bool live = i < a.n;
    uint32_t q = 0, j = 0, len = 0, rb0 = 0, s_first = 0, s_last = 0;
    uint64_t s = 0;
    int cut[P + 1];
    const uint32_t* rq = nullptr;
    if (live) {
      const uint32_t g = a.map[i];
      AWRY_CHK(g < a.npieces);
      q = g / P;
      j = g - q * P;
      const uint64_t o0 = a.qoff[q], o1 = a.qoff[q + 1];
      len = checked_len(o0, o1, ByteRange{a.b_lo, a.b_hi});  // 0: refused by the prepass (the call fails)
      const uint2 r = a.sp_cnt[g];
      uint64_t p;
      if (r.y == CNT_AT_TEXT_POS) {  // finished in the text by the search kernel: the piece's one occurrence
        p = r.x;
      } else {
        const uint64_t row = uint64_t(r.x) + (a.c0 + i - a.hoff[g]);
        AWRY_CHK(row < ix.n_full_sa);
        p = __ldg(ix.full_sa + row);
      }
      const uint64_t aj = uint64_t(j) * len / P;
      live = len > uint32_t(K) && p >= aj && p - aj + len <= n_text;
      if (live) {
        s = p - aj;
#pragma unroll
        for (int t = 0; t <= P; t++) cut[t] = int(len - uint32_t(uint64_t(P - t) * len / P));  // search order: piece P-1-t
        const uint64_t w0 = 4 * (q + (o0 >> 6));
        AWRY_CHK(w0 >= a.qw_lo && w0 - a.qw_lo + (len + 7) / 8 / 2 + 8 < a.qw_n);
        rq = reinterpret_cast<const uint32_t*>(a.qwords + w0);
        rb0 = uint32_t(ix.bwt_len - s - len);
        s_first = rb0 >> 6;
        s_last = (rb0 + len - 1) >> 6;
      }
    }
    uint32_t mm[P];
#pragma unroll
    for (int t = 0; t < P; t++) mm[t] = 0;
    uint32_t tot = 0;
    bool going = live;
    for (uint32_t round = 0; __any_sync(FULL, going); round++) {
      const uint32_t sec = s_first + 4 * round + sub;
      if (going && sec <= s_last) {
        AWRY_CHK(uint64_t(sec) * 32 + 31 < ix.n_rtext);
        const u32x8 t = ldg256(ix.rtext + size_t(sec) * 32);
        text_sector_mismatches<P>(t, rq, sec, rb0, cut, mm);
      }
      tot = 0;
#pragma unroll
      for (int t = 0; t < P; t++) tot += mm[t];
      tot += __shfl_xor_sync(FULL, tot, 1);
      tot += __shfl_xor_sync(FULL, tot, 2);
      if (tot > uint32_t(K) || s_first + 4 * (round + 1) > s_last) going = false;
    }
    uint32_t hit_pieces = 0;  // bit t: search-order piece t (original piece P-1-t) has a mismatch
#pragma unroll
    for (int t = 0; t < P; t++) hit_pieces |= (mm[t] != 0u) << t;
    hit_pieces |= __shfl_xor_sync(FULL, hit_pieces, 1);
    hit_pieces |= __shfl_xor_sync(FULL, hit_pieces, 2);
    // pieces 0 .. j-1 are search-order pieces P-j .. P-1
    const uint32_t before = ((1u << P) - 1u) & ~((1u << (P - j)) - 1u);
    const bool accept = live && tot <= uint32_t(K) && (hit_pieces & before) == before;
    if (sub == 0 && i < a.n) {
      if (MODE == VERIFY_LOCATE) {
        a.keys[i] = accept ? (s << 2) | tot : ~0ull;
        if (accept) atomicAdd(reinterpret_cast<unsigned long long*>(a.acc) + (q - a.q0), 1ull);
      } else if (MODE == VERIFY_PLACE) {
        if (accept) {
          const uint64_t at = a.hit_off[q] + atomicAdd(reinterpret_cast<unsigned long long*>(a.acc) + q, 1ull);
          AWRY_CHK(at < a.hit_off[q + 1]);
          a.keys[at] = (s << 2) | tot;
        }
      } else if (accept) {
        atomicAdd(reinterpret_cast<unsigned long long*>(a.counts) + (uint64_t(q) * P + tot), 1ull);
      }
    }
  }
}

template <int K>
static void launch_verify_k(const IndexView& ix, const HammingSlice& a, VerifyMode mode, unsigned grid, cudaStream_t s) {
  if (mode == VERIFY_LOCATE)
    hamming_verify_kernel<K, VERIFY_LOCATE><<<grid, 256, 0, s>>>(ix, a);
  else if (mode == VERIFY_PLACE)
    hamming_verify_kernel<K, VERIFY_PLACE><<<grid, 256, 0, s>>>(ix, a);
  else
    hamming_verify_kernel<K, VERIFY_COUNT><<<grid, 256, 0, s>>>(ix, a);
}

cudaError_t launch_hamming_verify(const IndexView& ix, const HammingSlice& a, uint32_t k, VerifyMode mode, int sm_count,
                                  cudaStream_t s) {
  if (a.n == 0) return cudaSuccess;
  if (k > 3 || ix.rtext == nullptr || ix.full_sa == nullptr) return cudaErrorInvalidValue;
  const unsigned grid = unsigned(std::max<uint64_t>(1, std::min<uint64_t>(uint64_t(sm_count) * 8, (a.n + 63) / 64)));
  switch (k) {
    case 0: launch_verify_k<0>(ix, a, mode, grid, s); break;
    case 1: launch_verify_k<1>(ix, a, mode, grid, s); break;
    case 2: launch_verify_k<2>(ix, a, mode, grid, s); break;
    default: launch_verify_k<3>(ix, a, mode, grid, s); break;
  }
  COUNT_LAUNCH();
  return cudaGetLastError();
}

// locate: keys of the slice sorted per query (rejected keys, ~0, go to the end of their segment).  The segment
// bounds are the reads' candidate bounds made slice-local (qcand[i] - c0): CUB's segmented sort reads its offsets as
// int, so the slice holds fewer than 2^31 candidates and its bounds must not be the absolute ones.
struct SliceBound {
  const uint64_t* qcand;
  uint64_t c0;
  __host__ __device__ long long operator()(uint64_t i) const { return (long long)(qcand[i] - c0); }
};
cudaError_t sort_hamming_keys(const uint64_t* d_keys, uint64_t* d_sorted, uint64_t n, uint64_t nseg,
                              const uint64_t* d_qcand, uint64_t c0, void* d_temp, size_t& temp_bytes, cudaStream_t s) {
  if (n >= (1ull << 31)) return cudaErrorInvalidValue;
  thrust::counting_iterator<uint64_t> idx(0);
  auto begin = thrust::make_transform_iterator(idx, SliceBound{d_qcand, c0});
  cudaError_t e = cub::DeviceSegmentedSort::SortKeys(d_temp, temp_bytes, d_keys, d_sorted, (long long)n, (long long)nseg,
                                                     begin, begin + 1, s);
  if (d_temp != nullptr) COUNT_LAUNCH();
  return e;
}

// exclusive sum of n u64 (the per-query accepted counts -> the slice's CSR offsets)
cudaError_t scan_u64(const uint64_t* d_in, uint64_t* d_out, uint64_t n, void* d_temp, size_t& temp_bytes, cudaStream_t s) {
  cudaError_t e = cub::DeviceScan::ExclusiveSum(d_temp, temp_bytes, d_in, d_out, (long long)n, s);
  if (d_temp != nullptr) COUNT_LAUNCH();
  return e;
}

__global__ void hamming_row_sums_kernel(const uint64_t* __restrict__ counts, uint32_t P, uint64_t nq,
                                        uint64_t* __restrict__ sums) {
  const uint64_t stride = gridDim.x * uint64_t(blockDim.x);
  for (uint64_t q = blockIdx.x * uint64_t(blockDim.x) + threadIdx.x; q <= nq; q += stride) {
    uint64_t t = 0;
    if (q < nq)
      for (uint32_t d = 0; d < P; d++) t += counts[q * P + d];
    sums[q] = t;
  }
}

cudaError_t launch_hamming_row_sums(const uint64_t* d_counts, uint32_t k, uint64_t nq, uint64_t* d_sums, cudaStream_t s) {
  const unsigned grid = unsigned(std::min<uint64_t>((nq + 256) / 256, 148 * 16));
  hamming_row_sums_kernel<<<grid, 256, 0, s>>>(d_counts, k + 1, nq, d_sums);
  COUNT_LAUNCH();
  return cudaGetLastError();
}

__global__ void hamming_decode_kernel(uint64_t* __restrict__ keys, uint64_t n, uint8_t* __restrict__ dist) {
  const uint64_t stride = gridDim.x * uint64_t(blockDim.x);
  for (uint64_t i = blockIdx.x * uint64_t(blockDim.x) + threadIdx.x; i < n; i += stride) {
    const uint64_t key = keys[i];
    keys[i] = key >> 2;
    if (dist) dist[i] = uint8_t(key & 3);
  }
}

cudaError_t launch_hamming_decode(uint64_t* d_keys, uint64_t n, uint8_t* d_dist, cudaStream_t s) {
  if (n == 0) return cudaSuccess;
  const unsigned grid = unsigned(std::min<uint64_t>((n + 255) / 256, 148 * 16));
  hamming_decode_kernel<<<grid, 256, 0, s>>>(d_keys, n, d_dist);
  COUNT_LAUNCH();
  return cudaGetLastError();
}

// sorted keys -> text positions and distances at the query's CSR slot: the accepted keys lead their segment
__global__ void hamming_compact_kernel(const uint64_t* __restrict__ sorted, const uint32_t* __restrict__ map, uint64_t n,
                                       uint32_t pieces, const uint64_t* __restrict__ qcand, uint64_t c0, uint64_t q0,
                                       const uint64_t* __restrict__ qh, uint64_t* __restrict__ pos, uint8_t* __restrict__ dist) {
  const uint64_t stride = gridDim.x * uint64_t(blockDim.x);
  for (uint64_t i = blockIdx.x * uint64_t(blockDim.x) + threadIdx.x; i < n; i += stride) {
    const uint64_t key = sorted[i];
    if (key == ~0ull) continue;
    const uint64_t q = map[i] / pieces;
    const uint64_t o = qh[q - q0] + (c0 + i - qcand[q]);
    pos[o] = key >> 2;
    dist[o] = uint8_t(key & 3);
  }
}

cudaError_t launch_hamming_compact(const uint64_t* d_sorted, const uint32_t* d_map, uint64_t n, uint32_t k,
                                   const uint64_t* d_qcand, uint64_t c0, uint64_t q0, const uint64_t* d_qh, uint64_t* d_pos,
                                   uint8_t* d_dist, cudaStream_t s) {
  if (n == 0) return cudaSuccess;
  const unsigned grid = unsigned(std::min<uint64_t>((n + 255) / 256, 148 * 16));
  hamming_compact_kernel<<<grid, 256, 0, s>>>(d_sorted, d_map, n, k + 1, d_qcand, c0, q0, d_qh, d_pos, d_dist);
  COUNT_LAUNCH();
  return cudaGetLastError();
}

}  // namespace awry
