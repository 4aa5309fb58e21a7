// kernels_map.cu -- read mapping: the best locus per read over the searched strands (awry_map_*, include/awry_b200.h,
// DESIGN.md §1h).  The locate flow of batch.cu counts every read's hits per distance; the kernels here turn the counts
// into each read's bound (best + 1, capped at k), and, once the hits within it are placed and sorted per read, mark the
// first entry of each start, rank the ones at the best distance with a scan, and write one record per read.  No kernel
// walks the hits of one read on one thread: repeat-rich reads hold tens of thousands.
#include "../../include/awry_b200.h"
#include "kernels_common.cuh"

namespace awry {

static_assert(sizeof(awry_mapping) == 32, "4 u64 per mapping");

__constant__ uint8_t c_mapq_second[256] = AWRY_MAPQ_SECOND;

__global__ void map_bound_kernel(const uint64_t* __restrict__ counts, const uint32_t* __restrict__ qlen, uint64_t nq,
                                 uint32_t k, uint32_t shift, uint8_t* __restrict__ best, uint64_t* __restrict__ sums) {
  const uint64_t stride = gridDim.x * uint64_t(blockDim.x);
  const uint32_t P = k + 1, per = 1u << shift;
  for (uint64_t q = blockIdx.x * uint64_t(blockDim.x) + threadIdx.x; q <= nq; q += stride) {
    if (q == nq) {
      sums[nq << shift] = 0;
      continue;
    }
    const uint64_t v0 = q << shift;
    uint32_t b = 0xffu;
    if (qlen[v0] != 0)
      for (uint32_t v = 0; v < per; v++)
        for (uint32_t d = 0; d < P && d < b; d++)
          if (counts[(v0 + v) * P + d]) {
            b = d;
            break;
          }
    for (uint32_t v = 0; v < per; v++) {
      uint64_t t = 0;
      for (uint32_t d = 0; d < P; d++)
        if (within_map_bound(d, b, k)) t += counts[(v0 + v) * P + d];
      sums[v0 + v] = t;
      best[v0 + v] = uint8_t(b);
    }
  }
}

cudaError_t launch_map_bound(const uint64_t* d_counts, const uint32_t* d_qlen, uint64_t nq, uint32_t k, uint32_t shift,
                             uint8_t* d_best, uint64_t* d_sums, cudaStream_t s) {
  const unsigned grid = unsigned(std::min<uint64_t>((nq + 256) / 256, 148 * 16));
  map_bound_kernel<<<grid, 256, 0, s>>>(d_counts, d_qlen, nq, k, shift, d_best, d_sums);
  COUNT_LAUNCH();
  return cudaGetLastError();
}

__global__ void map_read_offsets_kernel(const uint64_t* __restrict__ hit_off, uint64_t nq, uint32_t shift,
                                        uint64_t* __restrict__ roff) {
  const uint64_t stride = gridDim.x * uint64_t(blockDim.x);
  for (uint64_t q = blockIdx.x * uint64_t(blockDim.x) + threadIdx.x; q <= nq; q += stride) roff[q] = hit_off[q << shift];
}

cudaError_t launch_map_read_offsets(const uint64_t* d_hit_off, uint64_t nq, uint32_t shift, uint64_t* d_roff,
                                    cudaStream_t s) {
  const unsigned grid = unsigned(std::min<uint64_t>((nq + 256) / 256, 148 * 16));
  map_read_offsets_kernel<<<grid, 256, 0, s>>>(d_hit_off, nq, shift, d_roff);
  COUNT_LAUNCH();
  return cudaGetLastError();
}

__global__ void map_rekey_kernel(const uint64_t* __restrict__ keys, const uint64_t* __restrict__ hit_off,
                                 const uint64_t* __restrict__ roff, const uint32_t* __restrict__ rmap, uint64_t nq,
                                 uint64_t n, uint32_t shift, uint64_t* __restrict__ out) {
  const uint64_t stride = gridDim.x * uint64_t(blockDim.x);
  const uint64_t total = roff[nq];
  AWRY_CHK(total <= n);
  for (uint64_t i = blockIdx.x * uint64_t(blockDim.x) + threadIdx.x; i < total; i += stride) {
    const uint32_t q = rmap[i];
    AWRY_CHK(q < nq && roff[q] <= i && i < roff[q + 1]);
    const uint64_t key = keys[i];
    const uint64_t strand = shift && i >= hit_off[2 * uint64_t(q) + 1];
    out[i] = ((key >> 2) << 3) | ((key & 3) << 1) | strand;
  }
}

cudaError_t launch_map_rekey(const uint64_t* d_keys, const uint64_t* d_hit_off, const uint64_t* d_roff,
                             const uint32_t* d_rmap, uint64_t nq, uint64_t n, uint32_t shift, uint64_t* d_out,
                             cudaStream_t s) {
  if (n == 0) return cudaSuccess;
  const unsigned grid = unsigned(std::min<uint64_t>((n + 255) / 256, 148 * 16));
  map_rekey_kernel<<<grid, 256, 0, s>>>(d_keys, d_hit_off, d_roff, d_rmap, nq, n, shift, d_out);
  COUNT_LAUNCH();
  return cudaGetLastError();
}

// keys (s << 3) | (d << 1) | strand: sorted, a start's entries are adjacent and its first has the smallest d, then
// strand 0 -- D(s) and strand(s) of the header
__global__ void map_flags_kernel(const uint64_t* __restrict__ keys, const uint64_t* __restrict__ roff,
                                 const uint32_t* __restrict__ rmap, const uint8_t* __restrict__ best, uint64_t nq,
                                 uint64_t n, uint32_t shift, uint64_t* __restrict__ flag, uint32_t* __restrict__ second) {
  const uint64_t stride = gridDim.x * uint64_t(blockDim.x);
  const uint64_t total = roff[nq];
  for (uint64_t i = blockIdx.x * uint64_t(blockDim.x) + threadIdx.x; i <= n; i += stride) {
    if (i >= total) {
      flag[i] = 0;
      continue;
    }
    const uint32_t q = rmap[i];
    AWRY_CHK(q < nq && roff[q] <= i && i < roff[q + 1]);
    const uint64_t key = keys[i];
    const bool first = i == roff[q] || (keys[i - 1] >> 3) != (key >> 3);
    const uint32_t d = uint32_t(key >> 1) & 3u, b = best[uint64_t(q) << shift];
    AWRY_CHK(b != 0xffu && d >= b && d <= b + 1);
    flag[i] = first && d == b;
    if (first && d == b + 1) atomicAdd(second + q, 1u);
  }
}

cudaError_t launch_map_flags(const uint64_t* d_keys, const uint64_t* d_roff, const uint32_t* d_rmap, const uint8_t* d_best,
                             uint64_t nq, uint64_t n, uint32_t shift, uint64_t* d_flag, uint32_t* d_second,
                             cudaStream_t s) {
  const unsigned grid = unsigned(std::min<uint64_t>((n + 256) / 256, 148 * 16));
  map_flags_kernel<<<grid, 256, 0, s>>>(d_keys, d_roff, d_rmap, d_best, nq, n, shift, d_flag, d_second);
  COUNT_LAUNCH();
  return cudaGetLastError();
}

// fmix64(FNV-1a-64 over the codes c_0 .. c_{L-1} of the read).  The words hold the codes in search order: symbol y =
// byte L - 1 - y is nibble y & 15 of word y >> 4, so the read's bytes come from the last symbol down.
__device__ __forceinline__ uint64_t read_hash(const uint64_t* __restrict__ w, uint32_t len) {
  uint64_t h = 0xcbf29ce484222325ull;
  for (int32_t wi = int32_t((len - 1) >> 4); wi >= 0; wi--) {
    const uint64_t x = __ldg(w + wi);
    const int top = uint32_t(wi) == (len - 1) >> 4 ? int((len - 1) & 15) : 15;
    for (int j = top; j >= 0; j--) {
      h ^= (x >> (4 * j)) & 15u;
      h *= 0x100000001b3ull;
    }
  }
  h ^= h >> 33;
  h *= 0xff51afd7ed558ccdull;
  h ^= h >> 33;
  h *= 0xc4ceb9fe1a85ec53ull;
  h ^= h >> 33;
  return h;
}

// one thread per read.  The primary is the best representative of rank h mod n_best: the first entry i of the read
// with rank[i + 1] > rank[lo] + that rank, found by bisection.
__global__ void __launch_bounds__(256) map_reads_kernel(IndexView ix, MapReads m) {
  const uint64_t stride = gridDim.x * uint64_t(blockDim.x);
  if (m.aln_end && blockIdx.x == 0 && threadIdx.x == 0) *m.aln_end = m.nq;
  for (uint64_t q = blockIdx.x * uint64_t(blockDim.x) + threadIdx.x; q < m.nq; q += stride) {
    const uint64_t v0 = q << m.shift;
    const uint32_t len = m.qlen[v0];
    const uint64_t lo = m.roff[q], hi = m.roff[q + 1];
    const uint64_t base = m.rank[lo], nb = m.rank[hi] - base;
    uint64_t hit[2] = {~0ull, ~0ull}, counts = 0, tail = (m.k + 1) | (uint64_t(AWRY_MAP_UNMAPPED) << 24);
    uint32_t v = uint32_t(v0);
    if (len == 0) {
      tail |= uint64_t(AWRY_MAP_REFUSED) << 24;
    } else if (nb) {
      uint64_t t = 0;
      if (nb >= 2) {
        const uint64_t w0 = 4 * (v0 + (m.qoff[v0] >> 6));
        AWRY_CHK(w0 >= m.qw_lo && w0 - m.qw_lo + (len + 15) / 16 <= m.qw_n);
        t = read_hash(m.qwords + w0, len) % nb;
      }
      uint64_t a = lo, b = hi - 1;
      while (a < b) {
        const uint64_t mid = (a + b) >> 1;
        if (m.rank[mid + 1] > base + t)
          b = mid;
        else
          a = mid + 1;
      }
      const uint64_t key = m.keys[a];
      const uint32_t d = uint32_t(key >> 1) & 3u, strand = uint32_t(key & 1), second = m.second[q];
      AWRY_CHK(nb < (1ull << 32) && d == m.best[v0]);
      const uint32_t mapq = nb >= 2 ? 0u : d == m.k ? 25u : uint32_t(c_mapq_second[min(second, 255u)]);
      map_location(ix, key >> 3, hit);
      counts = nb | (uint64_t(second) << 32);
      tail = d | (strand << 8) | (mapq << 16);
      v |= strand;
    }
    uint64_t* const dst = m.out + 4 * q;
    dst[0] = hit[0];
    dst[1] = hit[1];
    dst[2] = counts;
    dst[3] = tail;
    if (m.aln_map) {
      m.aln_map[q] = v;
      m.aln_hits[2 * q] = hit[0];
      m.aln_hits[2 * q + 1] = hit[1];
    }
  }
}

cudaError_t launch_map_reads(const IndexView& ix, const MapReads& m, cudaStream_t s) {
  if (m.nq == 0) return cudaSuccess;
  const unsigned grid = unsigned(std::min<uint64_t>((m.nq + 255) / 256, 148 * 16));
  map_reads_kernel<<<grid, 256, 0, s>>>(ix, m);
  COUNT_LAUNCH();
  return cudaGetLastError();
}

}  // namespace awry
