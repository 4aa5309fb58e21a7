// kernels_locate.cu -- locate pass 2 (CSR offsets, row expansion, LF-walk / unsampled-SA gather, position
// mapping), the load-time unsampling of the suffix array, and the two single-step kernels.
// Reference: FmIndex::locate_string / backstep (/root/reference/src/fm_index.rs:516-544, :585-593),
// CompressedSuffixArray::reconstruct_value (compressed_suffix_array.rs:76-106),
// SequenceIndex::get_seq_location (sequence_index.rs:108-141).
#include <algorithm>
#include <cub/device/device_scan.cuh>
#include <cub/device/device_segmented_sort.cuh>
#include <thrust/iterator/counting_iterator.h>
#include <thrust/iterator/transform_iterator.h>

#include "kernels_common.cuh"

namespace awry {

// ------------------------------------------------------------------ locate

struct CountOf {
  const uint2* r;
  uint64_t nq;
  __host__ __device__ uint64_t operator()(uint64_t i) const {
    return i < nq ? (r[i].y == CNT_AT_TEXT_POS ? 1ull : uint64_t(r[i].y)) : 0ull;
  }
};

// exclusive scan of the per-query hit counts -> CSR offsets, d_hit_off[nq] = total
cudaError_t scan_hit_offsets(const IndexView& ix, const void* d_sp_cnt, uint64_t nq, uint64_t* d_hit_off, void* d_temp,
                             size_t& temp_bytes, cudaStream_t s) {
  if (ix.wide) return scan_hit_offsets_wide(d_sp_cnt, nq, d_hit_off, d_temp, temp_bytes, s);
  thrust::counting_iterator<uint64_t> idx(0);
  auto in = thrust::make_transform_iterator(idx, CountOf{static_cast<const uint2*>(d_sp_cnt), nq});
  cudaError_t e = cub::DeviceScan::ExclusiveSum(d_temp, temp_bytes, in, d_hit_off, nq + 1, s);
  if (d_temp != nullptr) COUNT_LAUNCH();
  return e;
}

// Pass 2a: expand the CSR (query -> hit range) into one BWT row per hit, written into the low
// 32 bits of each output slot (the walk overwrites the slot with the result).  A lane writes the
// first 8 rows of its query; longer intervals are written by the whole warp, so a query with 10^5
// hits costs ~3000 coalesced warp iterations instead of serialising one thread.
__global__ void __launch_bounds__(256)
    expand_rows_kernel(const uint2* __restrict__ sp_cnt, const uint64_t* __restrict__ hit_off, uint64_t nq,
                       uint32_t* __restrict__ out32, uint32_t slot_u32) {
  const uint32_t lane = threadIdx.x & 31;
  const uint64_t warp = (blockIdx.x * uint64_t(blockDim.x) + threadIdx.x) >> 5;
  const uint64_t nwarps = (gridDim.x * uint64_t(blockDim.x)) >> 5;
  for (uint64_t base = warp * 32; base < nq; base += nwarps * 32) {
    uint64_t q = base + lane;
    uint32_t sp = 0, cnt = 0;
    uint64_t off = 0;
    if (q < nq) {
      uint2 r = sp_cnt[q];
      sp = r.x;
      cnt = r.y;
      off = hit_off[q];
    }
    uint32_t small = cnt < 8 ? cnt : 8;
    for (uint32_t i = 0; i < small; i++) out32[(off + i) * slot_u32] = sp + i;
    uint32_t big = __ballot_sync(0xffffffffu, cnt > 8);
    while (big) {
      int L = __ffs(big) - 1;
      big &= big - 1;
      uint32_t s = __shfl_sync(0xffffffffu, sp, L), c = __shfl_sync(0xffffffffu, cnt, L);
      uint64_t o = __shfl_sync(0xffffffffu, off, L);
      for (uint32_t i = 8 + lane; i < c; i += 32) out32[(o + i) * slot_u32] = s + i;
    }
  }
}

__device__ __forceinline__ void finish_hit(const IndexView& ix, uint32_t row, uint32_t steps, uint64_t* slot,
                                           bool map) {
  uint64_t loc = (sa_sample(ix, row) + steps) % ix.bwt_len;  // fm_index.rs:533-534
  if (map)
    map_location(ix, loc, slot);
  else
    slot[0] = loc;
}

// Pass 2b, nucleotide: 2 lanes per hit, each LDG.256 half of the 64-B block, so one LF step is ONE
// line request (a one-thread walk issues four LDG.128 to the same line).  Lanes refill: a pair whose
// walk ends takes the next hit, so the geometric walk lengths (rows, not text positions, are sampled:
// compressed_suffix_array.rs:109-111) do not idle the rest of the warp.  The lane holding the row's
// chunk extracts the BWT symbol and broadcasts it; both lanes rank their two chunks; xor-shuffle.
// Warp-convergent loop (exit by vote) so the shuffles use the full mask.
constexpr uint64_t WALK_TICKET = 32;  // hits per ticket (8 measured slower: 3.6 vs 2.5 ms per 10 M hits)

template <bool MAP>
__global__ void __launch_bounds__(256) walk_dna_kernel(IndexView ix, uint64_t n_hits, uint64_t* __restrict__ out, bool dynamic) {
  constexpr int SLOT = MAP ? 2 : 1;
  constexpr uint32_t FULL = 0xffffffffu;
  const uint32_t lane = threadIdx.x & 31, sub = lane & 1, gbase = lane - sub;
  // hits are handed out dynamically, WALK_TICKET at a time; the counter sits behind the output slots
  unsigned long long* const ticket = reinterpret_cast<unsigned long long*>(out + SLOT * n_hits);
  // small batches: a static stride keeps every group busy from the start (a ticket of 32 hits would feed
  // only n_hits / 32 groups, and smaller tickets serialise on the counter: same-address atomics retire at
  // ~0.35 G/s); large batches: tickets, so that the fast SMs take more
  const uint64_t stride = (gridDim.x * uint64_t(blockDim.x)) >> 1;
  uint64_t h = dynamic ? 0 : (blockIdx.x * uint64_t(blockDim.x) + threadIdx.x) >> 1, h_end = dynamic ? 0 : n_hits;
  const uint64_t step = dynamic ? 1 : stride;
  bool more = dynamic;
  uint64_t cur = 0;
  uint32_t row = 0, steps = 0;
  bool have = false;
  for (;;) {
    if (!have && h >= h_end && more) {
      unsigned long long t = 0;
      if (sub == 0) t = atomicAdd(ticket, (unsigned long long)WALK_TICKET);
      t = __shfl_sync(0x3u << gbase, t, gbase);
      more = t < n_hits;
      h = more ? t : 0;
      h_end = more ? (n_hits - t < WALK_TICKET ? n_hits : t + WALK_TICKET) : 0;
    }
    if (!have && h < h_end) {
      cur = h;
      h += step;
      row = uint32_t(out[SLOT * cur]);
      steps = 0;
      have = true;
    }
    if (__all_sync(FULL, !have && !more && h >= h_end)) break;
    if (have && row_is_sampled(ix, row)) {
      if (sub == 0) finish_hit(ix, row, steps, out + SLOT * cur, MAP);
      have = false;
    }
    const uint32_t blk = row >> 7, l = row & 127;
    LaneChunks<2> x;
    x.c[0] = x.c[1] = make_uint4(0, 0, 0, 0);
    AWRY_CHK(!have || uint64_t(blk) * DNA_BLOCK_UINT4 + 3 < ix.n_blocks_u4);
    if (have) x.load(ix.blocks + size_t(blk) * DNA_BLOCK_UINT4, sub);
    const uint4 ch = (l & 32) ? x.c[1] : x.c[0];
    const uint32_t t = l & 31;
    uint32_t c = ((ch.x >> t) & 1u) | (((ch.y >> t) & 1u) << 1) | (((ch.z >> t) & 1u) << 2);
    c = __shfl_sync(FULL, c, gbase + (l >> 6));  // from the lane that owns chunk l/32
    uint32_t r = 0;
    if (have && c < 4) r = dna_partial_rank<2>(x, sub, l, c, (c & 1) ? ~0u : 0u, (c & 2) ? ~0u : 0u);
    r += __shfl_xor_sync(FULL, r, 1);
    if (have) {
      if (c >= uint32_t(DNA_SENTINEL))
        row = 0;  // the '$' row: fm_index.rs:587-589
      else if (c == uint32_t(DNA_N))
        row = lf_backstep<0>(ix, row);  // rare: scalar step
      else
        row = ix.c_lo[c] + r - 1;
      steps++;
    }
  }
}

// Pass 2b, amino: 4 lanes per hit on the 128-B block (one line request per LF step); the lane that
// holds the row's 32-row slice extracts the symbol index from its 5 planes and broadcasts it.
template <bool MAP>
__global__ void __launch_bounds__(256) walk_amino_kernel(IndexView ix, uint64_t n_hits, uint64_t* __restrict__ out, bool dynamic) {
  constexpr int SLOT = MAP ? 2 : 1;
  constexpr uint32_t FULL = 0xffffffffu;
  const uint32_t lane = threadIdx.x & 31, sub = lane & 3, gbase = lane - sub;
  unsigned long long* const ticket = reinterpret_cast<unsigned long long*>(out + SLOT * n_hits);
  const uint64_t stride = (gridDim.x * uint64_t(blockDim.x)) >> 2;
  uint64_t h = dynamic ? 0 : (blockIdx.x * uint64_t(blockDim.x) + threadIdx.x) >> 2, h_end = dynamic ? 0 : n_hits;
  const uint64_t step = dynamic ? 1 : stride;
  bool more = dynamic;
  uint64_t cur = 0;
  uint32_t row = 0, steps = 0;
  bool have = false;
  for (;;) {
    if (!have && h >= h_end && more) {
      unsigned long long t = 0;
      if (sub == 0) t = atomicAdd(ticket, (unsigned long long)WALK_TICKET);
      t = __shfl_sync(0xfu << gbase, t, gbase);
      more = t < n_hits;
      h = more ? t : 0;
      h_end = more ? (n_hits - t < WALK_TICKET ? n_hits : t + WALK_TICKET) : 0;
    }
    if (!have && h < h_end) {
      cur = h;
      h += step;
      row = uint32_t(out[SLOT * cur]);
      steps = 0;
      have = true;
    }
    if (__all_sync(FULL, !have && !more && h >= h_end)) break;
    if (have && row_is_sampled(ix, row)) {
      if (sub == 0) finish_hit(ix, row, steps, out + SLOT * cur, MAP);
      have = false;
    }
    const uint32_t blk = row >> 6, l = row & 63;
    u32x8 x;
#pragma unroll
    for (int i = 0; i < 8; i++) x.v[i] = 0;
    AWRY_CHK(!have || uint64_t(blk) * AMINO_BLOCK_UINT4 + 7 < ix.n_blocks_u4);
    if (have) x = ldg256(ix.blocks + size_t(blk) * AMINO_BLOCK_UINT4 + 2 * sub);
    const uint32_t t = l & 31;
    uint32_t c = 0;
#pragma unroll
    for (int p = 0; p < 5; p++) c |= ((x.v[p] >> t) & 1u) << p;
    c = __shfl_sync(FULL, c, gbase + (l >> 5));  // from the lane that owns rows 32*(l/32)..
    uint32_t r = 0;
    if (have && c != uint32_t(AMINO_SENTINEL) && c <= 21) {
      AminoSlice s = amino_slice(x, sub, c);
      r = __popc(s.match & low_mask(int(l) + 1 - int(32 * sub))) + s.count;
    }
    r += __shfl_xor_sync(FULL, r, 1);
    r += __shfl_xor_sync(FULL, r, 2);
    if (have) {
      row = (c == uint32_t(AMINO_SENTINEL) || c > 21) ? 0u : ix.c_lo[c] + r - 1;  // '$' row -> 0
      steps++;
    }
  }
}

// ---- unsampled suffix array: the locate accelerator (derived at load time, like the pair index) ----
// The reference keeps SA[row] only for rows with row % ratio == 0 (compressed_suffix_array.rs:109-111)
// and pays a geometric LF-walk per hit (fm_index.rs:521-537).  180 GB of HBM hold the whole array:
// 4 B x bwt_len (12.4 GB for the 3.1 Gbp config).  It is rebuilt from the sampled one with ONE LF step
// per BWT row: a walker starts at every sampled row r with p = SA[r] and writes SA[LF^s(r)] = p - s
// until it reaches the next sampled row or the '$' row (SA = 0); the LF permutation is one cycle cut at
// the sampled rows, so every row is written exactly once.  Same lane-group step as the walk kernels.
constexpr uint64_t UNSAMPLE_TICKET = 32;  // sampled rows per ticket

// What a walker does with (row, SA[row]) at every row it passes:
//   UNSAMPLE_FULL   full[row] = SA[row]                                   (the unsampled array)
//   UNSAMPLE_MARK   sets the mark bit of rows with SA[row] % ratio == 0   (walk blocks, pass 1)
//   UNSAMPLE_POS    pos_samples[rank of the marked row] = SA[row] / ratio (pass 2, once the ranks exist)
enum UnsampleMode { UNSAMPLE_FULL = 0, UNSAMPLE_MARK = 1, UNSAMPLE_POS = 2 };

// word index (32-bit words) of row group g's planes inside a walk block: 4g .. 4g+2, mark = 4g+3
__device__ __forceinline__ uint32_t* walk_mark_word(uint4* walk, uint32_t row, uint32_t& bit) {
  const uint32_t blk = row / WALK_ROWS_PER_BLOCK, l = row - blk * WALK_ROWS_PER_BLOCK;
  bit = l & 31;
  return reinterpret_cast<uint32_t*>(walk + size_t(blk) * WALK_BLOCK_UINT4) + 4 * (l >> 5) + 3;
}
// marked rows before `row` inside its walk block (one thread; load time only)
__device__ __forceinline__ uint32_t walk_marks_before(const uint4* walk, uint32_t row) {
  const uint32_t blk = row / WALK_ROWS_PER_BLOCK, l = row - blk * WALK_ROWS_PER_BLOCK;
  const uint32_t* w = reinterpret_cast<const uint32_t*>(walk + size_t(blk) * WALK_BLOCK_UINT4);
  uint32_t n = 0;
  for (uint32_t g = 0; g < (l >> 5); g++) n += __popc(w[4 * g + 3]);
  return n + __popc(w[4 * (l >> 5) + 3] & ((1u << (l & 31)) - 1u));
}

template <int MODE>
__device__ __forceinline__ void unsample_visit(const IndexView& ix, uint32_t row, uint32_t p, uint32_t* __restrict__ full,
                                               uint4* __restrict__ walk, uint32_t* __restrict__ pos_samples) {
  if (MODE == UNSAMPLE_FULL) {
    AWRY_CHK(row < ix.bwt_len);
    full[row] = p;
    return;
  }
  if (p % ix.lean_ratio != 0) return;
  if (MODE == UNSAMPLE_MARK) {
    uint32_t bit;
    uint32_t* w = walk_mark_word(walk, row, bit);
    atomicOr(w, 1u << bit);
  } else {
    const uint32_t at = ix.walk_rank[row / WALK_ROWS_PER_BLOCK] + walk_marks_before(walk, row);
    AWRY_CHK(row / WALK_ROWS_PER_BLOCK < ix.n_walk_rank && at < ix.n_pos_samples);
    pos_samples[at] = p / ix.lean_ratio;
  }
}

template <int MODE>
__global__ void __launch_bounds__(256)
    unsample_dna_kernel(IndexView ix, uint64_t n_elems, uint32_t* __restrict__ full, uint4* __restrict__ walk,
                        uint32_t* __restrict__ pos_samples, unsigned long long* __restrict__ ticket) {
  constexpr uint32_t FULL = 0xffffffffu;
  const uint32_t lane = threadIdx.x & 31, sub = lane & 1, gbase = lane - sub;
  // sampled rows are handed out dynamically, UNSAMPLE_TICKET at a time (walk lengths are geometric and the
  // SMs do not all see the same random-access throughput)
  uint64_t e = 0, e_end = 0;
  bool more = true;
  uint32_t row = 0, p = 0;
  bool have = false;
  for (;;) {
    if (!have && e == e_end && more) {
      unsigned long long t = 0;
      if (sub == 0) t = atomicAdd(ticket, (unsigned long long)UNSAMPLE_TICKET);
      t = __shfl_sync(0x3u << gbase, t, gbase);
      more = t < n_elems;
      e = more ? t : 0;
      e_end = more ? (n_elems - t < UNSAMPLE_TICKET ? n_elems : t + UNSAMPLE_TICKET) : 0;
    }
    if (!have && e < e_end) {
      row = uint32_t(e * ix.sa_ratio);
      p = uint32_t(sa_sample(ix, row));
      e++;
      have = true;
      if (sub == 0) unsample_visit<MODE>(ix, row, p, full, walk, pos_samples);
    }
    if (__all_sync(FULL, !have && !more && e == e_end)) break;
    const uint32_t blk = row >> 7, l = row & 127;
    LaneChunks<2> x;
    x.c[0] = x.c[1] = make_uint4(0, 0, 0, 0);
    AWRY_CHK(!have || uint64_t(blk) * DNA_BLOCK_UINT4 + 3 < ix.n_blocks_u4);
    if (have) x.load(ix.blocks + size_t(blk) * DNA_BLOCK_UINT4, sub);
    const uint4 ch = (l & 32) ? x.c[1] : x.c[0];
    const uint32_t t = l & 31;
    uint32_t c = ((ch.x >> t) & 1u) | (((ch.y >> t) & 1u) << 1) | (((ch.z >> t) & 1u) << 2);
    c = __shfl_sync(FULL, c, gbase + (l >> 6));
    uint32_t r = 0;
    if (have && c < 4) r = dna_partial_rank<2>(x, sub, l, c, (c & 1) ? ~0u : 0u, (c & 2) ? ~0u : 0u);
    r += __shfl_xor_sync(FULL, r, 1);
    if (have) {
      if (c >= uint32_t(DNA_SENTINEL)) {
        have = false;  // the '$' row (SA = 0, already visited): LF would wrap to row 0, a sampled row
      } else {
        row = c == uint32_t(DNA_N) ? lf_backstep<0>(ix, row) : ix.c_lo[c] + r - 1;
        p--;
        if (row_is_sampled(ix, row))
          have = false;
        else if (sub == 0)
          unsample_visit<MODE>(ix, row, p, full, walk, pos_samples);
      }
    }
  }
}

__global__ void __launch_bounds__(256)
    unsample_amino_kernel(IndexView ix, uint64_t n_elems, uint32_t* __restrict__ full) {
  constexpr uint32_t FULL = 0xffffffffu;
  const uint32_t lane = threadIdx.x & 31, sub = lane & 3, gbase = lane - sub;
  unsigned long long* const ticket = reinterpret_cast<unsigned long long*>(full + ((size_t(ix.bwt_len) + 3) & ~size_t(1)));
  uint64_t e = 0, e_end = 0;
  bool more = true;
  uint32_t row = 0, p = 0;
  bool have = false;
  for (;;) {
    if (!have && e == e_end && more) {
      unsigned long long t = 0;
      if (sub == 0) t = atomicAdd(ticket, (unsigned long long)UNSAMPLE_TICKET);
      t = __shfl_sync(0xfu << gbase, t, gbase);
      more = t < n_elems;
      e = more ? t : 0;
      e_end = more ? (n_elems - t < UNSAMPLE_TICKET ? n_elems : t + UNSAMPLE_TICKET) : 0;
    }
    if (!have && e < e_end) {
      row = uint32_t(e * ix.sa_ratio);
      p = uint32_t(sa_sample(ix, row));
      e++;
      have = true;
      if (sub == 0) full[row] = p;
    }
    if (__all_sync(FULL, !have && !more && e == e_end)) break;
    const uint32_t blk = row >> 6, l = row & 63;
    u32x8 x;
#pragma unroll
    for (int i = 0; i < 8; i++) x.v[i] = 0;
    AWRY_CHK(!have || uint64_t(blk) * AMINO_BLOCK_UINT4 + 7 < ix.n_blocks_u4);
    if (have) x = ldg256(ix.blocks + size_t(blk) * AMINO_BLOCK_UINT4 + 2 * sub);
    const uint32_t t = l & 31;
    uint32_t c = 0;
#pragma unroll
    for (int q = 0; q < 5; q++) c |= ((x.v[q] >> t) & 1u) << q;
    c = __shfl_sync(FULL, c, gbase + (l >> 5));
    uint32_t r = 0;
    const bool sym_ok = c != uint32_t(AMINO_SENTINEL) && c <= 21;
    if (have && sym_ok) {
      AminoSlice sl = amino_slice(x, sub, c);
      r = __popc(sl.match & low_mask(int(l) + 1 - int(32 * sub))) + sl.count;
    }
    r += __shfl_xor_sync(FULL, r, 1);
    r += __shfl_xor_sync(FULL, r, 2);
    if (have) {
      if (!sym_ok) {
        have = false;
      } else {
        row = ix.c_lo[c] + r - 1;
        p--;
        if (row_is_sampled(ix, row))
          have = false;
        else if (sub == 0)
          full[row] = p;
      }
    }
  }
}

cudaError_t build_full_sa(const IndexView& ix, uint32_t* d_full, int sm_count, cudaStream_t s) {
  const uint64_t n_elems = (uint64_t(ix.bwt_len) + ix.sa_ratio - 1) / ix.sa_ratio;
  const uint64_t lanes = ix.alphabet == 0 ? 2 : 4;
  unsigned grid = unsigned(std::max<uint64_t>(1, std::min<uint64_t>(uint64_t(sm_count) * 8, (lanes * n_elems + 255) / 256)));
  // ticket counter: 8 aligned bytes behind the array (the caller allocates 4 * bwt_len + 256)
  cudaError_t e0 = cudaMemsetAsync(d_full + ((size_t(ix.bwt_len) + 3) & ~size_t(1)), 0, 8, s);
  if (e0 != cudaSuccess) return e0;
  if (ix.alphabet == 0)
    unsample_dna_kernel<UNSAMPLE_FULL><<<grid, 256, 0, s>>>(
        ix, n_elems, d_full, nullptr, nullptr,
        reinterpret_cast<unsigned long long*>(d_full + ((size_t(ix.bwt_len) + 3) & ~size_t(1))));
  else
    unsample_amino_kernel<<<grid, 256, 0, s>>>(ix, n_elems, d_full);
  COUNT_LAUNCH();
  return cudaGetLastError();
}

// ---- the text, reversed (IndexView::rtext): text[SA[row] - 1] = BWT[row], so reversed index n - SA[row] (0 for
// the '$' row, whose SA is 0) gets the row's device symbol.  One thread per row: rows and suffix-array elements
// are read in order, the nibbles land at random (atomicOr into a zeroed array). ----
__global__ void __launch_bounds__(256) rtext_kernel(IndexView ix, uint32_t* __restrict__ rtext) {
  const uint64_t stride = gridDim.x * uint64_t(blockDim.x);
  const uint32_t n = ix.bwt_len;
  for (uint64_t r64 = blockIdx.x * uint64_t(blockDim.x) + threadIdx.x; r64 < n; r64 += stride) {
    const uint32_t row = uint32_t(r64), l = row & 127, t = l & 31;
    AWRY_CHK(uint64_t(row >> 7) * DNA_BLOCK_UINT4 + 3 < ix.n_blocks_u4 && row < ix.n_full_sa);
    const uint4 ch = ldg128(ix.blocks + size_t(row >> 7) * DNA_BLOCK_UINT4 + (l >> 5));
    const uint32_t c = ((ch.x >> t) & 1u) | (((ch.y >> t) & 1u) << 1) | (((ch.z >> t) & 1u) << 2);
    const uint32_t p = __ldg(ix.full_sa + row);
    const uint32_t i = p == 0 ? 0u : n - p;
    AWRY_CHK(p < n && uint64_t(i >> 3) * 4 + 3 < ix.n_rtext);
    atomicOr(rtext + (i >> 3), c << (4u * (i & 7u)));
  }
}

// protein: one byte per symbol, so plain byte stores
__global__ void __launch_bounds__(256) rtext_amino_kernel(IndexView ix, uint8_t* __restrict__ rtext) {
  const uint64_t stride = gridDim.x * uint64_t(blockDim.x);
  const uint32_t n = ix.bwt_len;
  for (uint64_t r64 = blockIdx.x * uint64_t(blockDim.x) + threadIdx.x; r64 < n; r64 += stride) {
    const uint32_t row = uint32_t(r64);
    AWRY_CHK(row < ix.n_full_sa);
    const uint32_t c = amino_symbol_at(ix, row);
    const uint32_t p = __ldg(ix.full_sa + row);
    const uint32_t i = p == 0 ? 0u : n - p;
    AWRY_CHK(p < n && i < ix.n_rtext);
    rtext[i] = uint8_t(c);
  }
}

cudaError_t build_rtext(const IndexView& ix, uint8_t* d_rtext, cudaStream_t s) {
  if (ix.full_sa == nullptr || ix.wide != nullptr) return cudaErrorInvalidValue;
  const size_t bytes = rtext_bytes(int(ix.alphabet), ix.bwt_len);
  cudaError_t e = cudaMemsetAsync(d_rtext, 0, bytes, s);
  if (e != cudaSuccess) return e;
  IndexView v = ix;
  v.n_rtext = bytes;
  const unsigned grid = unsigned(std::max<uint64_t>(1, std::min<uint64_t>(1u << 20, (uint64_t(ix.bwt_len) + 255) / 256)));
  if (ix.alphabet != 0)
    rtext_amino_kernel<<<grid, 256, 0, s>>>(v, d_rtext);
  else
  rtext_kernel<<<grid, 256, 0, s>>>(v, reinterpret_cast<uint32_t*>(d_rtext));
  COUNT_LAUNCH();
  return cudaGetLastError();
}

// ---- memory-lean bounded locate: walk blocks + position-sampled suffix array (layout.cuh) ----

// planes of the 1-step blocks re-laid into walk blocks (a 32-row group of a walk block is exactly one 32-row
// chunk of a 64-B block: 224 = 7 x 32), marks cleared; the thread of group 6 also ranks A, C, G, T up to the
// block start.  One thread per (walk block, row group).
__global__ void walk_planes_kernel(IndexView ix, uint4* __restrict__ walk, uint64_t n_wblocks) {
  const uint64_t t = blockIdx.x * uint64_t(blockDim.x) + threadIdx.x;
  if (t >= n_wblocks * 7) return;
  const uint64_t blk = t / 7;
  const uint32_t g = uint32_t(t - blk * 7);
  const uint64_t row0 = blk * WALK_ROWS_PER_BLOCK + 32 * g;
  const uint64_t covered = ((uint64_t(ix.bwt_len) + 255) / 256) * 256;  // rows the 1-step blocks hold (padded with code 7)
  uint4 ch = make_uint4(~0u, ~0u, ~0u, 0u);
  if (row0 < covered) ch = ldg128(ix.blocks + size_t(row0 >> 7) * DNA_BLOCK_UINT4 + ((row0 >> 5) & 3));
  uint32_t* w = reinterpret_cast<uint32_t*>(walk + blk * WALK_BLOCK_UINT4);
  w[4 * g + 0] = ch.x;
  w[4 * g + 1] = ch.y;
  w[4 * g + 2] = ch.z;
  w[4 * g + 3] = 0;
  if (g == 6) {
    const uint64_t start = blk * WALK_ROWS_PER_BLOCK;
    uint32_t cnt[4] = {0, 0, 0, 0};
    if (start != 0 && start - 1 < covered) {
      const uint32_t pos = uint32_t(start - 1);
      DnaBlockRegs b = dna_load_block(ix, pos >> 7);
      for (uint32_t c = 0; c < 4; c++) cnt[c] = dna_occ_in_block(ix, b, pos >> 7, pos & 127, c);
    }
    for (int c = 0; c < 4; c++) w[28 + c] = cnt[c];
  }
}

__global__ void walk_mark_counts_kernel(const uint4* __restrict__ walk, uint64_t n_wblocks, uint32_t* __restrict__ out) {
  const uint64_t blk = blockIdx.x * uint64_t(blockDim.x) + threadIdx.x;
  if (blk >= n_wblocks) return;
  const uint32_t* w = reinterpret_cast<const uint32_t*>(walk + blk * WALK_BLOCK_UINT4);
  uint32_t n = 0;
  for (int g = 0; g < 7; g++) n += __popc(w[4 * g + 3]);
  out[blk] = n;
}

uint64_t walk_block_count(uint64_t bwt_len) { return (bwt_len + WALK_ROWS_PER_BLOCK - 1) / WALK_ROWS_PER_BLOCK; }

// view: blocks / sa_words / lean_ratio set; d_walk: walk_block_count x 128 B; d_rank: walk_block_count + 1 u32;
// d_pos: ceil(bwt_len / lean_ratio) + 4 u32 (the last words serve as the walkers' ticket counter)
cudaError_t build_lean_sa(const IndexView& ix, uint4* d_walk, uint32_t* d_rank, uint32_t* d_pos, int sm_count,
                          cudaStream_t s) {
  if (ix.alphabet != 0) return cudaErrorInvalidValue;
  const uint64_t nb = walk_block_count(ix.bwt_len);
  const uint64_t n_elems = (uint64_t(ix.bwt_len) + ix.sa_ratio - 1) / ix.sa_ratio;  // walkers: one per row the FILE sampled
  const uint64_t n_pos = (uint64_t(ix.bwt_len) + ix.lean_ratio - 1) / ix.lean_ratio;  // marked rows
  walk_planes_kernel<<<unsigned((nb * 7 + 255) / 256), 256, 0, s>>>(ix, d_walk, nb);
  COUNT_LAUNCH();
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return e;
  unsigned long long* ticket = reinterpret_cast<unsigned long long*>(d_pos + ((n_pos + 1) & ~uint64_t(1)));
  const unsigned grid = unsigned(std::max<uint64_t>(1, std::min<uint64_t>(uint64_t(sm_count) * 8, (2 * n_elems + 255) / 256)));
  if ((e = cudaMemsetAsync(ticket, 0, 8, s)) != cudaSuccess) return e;
  unsample_dna_kernel<UNSAMPLE_MARK><<<grid, 256, 0, s>>>(ix, n_elems, nullptr, d_walk, nullptr, ticket);
  COUNT_LAUNCH();
  if ((e = cudaGetLastError()) != cudaSuccess) return e;
  walk_mark_counts_kernel<<<unsigned((nb + 255) / 256), 256, 0, s>>>(d_walk, nb, d_rank);
  COUNT_LAUNCH();
  if ((e = cudaGetLastError()) != cudaSuccess) return e;
  size_t tb = 0;
  if ((e = cub::DeviceScan::ExclusiveSum(nullptr, tb, d_rank, d_rank, (long long)(nb + 1), s)) != cudaSuccess) return e;
  void* d_temp = nullptr;
  if ((e = cudaMalloc(&d_temp, tb + 16)) != cudaSuccess) return e;
  e = cub::DeviceScan::ExclusiveSum(d_temp, tb, d_rank, d_rank, (long long)(nb + 1), s);
  COUNT_LAUNCH();
  if (e == cudaSuccess) e = cudaMemsetAsync(ticket, 0, 8, s);
  if (e == cudaSuccess) {
    IndexView v = ix;
    v.walk_blocks = d_walk;
    v.walk_rank = d_rank;
    unsample_dna_kernel<UNSAMPLE_POS><<<grid, 256, 0, s>>>(v, n_elems, nullptr, d_walk, d_pos, ticket);
    COUNT_LAUNCH();
    e = cudaGetLastError();
  }
  cudaError_t e2 = cudaStreamSynchronize(s);
  cudaFree(d_temp);
  return e != cudaSuccess ? e : e2;
}

// Pass 2b on the walk blocks: 4 lanes per hit, one LDG.256 each = ONE line request per LF step; the lane
// that holds the row's 32-row group extracts the symbol and the mark bit and broadcasts them.  A marked row
// ends the walk: its rank among the marked rows (walk_rank + the marks before it in the block, already in
// registers) indexes the position samples, and the hit is sample * ratio + steps.  At most ratio - 1 steps, no
// wrap through the '$' row (text position 0 is marked).  Hits are handed out to a WARP in runs of consecutive
// hit numbers (a pool in registers topped up with one atomic): the hits of a long interval are consecutive BWT
// rows whose walks stay next to each other while their BWT symbols agree, so their block reads fall into the
// same lines of the same load instruction and are served by one request (repeat-rich text, BASELINE cfg5).
constexpr uint32_t LEAN_TICKET = 64;  // hits per warp ticket

template <bool MAP>
__global__ void __launch_bounds__(256) walk_lean_kernel(IndexView ix, uint64_t n_hits, uint64_t* __restrict__ out) {
  constexpr int SLOT = MAP ? 2 : 1;
  constexpr uint32_t FULL = 0xffffffffu;
  const uint32_t lane = threadIdx.x & 31, sub = lane & 3, gbase = lane - sub;
  unsigned long long* const ticket = reinterpret_cast<unsigned long long*>(out + SLOT * n_hits);
  uint64_t pn = 0, pe = 0;  // the warp's pool of hit numbers
  bool more = true;
  uint64_t cur = 0;
  uint32_t row = 0, steps = 0;
  bool have = false;
  for (;;) {
    const uint32_t wmask = __ballot_sync(FULL, !have && sub == 0);
    if (wmask != 0 && (pn != pe || more)) {
      const uint32_t n_want = __popc(wmask);
      if (pe - pn < n_want && more) {  // top the pool up (the few hits left in it are taken first)
        // (pool ranges are contiguous only within one ticket: drain the old one before drawing)
        if (pn == pe) {
          unsigned long long t = 0;
          if (lane == 0) t = atomicAdd(ticket, (unsigned long long)LEAN_TICKET);
          t = __shfl_sync(FULL, t, 0);
          more = t < n_hits;
          pn = more ? t : 0;
          pe = more ? (n_hits - t < LEAN_TICKET ? n_hits : t + LEAN_TICKET) : 0;
        }
      }
      const uint32_t r = __popc(wmask & ((1u << gbase) - 1u));
      if (!have && pn + r < pe) {
        cur = pn + r;
        row = uint32_t(out[SLOT * cur]);
        steps = 0;
        have = true;
      }
      pn = pn + n_want < pe ? pn + n_want : pe;
    }
    if (__all_sync(FULL, !have && pn == pe && !more)) break;
    const uint32_t blk = (row >> 5) / 7u;  // / 224
    const uint32_t l = row - blk * WALK_ROWS_PER_BLOCK;
    u32x8 x;
#pragma unroll
    for (int i = 0; i < 8; i++) x.v[i] = 0;
    AWRY_CHK(!have || uint64_t(blk) * WALK_BLOCK_UINT4 + 7 < ix.n_walk_u4);
    if (have) x = ldg256(ix.walk_blocks + size_t(blk) * WALK_BLOCK_UINT4 + 2 * sub);
    // the lane that holds the row's group reads its code and mark
    const uint32_t g = l >> 5, t = l & 31, half = g & 1;
    const uint32_t p0 = half ? x.v[4] : x.v[0], p1 = half ? x.v[5] : x.v[1], p2 = half ? x.v[6] : x.v[2],
                   mk = half ? x.v[7] : x.v[3];
    uint32_t cm = ((p0 >> t) & 1u) | (((p1 >> t) & 1u) << 1) | (((p2 >> t) & 1u) << 2) | (((mk >> t) & 1u) << 3);
    cm = __shfl_sync(FULL, cm, gbase + (g >> 1));
    const uint32_t c = cm & 7u;
    const bool marked = have && (cm & 8u);
    // rows of this lane's groups at or before the row: group 2*sub (words 0..3) and 2*sub+1 (words 4..7);
    // lane 3 holds group 6 only (its words 4..7 are the counts)
    const uint32_t ma = low_mask(int(l) + 1 - int(64 * sub)), mb = sub < 3 ? low_mask(int(l) + 1 - int(64 * sub + 32)) : 0u;
    uint32_t r = 0;
    if (have) {
      if (marked) {  // marks strictly before the row
        const uint32_t below_a = low_mask(int(l) - int(64 * sub)), below_b = sub < 3 ? low_mask(int(l) - int(64 * sub + 32)) : 0u;
        r = __popc(x.v[3] & below_a) + __popc(x.v[7] & below_b);
      } else if (c < 4) {
        const uint32_t m0 = (c & 1) ? ~0u : 0u, m1 = (c & 2) ? ~0u : 0u;
        r = __popc(~x.v[2] & ~(x.v[0] ^ m0) & ~(x.v[1] ^ m1) & ma) + __popc(~x.v[6] & ~(x.v[4] ^ m0) & ~(x.v[5] ^ m1) & mb);
        if (sub == 3) r += c == 0 ? x.v[4] : c == 1 ? x.v[5] : c == 2 ? x.v[6] : x.v[7];
      }
    }
    r += __shfl_xor_sync(FULL, r, 1);
    r += __shfl_xor_sync(FULL, r, 2);
    if (have) {
      if (marked) {
        if (sub == 0) {
          AWRY_CHK(blk < ix.n_walk_rank && uint64_t(__ldg(ix.walk_rank + blk)) + r < ix.n_pos_samples && steps < ix.lean_ratio);
          const uint64_t loc = uint64_t(__ldg(ix.pos_samples + __ldg(ix.walk_rank + blk) + r)) * ix.lean_ratio + steps;
          if (MAP)
            map_location(ix, loc, out + SLOT * cur);
          else
            out[cur] = loc;
        }
        have = false;
      } else {
        // (a '$' row is always marked -- text position 0 -- so c is A, C, G, T or N here)
        row = c < 4 ? ix.c_lo[c] + r - 1 : lf_backstep<0>(ix, row);
        steps++;
      }
    }
  }
}


// Locate pass 2 on the unsampled array: hit i of query q is SA[sp + i] -- no walk.  Same work split as
// expand_rows_kernel: a lane copies the first 8 hits of its query, longer intervals are copied by the
// whole warp (coalesced 128-B reads of SA, coalesced writes), so skewed hit counts cost bandwidth, not
// serial steps.
template <bool MAP>
__global__ void __launch_bounds__(256)
    gather_sa_kernel(IndexView ix, const uint2* __restrict__ sp_cnt, const uint64_t* __restrict__ hit_off,
                     uint64_t nq, uint64_t* __restrict__ out) {
  constexpr int SLOT = MAP ? 2 : 1;
  const uint32_t* __restrict__ full = ix.full_sa;
  const uint32_t lane = threadIdx.x & 31;
  const uint64_t warp = (blockIdx.x * uint64_t(blockDim.x) + threadIdx.x) >> 5;
  const uint64_t nwarps = (gridDim.x * uint64_t(blockDim.x)) >> 5;
  for (uint64_t base = warp * 32; base < nq; base += nwarps * 32) {
    uint64_t q = base + lane;
    uint32_t sp = 0, cnt = 0;
    uint64_t off = 0;
    if (q < nq) {
      uint2 r = sp_cnt[q];
      sp = r.x;
      cnt = r.y;
      off = hit_off[q];
    }
    const bool at_pos = cnt == CNT_AT_TEXT_POS;  // finished in the text by the search kernel: sp IS the position
    if (at_pos) cnt = 1;
    uint32_t small = cnt < 8 ? cnt : 8;
    for (uint32_t i = 0; i < small; i++) {
      AWRY_CHK(at_pos || uint64_t(sp) + i < ix.n_full_sa);
      uint64_t loc = at_pos ? uint64_t(sp) : uint64_t(__ldg(full + sp + i));
      if (MAP)
        map_location(ix, loc, out + SLOT * (off + i));
      else
        out[off + i] = loc;
    }
    uint32_t big = __ballot_sync(0xffffffffu, cnt > 8);
    while (big) {
      int L = __ffs(big) - 1;
      big &= big - 1;
      uint32_t s = __shfl_sync(0xffffffffu, sp, L), c = __shfl_sync(0xffffffffu, cnt, L);
      uint64_t o = __shfl_sync(0xffffffffu, off, L);
      for (uint32_t i = 8 + lane; i < c; i += 32) {
        AWRY_CHK(uint64_t(s) + i < ix.n_full_sa);
        uint64_t loc = __ldg(full + s + i);
        if (MAP)
          map_location(ix, loc, out + SLOT * (o + i));
        else
          out[o + i] = loc;
      }
    }
  }
}

// ---- locate pass 2 without a host round trip (awry_locate_batch_into on the unsampled array) ----
// The two-pass scheme needs the hit total of a chunk only to place its hits behind those of the chunks before
// it.  That running total lives on the device: advance_hit_base_kernel (one thread, ordered after the same
// kernel of the previous chunk by an event) hands the chunk its base and adds the chunk's total; the gather
// then writes every hit at base + local offset STRAIGHT INTO THE CALLER'S PINNED BUFFER (`out` is the device
// view of host memory: 16-byte stores, 512 contiguous bytes per warp for singleton queries) and the rebased
// CSR offsets into a device array that one copy returns.  Hits past `capacity` are dropped; the total still
// counts them (AWRY_ERR_CAPACITY).
__global__ void advance_hit_base_kernel(const uint64_t* __restrict__ local_off, uint64_t nq,
                                        unsigned long long* running, unsigned long long* chunk_base) {
  const unsigned long long b = *running;
  *chunk_base = b;
  *running = b + local_off[nq];
}

__global__ void __launch_bounds__(256)
    gather_sa_direct_kernel(IndexView ix, const uint2* __restrict__ sp_cnt, const uint64_t* __restrict__ local_off,
                            uint64_t nq, const unsigned long long* __restrict__ chunk_base,
                            ulonglong2* __restrict__ out, uint64_t capacity, uint64_t* __restrict__ off_out) {
  const uint32_t* __restrict__ full = ix.full_sa;
  const uint32_t lane = threadIdx.x & 31;
  const uint64_t warp = (blockIdx.x * uint64_t(blockDim.x) + threadIdx.x) >> 5;
  const uint64_t nwarps = (gridDim.x * uint64_t(blockDim.x)) >> 5;
  const uint64_t hbase = *chunk_base;
  for (uint64_t base = warp * 32; base < nq; base += nwarps * 32) {
    uint64_t q = base + lane;
    uint32_t sp = 0, cnt = 0;
    uint64_t off = 0;
    if (q < nq) {
      uint2 r = sp_cnt[q];
      sp = r.x;
      cnt = r.y;
      off = hbase + local_off[q];
      off_out[q] = off;
    }
    const bool at_pos = cnt == CNT_AT_TEXT_POS;  // finished in the text by the search kernel: sp IS the position
    if (at_pos) cnt = 1;
    uint32_t small = cnt < 8 ? cnt : 8;
    for (uint32_t i = 0; i < small; i++) {
      uint64_t pr[2];
      AWRY_CHK(at_pos || uint64_t(sp) + i < ix.n_full_sa);
      map_location(ix, at_pos ? uint64_t(sp) : uint64_t(__ldg(full + sp + i)), pr);
      if (off + i < capacity) out[off + i] = make_ulonglong2(pr[0], pr[1]);
    }
    uint32_t big = __ballot_sync(0xffffffffu, cnt > 8);
    while (big) {
      int L = __ffs(big) - 1;
      big &= big - 1;
      uint32_t s = __shfl_sync(0xffffffffu, sp, L), c = __shfl_sync(0xffffffffu, cnt, L);
      uint64_t o = __shfl_sync(0xffffffffu, off, L);
      for (uint32_t i = 8 + lane; i < c; i += 32) {
        uint64_t pr[2];
        AWRY_CHK(uint64_t(s) + i < ix.n_full_sa);
        map_location(ix, __ldg(full + s + i), pr);
        if (o + i < capacity) out[o + i] = make_ulonglong2(pr[0], pr[1]);
      }
    }
  }
}

cudaError_t launch_gather_direct(const IndexView& ix, const uint2* d_sp_cnt, const uint64_t* d_local_off, uint64_t nq,
                                 unsigned long long* d_running, unsigned long long* d_chunk_base, void* out_hits,
                                 uint64_t capacity, uint64_t* d_off_out, int sm_count, cudaEvent_t wait_before_advance,
                                 cudaEvent_t record_after_advance, cudaStream_t s) {
  if (nq == 0 || ix.full_sa == nullptr) return cudaErrorInvalidValue;
  cudaError_t e;
  if (wait_before_advance && (e = cudaStreamWaitEvent(s, wait_before_advance, 0)) != cudaSuccess) return e;
  advance_hit_base_kernel<<<1, 1, 0, s>>>(d_local_off, nq, d_running, d_chunk_base);
  COUNT_LAUNCH();
  if ((e = cudaGetLastError()) != cudaSuccess) return e;
  if (record_after_advance && (e = cudaEventRecord(record_after_advance, s)) != cudaSuccess) return e;
  unsigned grid = unsigned(std::max<uint64_t>(1, std::min<uint64_t>(uint64_t(sm_count) * 8, (nq + 255) / 256)));
  gather_sa_direct_kernel<<<grid, 256, 0, s>>>(ix, d_sp_cnt, d_local_off, nq, d_chunk_base,
                                               static_cast<ulonglong2*>(out_hits), capacity, d_off_out);
  COUNT_LAUNCH();
  return cudaGetLastError();
}

cudaError_t launch_walk(const IndexView& ix, const void* d_sp_cnt_v, const uint64_t* d_hit_off,
                        uint64_t nq, uint64_t n_hits, uint64_t* d_hits_pairs, uint64_t* d_locs,
                        int sm_count, cudaStream_t s) {
  if (n_hits == 0 || nq == 0) return cudaSuccess;
  if (ix.wide) return launch_walk_wide(*ix.wide, d_sp_cnt_v, d_hit_off, nq, n_hits, d_hits_pairs, d_locs, sm_count, s);
  const uint2* d_sp_cnt = static_cast<const uint2*>(d_sp_cnt_v);
  const bool map = d_hits_pairs != nullptr;
  uint64_t* out = map ? d_hits_pairs : d_locs;
  if (ix.full_sa != nullptr) {  // unsampled array present: a gather instead of expand + walk
    unsigned grid = unsigned(std::max<uint64_t>(1, std::min<uint64_t>(uint64_t(sm_count) * 8, (nq + 255) / 256)));
    if (map)
      gather_sa_kernel<true><<<grid, 256, 0, s>>>(ix, d_sp_cnt, d_hit_off, nq, out);
    else
      gather_sa_kernel<false><<<grid, 256, 0, s>>>(ix, d_sp_cnt, d_hit_off, nq, out);
    COUNT_LAUNCH();
    return cudaGetLastError();
  }
  {
    unsigned grid = unsigned(std::max<uint64_t>(1, std::min<uint64_t>(uint64_t(sm_count) * 8, (nq + 255) / 256)));
    expand_rows_kernel<<<grid, 256, 0, s>>>(d_sp_cnt, d_hit_off, nq, reinterpret_cast<uint32_t*>(out), map ? 4u : 2u);
    COUNT_LAUNCH();
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return e;
  }
  {  // ticket counter of the walk kernels: 8 bytes behind the output slots (the caller allocates +16)
    cudaError_t e = cudaMemsetAsync(out + (map ? 2 : 1) * n_hits, 0, 8, s);
    if (e != cudaSuccess) return e;
  }
  if (ix.alphabet == 0 && ix.walk_blocks != nullptr) {  // bounded walk on the position-sampled array
    unsigned grid = unsigned(std::max<uint64_t>(1, std::min<uint64_t>(uint64_t(sm_count) * 8, (4 * n_hits + 255) / 256)));
    if (map)
      walk_lean_kernel<true><<<grid, 256, 0, s>>>(ix, n_hits, out);
    else
      walk_lean_kernel<false><<<grid, 256, 0, s>>>(ix, n_hits, out);
  } else if (ix.alphabet == 0) {
    unsigned grid = unsigned(std::max<uint64_t>(1, std::min<uint64_t>(uint64_t(sm_count) * 8, (2 * n_hits + 255) / 256)));
    const bool dynamic = n_hits >= 64 * ((uint64_t(grid) * 256) >> 1);
    if (map)
      walk_dna_kernel<true><<<grid, 256, 0, s>>>(ix, n_hits, out, dynamic);
    else
      walk_dna_kernel<false><<<grid, 256, 0, s>>>(ix, n_hits, out, dynamic);
  } else {
    unsigned grid = unsigned(std::max<uint64_t>(1, std::min<uint64_t>(uint64_t(sm_count) * 8, (4 * n_hits + 255) / 256)));
    const bool dynamic = n_hits >= 64 * ((uint64_t(grid) * 256) >> 2);
    if (map)
      walk_amino_kernel<true><<<grid, 256, 0, s>>>(ix, n_hits, out, dynamic);
    else
      walk_amino_kernel<false><<<grid, 256, 0, s>>>(ix, n_hits, out, dynamic);
  }
  COUNT_LAUNCH();
  return cudaGetLastError();
}

// per-query ascending sort of global text positions (== (seq_idx, local_pos) order)
cudaError_t sort_hit_segments(uint64_t* d_locs_in, uint64_t* d_locs_out, uint64_t n_hits,
                              uint64_t nq, const uint64_t* d_hit_off, void* d_temp,
                              size_t& temp_bytes, cudaStream_t s) {
  cudaError_t e = cub::DeviceSegmentedSort::SortKeys(d_temp, temp_bytes, d_locs_in, d_locs_out,
                                                     (long long)n_hits, (long long)nq, d_hit_off,
                                                     d_hit_off + 1, s);
  if (d_temp != nullptr) COUNT_LAUNCH();
  return e;
}

__global__ void map_locations_kernel(IndexView ix, const uint64_t* __restrict__ locs, uint64_t n,
                                     uint64_t* __restrict__ out) {
  uint64_t stride = gridDim.x * uint64_t(blockDim.x);
  for (uint64_t i = blockIdx.x * uint64_t(blockDim.x) + threadIdx.x; i < n; i += stride)
    map_location(ix, locs[i], out + 2 * i);
}

cudaError_t launch_map_locations(const IndexView& ix, const uint64_t* d_locs, uint64_t n_hits,
                                 uint64_t* d_hits_pairs, cudaStream_t s) {
  if (n_hits == 0) return cudaSuccess;
  unsigned grid = unsigned(std::min<uint64_t>((n_hits + 255) / 256, 148 * 16));
  map_locations_kernel<<<grid, 256, 0, s>>>(ix, d_locs, n_hits, d_hits_pairs);
  COUNT_LAUNCH();
  return cudaGetLastError();
}

// ------------------------------------------------------------------ single steps

template <int ALPHA>
__global__ void single_update_kernel(IndexView ix, uint32_t sp, uint32_t ep, uint32_t c, uint64_t* out) {
  lf_update<ALPHA>(ix, sp, ep, c);
  out[0] = sp;
  out[1] = ep;
}
template <int ALPHA>
__global__ void single_backstep_kernel(IndexView ix, uint32_t row, uint64_t* out) {
  out[0] = lf_backstep<ALPHA>(ix, row);
}
cudaError_t launch_single_update(const IndexView& ix, uint64_t sp, uint64_t ep, uint32_t dsym,
                                 uint64_t* d_out2, cudaStream_t s) {
  if (ix.wide) return launch_single_update_wide(*ix.wide, sp, ep, dsym, d_out2, s);
  if (ix.alphabet == 0)
    single_update_kernel<0><<<1, 1, 0, s>>>(ix, uint32_t(sp), uint32_t(ep), dsym, d_out2);
  else
    single_update_kernel<1><<<1, 1, 0, s>>>(ix, uint32_t(sp), uint32_t(ep), dsym, d_out2);
  COUNT_LAUNCH();
  return cudaGetLastError();
}
cudaError_t launch_single_backstep(const IndexView& ix, uint64_t row, uint64_t* d_out, cudaStream_t s) {
  if (ix.wide) return launch_single_backstep_wide(*ix.wide, row, d_out, s);
  if (ix.alphabet == 0)
    single_backstep_kernel<0><<<1, 1, 0, s>>>(ix, uint32_t(row), d_out);
  else
    single_backstep_kernel<1><<<1, 1, 0, s>>>(ix, uint32_t(row), d_out);
  COUNT_LAUNCH();
  return cudaGetLastError();
}

}  // namespace awry
