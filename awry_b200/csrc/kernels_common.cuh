// kernels_common.cuh -- device helpers shared by the kernel translation units (kernels.cu: load-time
// re-layout, seed table, pair index, query packing, backward search; kernels_locate.cu: locate pass 2, the
// unsampled suffix array, single steps; kernels_probe.cu: the random-gather roofline probe).
#pragma once
#include <atomic>

#include "kernels.hpp"

namespace awry {

extern std::atomic<uint64_t> g_launches;  // kernels launched by this library (awry_profile_get)
#define COUNT_LAUNCH() ::awry::g_launches.fetch_add(1, std::memory_order_relaxed)

// ---- shared by the search kernels (kernels.cu, kernels_wide.cu) ----

template <int MODE>
__device__ __forceinline__ void store_result(void* out, uint64_t q, uint32_t sp, uint32_t ep) {
  bool empty = sp > ep;
  if (MODE == OUT_COUNT_U64) {
    reinterpret_cast<uint64_t*>(out)[q] = empty ? 0ull : uint64_t(ep - sp) + 1ull;  // search.rs:66-71
  } else if (MODE == OUT_RANGE_U64) {
    reinterpret_cast<ulonglong2*>(out)[q] = empty ? make_ulonglong2(1, 0) : make_ulonglong2(sp, ep);
  } else {
    reinterpret_cast<uint2*>(out)[q] = empty ? make_uint2(1u, 0u) : make_uint2(sp, ep - sp + 1u);
  }
}

// Length of query (o0, o1) of a batch whose bytes span [b.lo, b.hi]; 0 for a query the prepass refused
// (offsets outside the range: its packed words were never written) -- it is stored as an empty result and the
// call fails with the prepass's error.
struct ByteRange {
  uint64_t lo, hi;
};
// checked build: a 32-byte read of packed query words at absolute word index w (the buffer pointer is biased
// by the batch's first byte) stays inside the packed_words() the batch was given
#define AWRY_CHK_QWORDS(w, br, nq, shift) \
  AWRY_CHK(uint64_t(w) >= 4 * ((br).lo >> (shift)) && uint64_t(w) - 4 * ((br).lo >> (shift)) + 3 < 4 * ((nq) + (((br).hi - (br).lo) >> (shift)) + 2) + 32)
__device__ __forceinline__ uint32_t checked_len(uint64_t o0, uint64_t o1, const ByteRange& b) {
  return (o0 < b.lo || o1 > b.hi || o1 < o0 || o1 - o0 >= (1ull << 32)) ? 0u : uint32_t(o1 - o0);
}

// Packed-symbol reader: current word in a register, the next one prefetched.  Word positions are
// 32-bit indices into the packed buffer (a launch never packs more than 2^32 words = 32 GiB).
template <int ALPHA>
struct QueryStream {
  static constexpr int BITS = ALPHA == 0 ? 4 : 8;
  static constexpr int SPW = 64 / BITS;
  static constexpr int UNIT_SHIFT = ALPHA == 0 ? 6 : 5;
  uint64_t w, wnext;
  uint32_t widx;    // index of the word held in wnext
  uint32_t inword;
  __device__ __forceinline__ void open(const uint64_t* __restrict__ qwords, uint32_t q, uint64_t o0) {
    widx = 4 * (q + uint32_t(o0 >> UNIT_SHIFT)) + 1;
    w = __ldg(qwords + (widx - 1));
    wnext = __ldg(qwords + widx);  // buffer is padded
    inword = 0;
  }
  __device__ __forceinline__ uint32_t next(const uint64_t* __restrict__ qwords) {
    uint32_t c = uint32_t(w) & ((1u << BITS) - 1u);
    w >>= BITS;
    if (++inword == SPW) {
      w = wnext;
      widx++;
      wnext = __ldg(qwords + widx);
      inword = 0;
    }
    return c;
  }
};

// ---- a lane's share of a 64-B nucleotide block: LANES lanes cooperate on one block ----
template <int LANES>
struct LaneChunks;
template <>
struct LaneChunks<4> {
  uint4 c[1];
  __device__ __forceinline__ void load(const uint4* blk, uint32_t sub) { c[0] = ldg128(blk + sub); }
};
template <>
struct LaneChunks<2> {
  uint4 c[2];
  __device__ __forceinline__ void load(const uint4* blk, uint32_t sub) {
    u32x8 v = ldg256(blk + 2 * sub);
    c[0] = make_uint4(v.v[0], v.v[1], v.v[2], v.v[3]);
    c[1] = make_uint4(v.v[4], v.v[5], v.v[6], v.v[7]);
  }
};
template <>
struct LaneChunks<1> {
  uint4 c[4];
  __device__ __forceinline__ void load(const uint4* blk, uint32_t) {
    u32x8 v = ldg256(blk);
    u32x8 u = ldg256(blk + 2);
    c[0] = make_uint4(v.v[0], v.v[1], v.v[2], v.v[3]);
    c[1] = make_uint4(v.v[4], v.v[5], v.v[6], v.v[7]);
    c[2] = make_uint4(u.v[0], u.v[1], u.v[2], u.v[3]);
    c[3] = make_uint4(u.v[4], u.v[5], u.v[6], u.v[7]);
  }
};

template <int LANES>
__device__ __forceinline__ uint32_t dna_partial_rank(const LaneChunks<LANES>& x, uint32_t sub,
                                                     uint32_t local, uint32_t c, uint32_t m0,
                                                     uint32_t m1) {
  constexpr int CH = 4 / LANES;
  uint32_t r = 0;
#pragma unroll
  for (int i = 0; i < CH; i++) {
    uint32_t j = sub * CH + i;
    uint32_t pred = ~x.c[i].z & ~(x.c[i].x ^ m0) & ~(x.c[i].y ^ m1);
    r += __popc(pred & chunk_mask(local, j));
    r += (j == c) ? x.c[i].w : 0u;
  }
  return r;
}


// Seed-table index of the first k <= 16 symbols of a packed nucleotide word: the low 2 bits of nibbles 0 .. k-1,
// squeezed together (symbol j at bits 2j).  Four mask-and-shift rounds per 32-bit half instead of a k-trip loop,
// which was 17 % of the count kernel's instructions once a 150-bp read took ~8 loads instead of ~70.
__device__ __forceinline__ uint32_t squeeze8(uint32_t x) {  // 8 nibbles -> 8 crumbs (16 bits)
  x &= 0x33333333u;
  x = (x | (x >> 2)) & 0x0F0F0F0Fu;
  x = (x | (x >> 4)) & 0x00FF00FFu;
  x = (x | (x >> 8)) & 0x0000FFFFu;
  return x;
}
__device__ __forceinline__ uint64_t kmer_index(uint64_t w, uint32_t k) {
  const uint32_t v = squeeze8(uint32_t(w)) | (squeeze8(uint32_t(w >> 32)) << 16);
  return k >= 16 ? uint64_t(v) : uint64_t(v & ((1u << (2 * k)) - 1u));
}

// low `n` bits set, n clamped to [0, 32] (BMSK)
__device__ __forceinline__ uint32_t low_mask(int n) {
  uint32_t m, len = uint32_t(n < 0 ? 0 : n);
  asm("bmsk.clamp.b32 %0, %1, %2;" : "=r"(m) : "r"(0u), "r"(len));
  return m;
}


// ---- "finish in the text" (layout.cuh: IndexView::rtext): one 32-byte sector of the reversed text (64 symbols,
// 8 per word) against the packed query in the group's shared-memory ring.  `rb0` = reversed-text index of
// search-order symbol 0, so the sector's first symbol has search-order index j0 = 64 * sec - rb0 (negative for
// the sector the window starts in); symbols [done, len) take part.  Returns non-zero on a mismatch.
// The ring is read as 32 words of 8 symbols; words outside the loaded part are masked out, not avoided.
// RING = false: the query is longer than the ring (256 symbols) and `ring` points at its packed words in global
// memory instead (read through L2: the words were fetched when the query started).
template <bool RING = true>
__device__ __forceinline__ uint32_t text_sector_mismatch(const u32x8& t, const uint64_t* ring, uint32_t sec, uint32_t rb0,
                                                         uint32_t done, uint32_t len) {
  const uint32_t* rq = reinterpret_cast<const uint32_t*>(ring);
  const int j0 = int(sec * 64u - rb0);
  const int a = j0 >> 3;  // floor
  const uint32_t sh = 4u * uint32_t(j0 & 7);
  // (global memory: the words in front of the query belong to no symbol that takes part -- they are masked out --
  // so word 0 stands in for them; behind the last query the buffer is padded by 32 words)
  uint32_t bad = 0, q_lo = RING ? rq[a & 31] : __ldg(rq + (a < 0 ? 0 : a));
#pragma unroll
  for (int w = 0; w < 8; w++) {
    const uint32_t q_hi = RING ? rq[(a + w + 1) & 31] : __ldg(rq + (a + w + 1 < 0 ? 0 : a + w + 1));
    const uint32_t qw = __funnelshift_r(q_lo, q_hi, sh);  // query symbols j0 + 8 w .. + 7
    const int jw = j0 + 8 * w;
    const uint32_t m = low_mask(4 * (int(len) - jw)) & ~low_mask(4 * (int(done) - jw));
    bad |= (qw ^ t.v[w]) & m;
    q_lo = q_hi;
  }
  return bad;
}

// Hamming search (kernels_hamming.cu): the same comparison, COUNTING mismatched symbols per piece of the read
// instead of testing for any.  `rq` = the read's packed words in global memory (search order, 8 symbols per u32;
// reads of any length, through L1/L2), rb0 = reversed-text index of its search-order symbol 0, cut[0 .. P] =
// ascending search-order piece bounds (piece t = symbols [cut[t], cut[t+1]), cut[0] = 0, cut[P] = read length).
// A word's mismatches are the nibbles of q ^ t with any bit set: popc((x | x>>1 | x>>2 | x>>3) & 0x11111111).
// Adds the mismatches of this 64-symbol sector to mm[t].
template <int P>
__device__ __forceinline__ void text_sector_mismatches(const u32x8& t, const uint32_t* rq, uint32_t sec, uint32_t rb0,
                                                       const int (&cut)[P + 1], uint32_t (&mm)[P]) {
  const int j0 = int(sec * 64u - rb0);
  const int a = j0 >> 3;  // floor
  const uint32_t sh = 4u * uint32_t(j0 & 7);
  // (words in front of the read hold no symbol that takes part -- masked out -- so word 0 stands in for them)
  uint32_t q_lo = __ldg(rq + (a < 0 ? 0 : a));
#pragma unroll
  for (int w = 0; w < 8; w++) {
    const uint32_t q_hi = __ldg(rq + (a + w + 1 < 0 ? 0 : a + w + 1));
    const uint32_t x = __funnelshift_r(q_lo, q_hi, sh) ^ t.v[w];  // read symbols j0 + 8 w .. + 7 against the text
    const uint32_t diff = (x | (x >> 1) | (x >> 2) | (x >> 3)) & 0x11111111u;
    const int jw = j0 + 8 * w;
#pragma unroll
    for (int p = 0; p < P; p++) mm[p] += __popc(diff & low_mask(4 * (cut[p + 1] - jw)) & ~low_mask(4 * (cut[p] - jw)));
    q_lo = q_hi;
  }
}

// ---- word readers of the edit-distance verification (kernels_edit.cu) and the alignment (kernels_align.cu)
// 8 symbols of the reversed text from nibble index x on (symbol t in nibble t); indices outside [0, bwt_len) read as
// 0xF, a code no read symbol has (as '$' at index 0, it is a text symbol nothing matches)
__device__ __forceinline__ uint32_t rtext8(const IndexView& ix, int64_t x) {
  const int64_t w = x >> 3;  // floor
  const uint32_t sh = 4u * uint32_t(x & 7);
  const uint64_t nw = ix.n_rtext / 4;
  const uint32_t* const rt = reinterpret_cast<const uint32_t*>(ix.rtext);
  const uint32_t lo = (w >= 0 && uint64_t(w) < nw) ? __ldg(rt + w) : 0xffffffffu;
  const uint32_t hi = (w + 1 >= 0 && uint64_t(w + 1) < nw) ? __ldg(rt + w + 1) : 0xffffffffu;
  uint32_t v = sh ? __funnelshift_r(lo, hi, sh) : lo;
  if (x < 0 || x + 8 > int64_t(ix.bwt_len)) {
#pragma unroll
    for (int t = 0; t < 8; t++)
      if (x + t < 0 || x + t >= int64_t(ix.bwt_len)) v |= 0xfu << (4 * t);
  }
  return v;
}

// 8 symbols of a packed read (search order, 8 per u32) from symbol y on; the buffer is padded behind every read
__device__ __forceinline__ uint32_t read8(const uint32_t* rq, uint32_t y) {
  const uint32_t w = y >> 3, sh = 4u * (y & 7);
  const uint32_t lo = __ldg(rq + w);
  return sh ? __funnelshift_r(lo, __ldg(rq + w + 1), sh) : lo;
}

// the descending reader: the 8 search-order symbols y, y - 1, .. y - 7 of a packed read with symbol y - t in nibble
// 7 - t (those below symbol 0 are garbage).  Search order runs backwards through the read, so these are 8 read
// symbols in their ORIGINAL order from the top nibble down; rtext8(ix, x - 7) is the same for the text from x on.
__device__ __forceinline__ uint32_t desc8(const uint32_t* rq, uint32_t y) {
  return y >= 7 ? read8(rq, y - 7) : read8(rq, 0) << (4 * (7 - y));
}

// protein: 8 bits per symbol, so a 32-byte sector holds 32 symbols, 4 per word, and the ring 128
__device__ __forceinline__ uint32_t text_sector_mismatch8(const u32x8& t, const uint64_t* ring, uint32_t sec, uint32_t rb0,
                                                          uint32_t done, uint32_t len) {
  const uint32_t* rq = reinterpret_cast<const uint32_t*>(ring);
  const int j0 = int(sec * 32u - rb0);
  const int a = j0 >> 2;  // floor
  const uint32_t sh = 8u * uint32_t(j0 & 3);
  uint32_t bad = 0, q_lo = rq[a & 31];
#pragma unroll
  for (int w = 0; w < 8; w++) {
    const uint32_t q_hi = rq[(a + w + 1) & 31];
    const uint32_t qw = __funnelshift_r(q_lo, q_hi, sh);  // query symbols j0 + 4 w .. + 3
    const int jw = j0 + 4 * w;
    const uint32_t m = low_mask(8 * (int(len) - jw)) & ~low_mask(8 * (int(done) - jw));
    bad |= (qw ^ t.v[w]) & m;
    q_lo = q_hi;
  }
  return bad;
}

// ---- a lane's share of a 128-B amino block (4 lanes): matching rows of its 32-row slice and, in the
// lane that holds it, the block-start count of the symbol ----
struct AminoSlice {
  uint32_t match, count;
};
__device__ __forceinline__ AminoSlice amino_slice(const u32x8& x, uint32_t sub, uint32_t sym) {
  AminoSlice r;
  r.match = sub < 2 ? amino_match(x, sym) : 0u;
  const uint32_t cw = amino_count_word(sym);  // word index in the block: lane = cw / 8, word = cw % 8
  const uint32_t word = cw & 7u;
  const uint32_t t0 = (word & 1) ? x.v[1] : x.v[0], t1 = (word & 1) ? x.v[3] : x.v[2];
  const uint32_t t2 = (word & 1) ? x.v[5] : x.v[4], t3 = (word & 1) ? x.v[7] : x.v[6];
  const uint32_t u0 = (word & 2) ? t1 : t0, u1 = (word & 2) ? t3 : t2;
  r.count = sub == (cw >> 3) ? ((word & 4) ? u1 : u0) : 0u;
  return r;
}

// get_seq_location, intended semantics (sequence_index.rs:108-141; SURVEY.md Q4)
__device__ __forceinline__ void map_location(const IndexView& ix, uint64_t loc, uint64_t* out2) {
  uint32_t lo = 0;
  if (ix.n_seqs > 1) {
    uint32_t hi = ix.n_seqs - 1;
    while (lo < hi) {
      uint32_t mid = (lo + hi + 1) >> 1;
      if (__ldg(ix.seq_starts + mid) <= loc)
        lo = mid;
      else
        hi = mid - 1;
    }
  }
  AWRY_CHK(lo < ix.n_seqs && loc >= __ldg(ix.seq_starts + lo));
  out2[0] = lo;
  out2[1] = loc - __ldg(ix.seq_starts + lo);
}

// VERIFY_PLACE_BEST (read mapping, DESIGN.md §1h): a hit at distance d of a read whose best distance is b (0xff: none)
// is placed iff d <= min(b + 1, k)
__device__ __forceinline__ bool within_map_bound(uint32_t d, uint32_t b, uint32_t k) { return b != 0xffu && d <= min(b + 1u, k); }

}  // namespace awry
