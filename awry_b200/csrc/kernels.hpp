// kernels.hpp -- host-callable launchers of the sm_100a kernels (internal to libawry_b200).
#pragma once
#include <algorithm>
#include <cstdint>
#include <cuda_runtime.h>

#include "layout.cuh"

namespace awry {

// packed query stream: DNA 4 bits / symbol (16 per u64), amino 8 bits / symbol (8 per u64);
// symbols are stored in SEARCH order (last query character first).  Every query starts on a
// 32-byte boundary so a lane group can stage it with aligned LDG.256: query q starts at word
// 4 * (q + (qoff[q] >> 6))  (DNA; amino: >> 5) -- monotone and overlap-free without a scan.
inline uint64_t packed_words(int alphabet, uint64_t nq, uint64_t total_bytes) {
  return 4 * (nq + (total_bytes >> (alphabet == 0 ? 6 : 5)) + 2) + 32;
}
inline int packed_unit_shift(int alphabet) { return alphabet == 0 ? 6 : 5; }

enum SearchOut { OUT_COUNT_U64 = 0, OUT_RANGE_U64 = 1, OUT_SP_CNT_U32 = 2 };
// OUT_SP_CNT_U32 with SearchVariant::locate_positions: count field of a query that was finished in the text -- it has ONE
// hit and the first field is its text position, not a BWT row (a real count is at most bwt_len - 1 < 2^32 - 257)
constexpr uint32_t CNT_AT_TEXT_POS = 0xffffffffu;

struct SearchVariant {
  int lanes = 0;          // nucleotide: 1, 2, 4 lanes per query on the 1-step blocks; 8 = pair-index
                          // kernel (default when the pair index exists); -1 = scalar kernel
  int tpb = 0;            // threads per block
  int blocks_per_sm = 0;  // 0 = occupancy-derived
  int slots = -1;         // pair kernel: 0 = search_dna_pair_kernel; 1 / 2 = search_dna_pairx_kernel with that many
                          // query slots per lane group; -1 = default (AWRY_B200_SLOTS, else the measured winner)
  bool finish_in_text = true;  // count mode, pair kernel: finish one-row intervals by comparing with the text
                               // (IndexView::rtext) instead of stepping on (awry_set_count_variant)
  bool locate_positions = false;  // OUT_SP_CNT_U32, pair kernel: a query finished in the text is stored as (text position,
                                  // CNT_AT_TEXT_POS) -- only for callers whose pass 2 is the gather from the unsampled array
  uint32_t avg_len = 0;   // mean query length of the batch (0 = unknown): sizes the tickets of the dynamic hand-out
  uint64_t b_lo = 0, b_hi = ~0ull;  // byte range of the batch's queries: offsets outside it are refused (see launch_pack)
};

// Queries per ticket of the per-GROUP dynamic hand-out (amino kernel).  Small tickets shorten the tail (a
// lane group needs ~130 us per 150-bp read: 64 / 16 / 4 / 1 reads per ticket gave 20.2 / 17.6 / 16.5 /
// 16.3 ms per 10 M reads in the pair kernel), but every ticket is an atomic on ONE counter and same-address
// atomics retire at ~0.5 G/s, so one query per ticket collapses once the groups of a warp drift apart
// (profiles/r01_s42_ticket_vs_mismatches.log); the pair kernel hands out per warp instead.
inline uint32_t ticket_size(uint32_t avg_len) {
  if (avg_len == 0) return 4;
  uint32_t t = 600 / avg_len;
  return t < 2 ? 2u : t > 16 ? 16u : t;
}

// ... and never so large that a lane group draws fewer than ~6 tickets over the batch: the kernel ends when the
// last ticket does, so with ~1 ticket per group it runs for up to two ticket times (small pipeline chunks).
// Very short queries keep a floor (50 / length queries per group): their tickets are cheap to finish and every
// ticket is an atomic on one counter.
inline uint32_t ticket_cap(uint32_t per_group, uint64_t nq, uint64_t n_groups, uint32_t avg_len) {
  const uint64_t cap = nq / (6 * (n_groups ? n_groups : 1));
  const uint64_t floor_ = avg_len ? std::max<uint32_t>(1, 50u / avg_len) : 1;
  return uint32_t(std::min<uint64_t>(per_group, std::max<uint64_t>(floor_, cap)));
}

struct LaunchCounters {
  uint64_t launches = 0;
};

cudaError_t init_device_tables();  // per device, once: ASCII -> device-symbol LUTs

// reference-layout blocks (staged on the device) -> device layout
// d_sb: nullptr, or (wide indexes) the superblock table [superblock][SB_STRIDE] the block counts are made
// relative to; sb_shift = log2(rows per superblock)
cudaError_t launch_transpose(int alphabet, const uint64_t* d_ref_blocks, uint64_t first_ref_block,
                             uint64_t n_ref_blocks, uint64_t bwt_len, uint4* d_blocks,
                             unsigned long long* d_dollar_row, const uint64_t* d_sb, uint32_t sb_shift, cudaStream_t s);
// wide indexes: absolute counts of the superblocks whose first reference block lies in [first, first + n)
// of a reference-layout block array on the device -> d_sb
cudaError_t launch_gather_superblocks(int alphabet, const uint64_t* d_ref_blocks, uint64_t first_ref_block,
                                      uint64_t n_ref_blocks, uint32_t sb_shift, uint64_t* d_sb, cudaStream_t s);
// the inverse (FmIndex::save of a handle that only holds the device layout): device blocks -> reference
// blocks [first_ref_block, first_ref_block + n_ref_blocks) written to d_ref_blocks[0 ..)
cudaError_t launch_untranspose(int alphabet, const uint4* d_blocks, uint64_t dollar_row, uint64_t first_ref_block,
                               uint64_t n_ref_blocks, uint64_t* d_ref_blocks, const uint64_t* d_sb, uint32_t sb_shift,
                               cudaStream_t s);
uint64_t table_entries(int alphabet, uint32_t k);
cudaError_t launch_build_table(const IndexView& ix, uint2* d_table, uint32_t k, cudaStream_t s);

// the reference's own (incomplete) k-mer table, for files written by awry_build_index_file
cudaError_t launch_ref_table(const IndexView& ix, uint64_t first, uint64_t count, uint32_t k, void* d_out,
                             cudaStream_t s);

// nucleotide pair index (two symbols per access), built from the 1-step device blocks
uint64_t pair_block_count(uint64_t bwt_len);
cudaError_t build_pair_index(const IndexView& ix, uint4* d_pair_blocks, uint32_t* c2_host /*16*/, cudaStream_t s);

// unsampled suffix array (locate accelerator): SA[row] for every row, 4 B each, from the sampled one
// d_qoff[i] = first + i * len for i in [0, n]: the offsets of a chunk of equally long queries, written on the
// device instead of copied to it
cudaError_t launch_fill_offsets(uint64_t* d_qoff, uint64_t first, uint64_t len, uint64_t n, cudaStream_t s);
cudaError_t build_full_sa(const IndexView& ix, uint32_t* d_full, int sm_count, cudaStream_t s);
// The indexed text, reversed, 4 bits per symbol (IndexView::rtext, layout.cuh), from the blocks and ix.full_sa:
// text[SA[row] - 1] = BWT[row].  Protein: one byte per symbol (the reference symbol index).  d_rtext: rtext_bytes() bytes.
inline size_t rtext_bytes(int alphabet, uint64_t bwt_len) {
  return ((alphabet == 0 ? (size_t(bwt_len) + 1) / 2 : size_t(bwt_len)) + 127) / 128 * 128 + 128;
}
cudaError_t build_rtext(const IndexView& ix, uint8_t* d_rtext, cudaStream_t s);

// The prepass latches the first query it refuses in *d_first_bad (atomicMin, ~0 = none) as
// bad_query_code(q, kind): an empty / sentinel-carrying query (the reference panics, fm_index.rs:406,
// bwt.rs:127), or a query whose offsets leave the batch's byte range [b_lo, b_hi] (offsets not monotone):
// such a query is never loaded or stored.
enum BadKind : unsigned { BAD_QUERY = 0, BAD_OFFSETS = 1 };
__host__ __device__ inline unsigned long long bad_query_code(uint64_t q, unsigned kind) { return (q << 1) | kind; }
// memory-lean bounded locate (nucleotide): walk blocks (planes + position marks), their mark ranks and the
// position-sampled suffix array, all derived from the 1-step blocks and the file's row-sampled array
uint64_t walk_block_count(uint64_t bwt_len);
cudaError_t build_lean_sa(const IndexView& ix, uint4* d_walk, uint32_t* d_rank, uint32_t* d_pos, int sm_count,
                          cudaStream_t s);

cudaError_t launch_pack(int alphabet, const uint8_t* d_qbytes, const uint64_t* d_qoff, uint64_t nq,
                        uint64_t* d_qwords, uint64_t b_lo, uint64_t b_hi, unsigned long long* d_first_bad,
                        cudaStream_t s);
// nucleotide queries packed to 2 bits (by hostpack.hpp, or by the caller: awry_*_batch_packed2): crumbs of
// the query bytes from absolute query offset `base` on, plus the exception list for bytes outside ACGT,
// entries ((position - exc_base) << 8) | byte
cudaError_t launch_pack2(const uint32_t* d_crumbs, uint64_t base, const uint64_t* d_qoff, uint64_t nq, uint64_t* d_qwords,
                         const uint64_t* d_exc, uint64_t n_exc, uint64_t exc_base, uint64_t b_lo, uint64_t b_hi,
                         unsigned long long* d_first_bad, cudaStream_t s);
// d_defer: defer_words(nq) u32 of scratch -- [0] count and [1 .. nq] list of the queries the cooperative kernel hands to
// the scalar kernel, [nq + 1] ticket counter; [nq + 2] count, [nq + 3] ticket counter and [nq + 4 ..] list of the queries
// the wave kernel hands to the refilling kernel
inline size_t defer_words(uint64_t nq) { return 2 * size_t(nq) + 8; }
cudaError_t launch_search(const IndexView& ix, const uint64_t* d_qwords, const uint64_t* d_qoff,
                          uint64_t nq, SearchOut mode, void* d_out, uint32_t* d_defer,
                          const SearchVariant& v, int sm_count, cudaStream_t s);
// ASCII queries searched by the wave kernel straight from their bytes: it packs them itself (the ring of every read it
// searches, and in d_qwords the words of the queries it hands on to the list kernels) and latches in *d_first_bad what
// launch_pack would.  search_packs_ascii: whether launch_search would run the wave kernel for this batch (and
// AWRY_B200_ASCII_WAVE, read per call, is not "0"); only then may launch_search_ascii be called -- otherwise the
// queries go through launch_pack + launch_search.
bool search_packs_ascii(const IndexView& ix, SearchOut mode, const SearchVariant& v);
cudaError_t launch_search_ascii(const IndexView& ix, const uint8_t* d_qbytes, const uint64_t* d_qoff, uint64_t nq,
                                uint64_t* d_qwords, unsigned long long* d_first_bad, SearchOut mode, void* d_out,
                                uint32_t* d_defer, const SearchVariant& v, int sm_count, cudaStream_t s,
                                bool strands = false);

// ---- both strands (awry_*_strands): read q of a batch stands for the VIRTUAL queries 2q (the read) and 2q + 1 (its
// reverse complement), which every search and locate kernel runs like any other queries.
// d_voff[2q] = 2 qoff[q], d_voff[2q + 1] = qoff[q] + qoff[q + 1] (2 nq + 1 entries, within [2 b_lo, 2 b_hi]): both
// virtual queries have the read's length and their own word slot.  A read whose offsets leave [b_lo, b_hi] gets
// d_voff[2q + 1] = ~0, which refuses both of its virtual queries (and no other).
cudaError_t launch_strand_offsets(const uint64_t* d_qoff, uint64_t nq, uint64_t b_lo, uint64_t b_hi, uint64_t* d_voff,
                                  cudaStream_t s);
// the words of the virtual queries from those of the reads (any prepass: launch_pack, launch_pack2): v = 2q a copy,
// v = 2q + 1 the reverse complement (nibble order reversed, codes below 4 XOR 3).  d_qwords is biased for the reads'
// range [b_lo, b_hi], d_vwords for the virtual one; a read the prepass refused (or an empty one) is skipped.
cudaError_t launch_strand_words(const uint64_t* d_qwords, const uint64_t* d_qoff, uint64_t nq, uint64_t b_lo, uint64_t b_hi,
                                const uint64_t* d_voff, uint64_t* d_vwords, cudaStream_t s);
// whether the strand flavour of the ASCII wave kernel may search the virtual queries straight from the reads' bytes
// (launch_search_ascii with strands = true, d_qoff = the virtual offsets, v.b_lo / b_hi their range): where
// search_packs_ascii holds and AWRY_B200_STRAND_WAVE, read per call, is not "0"
bool search_strands_ascii(const IndexView& ix, SearchOut mode, const SearchVariant& v);

// locate: CSR offsets from pass 1, LF-walk pass 2
// d_sp_cnt: the search kernels' OUT_SP_CNT result -- uint2 (sp, count) per query, ulonglong2 for a wide index
cudaError_t scan_hit_offsets(const IndexView& ix, const void* d_sp_cnt, uint64_t nq, uint64_t* d_hit_off, void* d_temp,
                             size_t& temp_bytes, cudaStream_t s);
inline size_t sp_cnt_bytes(const IndexView& ix) { return ix.wide ? 16 : 8; }
// writes either awry_hit {seq_idx, local_pos} (d_hits) or global text positions (d_locs); when
// ix.full_sa is set the walk is replaced by a gather from the unsampled array.  The output buffer must
// have 16 spare bytes behind its n_hits slots (the walk kernels' ticket counter).
cudaError_t launch_walk(const IndexView& ix, const void* d_sp_cnt, const uint64_t* d_hit_off,
                        uint64_t nq, uint64_t n_hits, uint64_t* d_hits_pairs, uint64_t* d_locs,
                        int sm_count, cudaStream_t s);
// sync-free pass 2 on the unsampled array (see kernels_locate.cu): hits go straight to `out_hits` (device view
// of the caller's pinned awry_hit buffer) at *d_running + local offset, rebased offsets to d_off_out
cudaError_t launch_gather_direct(const IndexView& ix, const uint2* d_sp_cnt, const uint64_t* d_local_off, uint64_t nq,
                                 unsigned long long* d_running, unsigned long long* d_chunk_base, void* out_hits,
                                 uint64_t capacity, uint64_t* d_off_out, int sm_count, cudaEvent_t wait_before_advance,
                                 cudaEvent_t record_after_advance, cudaStream_t s);
cudaError_t sort_hit_segments(uint64_t* d_locs_in, uint64_t* d_locs_out, uint64_t n_hits,
                              uint64_t nq, const uint64_t* d_hit_off, void* d_temp,
                              size_t& temp_bytes, cudaStream_t s);
cudaError_t launch_map_locations(const IndexView& ix, const uint64_t* d_locs, uint64_t n_hits,
                                 uint64_t* d_hits_pairs, cudaStream_t s);

// ---- kernels_hamming.cu: Hamming search (<= k substitutions) by k + 1 exactly searched pieces per read
// piece offsets (k+1) nq + 1 of a batch; a query with L <= k is latched in *d_first_bad as BAD_QUERY of query q >> shift
cudaError_t launch_hamming_pieces(const uint64_t* d_qoff, uint64_t nq, uint32_t k, uint64_t b_lo, uint64_t b_hi,
                                  uint32_t shift, uint64_t* d_poff, unsigned long long* d_first_bad, cudaStream_t s);
// the words of the (k+1) nq pieces from the words of their queries (any prepass, or launch_strand_words), bit for bit
// what launch_pack writes for the pieces' bytes.  d_qwords is biased for [b_lo, b_hi] as for launch_search, d_pwords
// likewise with the piece offsets of launch_hamming_pieces; a query refused by its prepass (or empty) is skipped.
cudaError_t launch_hamming_piece_words(const uint64_t* d_qwords, const uint64_t* d_qoff, uint64_t nq, uint64_t b_lo,
                                       uint64_t b_hi, uint32_t k, uint64_t* d_pwords, cudaStream_t s);
// piece of every candidate of the slice [c0, c0 + n) (cub convention: d_temp == nullptr sizes the scratch)
cudaError_t launch_hamming_map(const uint64_t* d_hoff, uint64_t npieces, uint64_t c0, uint64_t n, uint32_t* d_map,
                               void* d_temp, size_t& temp_bytes, cudaStream_t s);
// what the verification kernels do with an accepted candidate: COUNT adds it to counts, PLACE writes its key into
// its query's range of a CSR computed by a COUNT pass over the same candidates (locate, DESIGN.md §1e).  PLACE_BEST
// (read mapping, DESIGN.md §1h) places only the keys within the bound of HammingSlice::best, into a CSR counted under
// the same bound.
enum VerifyMode { VERIFY_COUNT = 0, VERIFY_PLACE = 1, VERIFY_PLACE_BEST = 2 };
// one slice of candidates for the verification kernel
struct HammingSlice {
  const uint64_t* qwords;       // packed reads, biased as for launch_search: read q at word 4 (q + (qoff[q] >> 6))
  uint64_t qw_lo, qw_n;         // the words that exist: [qw_lo, qw_lo + qw_n) (checked build)
  const uint64_t* qoff;         // the reads' offsets (nq + 1), absolute within [b_lo, b_hi]
  uint64_t b_lo, b_hi;
  const uint2* sp_cnt;          // exact search result of every piece (OUT_SP_CNT_U32)
  const uint64_t* hoff;         // candidate offsets of every piece (npieces + 1)
  uint64_t npieces;
  const uint32_t* map;          // piece of candidate c0 + i
  uint64_t c0, n;
  union {
    uint64_t* counts;           // count: (k+1) per read, zeroed by the caller
    const uint64_t* hit_off;    // place: read q's keys go to keys[hit_off[q] .. hit_off[q + 1])
  };
  uint64_t* keys;               // place: the keys (s << 2 | d) of the batch
  uint64_t* acc;                // place: keys placed so far per read of the batch (the cursor), zeroed by the caller
  const uint8_t* best;          // place-best: per query, the best distance of its read (0xff: none, nothing placed);
                                // a key at distance d is placed iff d <= min(best + 1, k)
};
cudaError_t launch_hamming_verify(const IndexView& ix, const HammingSlice& a, uint32_t k, VerifyMode mode, int sm_count,
                                  cudaStream_t s);
// the n < 2^31 keys of a part of a CSR sorted per query (segment i = d_off[i] - base .. d_off[i+1] - base)
cudaError_t sort_hamming_keys(const uint64_t* d_keys, uint64_t* d_sorted, uint64_t n, uint64_t nseg,
                              const uint64_t* d_off, uint64_t base, void* d_temp, size_t& temp_bytes, cudaStream_t s);
cudaError_t scan_u64(const uint64_t* d_in, uint64_t* d_out, uint64_t n, void* d_temp, size_t& temp_bytes, cudaStream_t s);
// device-resident locate: d_sums[q] = the sum of read q's k + 1 counts, q < nq, and d_sums[nq] = 0 (its exclusive scan
// is the CSR over the reads)
cudaError_t launch_hamming_row_sums(const uint64_t* d_counts, uint32_t k, uint64_t nq, uint64_t* d_sums, cudaStream_t s);
// sorted keys (s << 2 | d) -> the text positions s in place, and the distances d to d_dist unless it is null
cudaError_t launch_hamming_decode(uint64_t* d_keys, uint64_t n, uint8_t* d_dist, cudaStream_t s);

// ---- kernels_edit.cu: edit-distance search (<= k substitutions, insertions, deletions) on the Hamming candidates.
// Every candidate names 2k + 1 starts (start s0 - δ, δ = -k .. k).
cudaError_t launch_edit_verify(const IndexView& ix, const HammingSlice& a, uint32_t k, VerifyMode mode, int sm_count,
                               cudaStream_t s);
// loci of n edit-distance hits sorted per query (DESIGN.md §1g); d_keys: their keys (s << 2 | d), d_off: their CSR
// (nq + 1, from 0), d_map: the query of every hit (launch_hamming_map over d_off).  d_counts (nq (k+1), zeroed) not
// null: each locus adds 1 to d_counts[q (k+1) + d]; otherwise d_keep (n + 1) gets 1 per locus, 0 per other hit and at n.
cudaError_t launch_edit_loci(const uint64_t* d_keys, const uint64_t* d_off, const uint32_t* d_map, uint64_t n, uint32_t k,
                             uint64_t* d_keep, uint64_t* d_counts, cudaStream_t s);
// d_off[q] = d_P[d_off[q]], q = 0 .. nq: the loci's CSR from the exclusive scan d_P of the keep flags
cudaError_t launch_edit_loci_offsets(const uint64_t* d_P, uint64_t* d_off, uint64_t nq, cudaStream_t s);
// the keys of the loci (d_P[i + 1] > d_P[i]) among the n keys d_keys to slot d_P[i] of d_keys_out
cudaError_t launch_edit_loci_compact(const uint64_t* d_P, uint64_t n, const uint64_t* d_keys, uint64_t* d_keys_out,
                                     cudaStream_t s);

// ---- kernels_align.cu: the alignment of located Hamming and edit-distance hits (awry_align_*, DESIGN.md §1f)
// d_qlen[v] = the length L of search query v (read or virtual query, packed in d_qwords as for launch_search), or 0 when
// the prepass refused it, it is empty, holds '$' / '#' or has L <= k; the last is latched in *d_first_bad as BAD_QUERY
// of read v >> shift (the prepass latches the others)
cudaError_t launch_align_reads(const uint64_t* d_qwords, const uint64_t* d_qoff, uint64_t nq, uint64_t b_lo, uint64_t b_hi,
                               uint64_t qw_lo, uint64_t qw_n, uint32_t k, uint32_t shift, uint32_t* d_qlen,
                               unsigned long long* d_first_bad, cudaStream_t s);
// one slice of hits for the alignment kernel
struct AlignSlice {
  const uint64_t* qwords;  // packed search queries, biased as for launch_search
  uint64_t qw_lo, qw_n;    // the words that exist: [qw_lo, qw_lo + qw_n) (checked build)
  const uint64_t* qoff;    // their offsets (nq + 1)
  const uint32_t* qlen;    // launch_align_reads
  uint64_t nq;
  const uint32_t* map;     // query of every hit of the slice (launch_hamming_map over the hit offsets)
  const uint64_t* hits;    // (seq_idx, local_pos) of every hit of the slice
  uint32_t* out;           // one awry_alignment (11 u32) per hit of the slice
  uint64_t n;
  const uint64_t* hit_end; // checked build: *hit_end == hit_total (the hit offsets end where the hits do)
  uint64_t hit_total;
};
cudaError_t launch_align_hits(const IndexView& ix, const AlignSlice& a, uint32_t k, bool edit, int sm_count, cudaStream_t s);

// ---- kernels_map.cu: read mapping, the best locus per read (awry_map_*, DESIGN.md §1h).  Read q stands for the
// search queries v = q << shift .. (q << shift) + (1 << shift) - 1 (shift 1: both strands, v = 2q + 1 is rc(q)).
// From the count pass (d_counts, nv (k+1)): d_best[v] = the smallest d with a hit over all of q's queries, for each
// of them, 0xff when there is none or d_qlen[q << shift] == 0 (refused: nothing of it is placed); d_sums[v] = v's hits
// at d <= min(best + 1, k), d_sums[nv] = 0 (its exclusive scan is the CSR of the bounded place pass)
cudaError_t launch_map_bound(const uint64_t* d_counts, const uint32_t* d_qlen, uint64_t nq, uint32_t k, uint32_t shift,
                             uint8_t* d_best, uint64_t* d_sums, cudaStream_t s);
// d_roff[q] = d_hit_off[q << shift], q = 0 .. nq: the hits' CSR over the reads
cudaError_t launch_map_read_offsets(const uint64_t* d_hit_off, uint64_t nq, uint32_t shift, uint64_t* d_roff,
                                    cudaStream_t s);
// the hits' keys (s << 2 | d) -> (s << 3) | (d << 1) | strand, strand = whether the hit lies in the range of v = 2q + 1.
// d_rmap: the read of every hit (launch_hamming_map over d_roff); n bounds the hits, whose total is d_roff[nq]
cudaError_t launch_map_rekey(const uint64_t* d_keys, const uint64_t* d_hit_off, const uint64_t* d_roff,
                             const uint32_t* d_rmap, uint64_t nq, uint64_t n, uint32_t shift, uint64_t* d_out,
                             cudaStream_t s);
// over the re-keyed hits sorted per read: the first entry of each start represents it (smallest distance, then strand
// 0).  d_flag[i] (n + 1 entries, 0 past the total) = 1 for a representative at the read's best distance;
// d_second[q] (zeroed) += 1 for one at best + 1
cudaError_t launch_map_flags(const uint64_t* d_keys, const uint64_t* d_roff, const uint32_t* d_rmap, const uint8_t* d_best,
                             uint64_t nq, uint64_t n, uint32_t shift, uint64_t* d_flag, uint32_t* d_second,
                             cudaStream_t s);
// one read per thread: its awry_mapping record, and the inputs of launch_align_hits for its primary
struct MapReads {
  const uint64_t* qwords;  // packed search queries, biased as for launch_search (the read itself at v = q << shift)
  uint64_t qw_lo, qw_n;    // the words that exist: [qw_lo, qw_lo + qw_n) (checked build)
  const uint64_t* qoff;    // their offsets (nv + 1)
  const uint32_t* qlen;    // launch_align_reads (0: refused)
  const uint64_t* keys;    // re-keyed hits sorted per read
  const uint64_t* roff;    // nq + 1
  const uint64_t* rank;    // exclusive scan of launch_map_flags' flags
  const uint8_t* best;     // launch_map_bound
  const uint32_t* second;  // launch_map_flags
  uint64_t nq;
  uint32_t k, shift;
  uint64_t* out;           // 4 u64 per read (awry_mapping)
  uint32_t* aln_map;       // nullptr, or per read its primary's search query (for launch_align_hits)
  uint64_t* aln_hits;      // per read its primary (seq_idx, local_pos), ~0 when unmapped
  uint64_t* aln_end;       // [0] = nq (the AlignSlice hit total)
};
cudaError_t launch_map_reads(const IndexView& ix, const MapReads& m, cudaStream_t s);

cudaError_t launch_single_update(const IndexView& ix, uint64_t sp, uint64_t ep, uint32_t dsym,
                                 uint64_t* d_out2, cudaStream_t s);
cudaError_t launch_single_backstep(const IndexView& ix, uint64_t row, uint64_t* d_out, cudaStream_t s);

// ---- kernels_wide.cu: indexes with 64-bit row pointers (the launchers above dispatch on IndexView::wide)
cudaError_t launch_build_table_wide(const WideView& ix, ulonglong2* d_table, uint32_t k, cudaStream_t s);
cudaError_t launch_search_wide(const WideView& ix, const uint64_t* d_qwords, const uint64_t* d_qoff, uint64_t nq,
                               SearchOut mode, void* d_out, uint32_t* d_scratch /* >= 1 u32: ticket counter */,
                               const SearchVariant& v, int sm_count, cudaStream_t s);
cudaError_t scan_hit_offsets_wide(const void* d_sp_cnt, uint64_t nq, uint64_t* d_hit_off, void* d_temp, size_t& temp_bytes,
                                  cudaStream_t s);
cudaError_t launch_walk_wide(const WideView& ix, const void* d_sp_cnt, const uint64_t* d_hit_off, uint64_t nq, uint64_t n_hits,
                             uint64_t* d_hits_pairs, uint64_t* d_locs, int sm_count, cudaStream_t s);
cudaError_t launch_single_update_wide(const WideView& ix, uint64_t sp, uint64_t ep, uint32_t dsym, uint64_t* d_out2,
                                      cudaStream_t s);
cudaError_t launch_single_backstep_wide(const WideView& ix, uint64_t row, uint64_t* d_out, cudaStream_t s);
cudaError_t launch_ref_table_wide(const WideView& ix, uint64_t first, uint64_t count, uint32_t k, void* d_out, cudaStream_t s);

cudaError_t run_random_gather(uint64_t footprint_bytes, uint32_t granule, uint32_t lanes,
                              uint64_t n_reads, int iters, double* reads_per_s, double* gb_per_s);

uint64_t kernel_launch_count();
void kernel_launch_count_reset();

}  // namespace awry
