/*
 * awry_b200.h -- C ABI of the B200-native batched FM-index search path.
 *
 * Drop-in boundary for the query side of the Rust crate `awry` 0.3.1
 * (awry::fm_index::FmIndex).  The reference has no FFI of its own; a thin Rust facade
 * crate (rust/ in this repo, see INTEGRATION.md) keeps the reference's public signatures
 * and binds exactly these entry points.  Each declaration cites the reference interface it
 * replaces (paths under /root/reference/src).
 *
 * Conventions: every function returns AWRY_OK (0) or a negative awry_status; nothing
 * unwinds or aborts across this boundary; awry_last_error() gives a thread-local message.
 * An awry_index is immutable after creation, so the *_batch calls may be issued
 * concurrently from many host threads (each call uses a private stream and workspace),
 * like `&self` methods called from the rayon pool in the reference.
 * There is NO CPU fallback: every search entry point fails with AWRY_ERR_CUDA when no
 * usable sm_100 device is present.
 */
#ifndef AWRY_B200_H
#define AWRY_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef enum awry_status {
  AWRY_OK = 0,
  AWRY_ERR_INVALID_ARG = -1, /* null pointer, query offsets not monotone, ... */
  AWRY_ERR_IO = -2,          /* FmIndex::load -> io::Error (fm_index_file.rs:132)              */
  AWRY_ERR_FORMAT = -3,      /* bad label / header (fm_index_file.rs:145-150)                  */
  AWRY_ERR_CUDA = -4,        /* no device, allocation or launch failure                        */
  AWRY_ERR_INVALID_QUERY = -5, /* empty query or a query containing '$'/'#': the reference
                                  panics or is UB here (fm_index.rs:406, bwt.rs:127)           */
  AWRY_ERR_UNSUPPORTED = -6, /* e.g. 2-bit packed queries on a protein index                       */
  AWRY_ERR_NOMEM = -7,
  AWRY_ERR_CAPACITY = -8     /* caller-owned output buffer too small; the needed size is reported */
} awry_status;

/* awry::alphabet::SymbolAlphabet (alphabet.rs:28-31); values = the file header's alphabet id */
enum { AWRY_NUCLEOTIDE = 0, AWRY_AMINO = 1 };

typedef struct awry_index awry_index; /* opaque; replaces awry::fm_index::FmIndex (fm_index.rs:41-56) */

/* awry::search::SearchRange (search.rs:25-28): inclusive [start_ptr, end_ptr], empty iff start > end */
typedef struct awry_range {
  uint64_t start_ptr;
  uint64_t end_ptr;
} awry_range;

/* awry::sequence_index::LocalizedSequencePosition (sequence_index.rs:33-36) */
typedef struct awry_hit {
  uint64_t seq_idx;
  uint64_t local_pos;
} awry_hit;

/* Getters of FmIndex (fm_index.rs:302-368) plus sizes of the device replica. */
typedef struct awry_info {
  uint64_t version;          /* version_number()  fm_index.rs:350 */
  uint64_t sa_ratio;         /* suffix_array_compression_ratio()  fm_index.rs:320 */
  uint64_t bwt_len;          /* bwt_len()  fm_index.rs:335 */
  uint32_t alphabet;         /* alphabet()  fm_index.rs:302 */
  uint32_t kmer_len;         /* KmerLookupTable::kmer_len  kmer_lookup_table.rs:86 */
  uint32_t n_prefix_sums;    /* 7 / 23 */
  uint32_t n_devices;
  uint64_t prefix_sums[23];  /* prefix_sums()  fm_index.rs:368 */
  uint64_t n_sequences;
  uint64_t device_bytes_blocks; /* per replica */
  uint64_t device_bytes_sa;
  uint64_t device_bytes_table;
  uint64_t device_bytes_pair;   /* nucleotide two-symbol accelerator blocks */
  uint64_t device_bytes_full_sa; /* unsampled suffix array (locate accelerator), 0 if not built */
  uint64_t device_bytes_lean_sa; /* walk blocks + position-sampled suffix array (bounded locate), 0 if not built */
  int32_t devices[16];
  uint32_t row_pointer_bits;    /* 32 while bwt_len < 2^32 - 256, else 64 (SearchPtr = u64, search.rs:7) */
  uint32_t lean_sa_ratio;       /* sampling distance of the derived position-sampled suffix array, 0 if not built */
  uint64_t device_bytes_text;   /* nucleotide: the indexed text, reversed, 4 bits per symbol (count accelerator), 0 if not built */
} awry_info;

/* The fields FmIndex::new hands over after the reference's CPU construction
 * (fm_index.rs:242-251), all in the reference's own in-memory layout:
 *   blocks      ceil(bwt_len/256) blocks, each = planes (3|5 x 4 u64) then milestones (8|24 u64)
 *               (bwt.rs:12-25; same bytes as the file, fm_index_file.rs:58-68)
 *   prefix_sums card+1 u64 (fm_index.rs:233-240)
 *   sa_words    CompressedSuffixArray::data (compressed_suffix_array.rs:13,113-123)
 *   seq_starts  SequenceIndex start positions (sequence_index.rs:10-13); headers optional */
typedef struct awry_parts {
  uint32_t alphabet;
  uint32_t kmer_len;
  uint64_t sa_ratio;
  uint64_t bwt_len;
  uint64_t version;
  const uint64_t *blocks;
  const uint64_t *prefix_sums;
  const uint64_t *sa_words;
  const uint64_t *seq_starts;
  const char *const *headers; /* may be NULL */
  uint64_t n_sequences;
} awry_parts;

/* ------------------------------------------------------------------ index lifetime */

/* FmIndex::load (fm_index_file.rs:132-160, :184-287): reads an `.awry` v1 file, re-lays the
 * BWT blocks out for the device, rebuilds the k-mer seed table on the device (the file's table
 * is never consulted, as in the reference: kmer_lookup_table.rs:90-110) and replicates the
 * index on each listed CUDA device.  devices == NULL / n_dev == 0 means device 0. */
int awry_index_load(const char *path, const int *devices, int n_dev, awry_index **out);

/* Device replica of an index the reference's FmIndex::new (fm_index.rs:142-268) just built. */
int awry_index_from_parts(const awry_parts *parts, const int *devices, int n_dev, awry_index **out);

void awry_index_free(awry_index *index);

int awry_index_info(const awry_index *index, awry_info *info);

/* SequenceIndex header lookup (sequence_index.rs:10-13); pointer valid until awry_index_free */
int awry_index_sequence_header(const awry_index *index, uint64_t seq_idx, const char **header,
                               uint64_t *header_len);

/* FmIndex::save (fm_index_file.rs:42-106) of any handle -- loaded, handed over or built: writes an
 * `.awry` v1 file the reference (and awry_index_load) reads.  The handle keeps only the device layout, so
 * the bwt.rs blocks are re-derived from it on replica 0 (bit planes re-encoded to the reference's symbol
 * codes, milestones from the block-start counts) and streamed out with the sampled suffix-array words; the
 * k-mer table section is re-populated the way kmer_lookup_table.rs:121-167 does.  For a file the
 * reference wrote, load followed by save reproduces it byte for byte.  An existing file is truncated. */
int awry_index_save(const awry_index *index, const char *path);

/* ------------------------------------------------------------------ index construction on the GPU
 * SURVEY.md 8(f): the reference builds on the CPU (FmIndex::new, fm_index.rs:142-268, libsufr suffix
 * sort) and that path stays valid (awry_index_from_parts).  These entry points do the same work on
 * the device and emit the reference's layout / file format. */

/* FmBuildArgs (fm_index.rs:78-96), the fields that still mean something without libsufr */
typedef struct awry_build_args {
  const char *input_file_src;   /* FASTA or FASTQ */
  const char *output_file_src;  /* `.awry` v1 file to write (FmIndex::save, fm_index_file.rs:42), or NULL */
  uint32_t alphabet;            /* AWRY_NUCLEOTIDE / AWRY_AMINO */
  uint32_t lookup_table_kmer_len;          /* 0 = default 10 / 4 (kmer_lookup_table.rs:23-24) */
  uint64_t suffix_array_compression_ratio; /* 0 = default 8 (fm_index.rs:122) */
  int32_t device;
} awry_build_args;

/* FmIndex::new (fm_index.rs:142-268): reads the sequence file (records upper-cased and joined by
 * 'N' / 'X', as libsufr's read_sequence_file does for the reference), builds the index on
 * devices[0] (args->device when `devices` is NULL) and returns a ready-to-search handle replicated on
 * `devices`, like awry_index_load.  When args->output_file_src is not NULL it also does FmIndex::save
 * (fm_index_file.rs:42-106): an `.awry` v1 file the reference can load, including its k-mer table
 * section populated the way kmer_lookup_table.rs:121-167 does.  `out` may be NULL (file only).
 * I/O and format errors of the input are reported before any device is touched. */
int awry_index_build(const awry_build_args *args, const int *devices, int n_dev, awry_index **out);

/* What the reference gets from libsufr::util::read_sequence_file (fm_index.rs:153): the records of a
 * FASTA / FASTQ file concatenated with 'N' / 'X' between them, and each record's start offset.  Host
 * only (no device needed); large FASTA files are parsed by several threads.  *text and *starts are
 * library-owned: release with awry_buffer_free. */
int awry_read_sequence_file(const char *path, uint32_t alphabet, uint8_t **text, uint64_t *n_text,
                            uint64_t **starts, uint64_t *n_records);

/* FmIndex::new + FmIndex::save without keeping the index: awry_index_build(args, NULL, 0, NULL). */
int awry_build_index_file(const awry_build_args *args);

/* The single construction pass of fm_index.rs:202-240 for text[0..n) + '$' (ASCII, host OR device
 * pointer): fills caller-owned reference-layout arrays sized by the helpers below, ready for
 * awry_index_from_parts.  phase_seconds: 8 doubles or NULL. */
int awry_build_parts(uint32_t alphabet, const uint8_t *text, uint64_t n, uint64_t sa_ratio, int device,
                     uint64_t *blocks, uint64_t *prefix_sums, uint64_t *sa_words, double *phase_seconds);
uint64_t awry_parts_num_blocks(uint64_t bwt_len);                   /* bwt.rs:302-304 */
uint64_t awry_parts_block_words(uint32_t alphabet);                 /* 20 / 44 u64 per block */
uint64_t awry_parts_sa_words(uint64_t bwt_len, uint64_t sa_ratio);  /* compressed_suffix_array.rs:113-123 */

/* ------------------------------------------------------------------ batched search (host buffers) */

/* FmIndex::parallel_count (fm_index.rs:455-460); count_string (:499-501) is a batch of one.
 * Queries are ASCII, concatenated in qbytes; query i = qbytes[qoff[i] .. qoff[i+1]).
 * counts (caller-owned, nq entries) are written in input order. */
int awry_count_batch(const awry_index *index, const uint8_t *qbytes, const uint64_t *qoff,
                     uint64_t nq, uint64_t *counts);

/* Same search, returning the final SearchRange per query (get_search_range_for_string,
 * fm_index.rs:402-438).  Empty ranges are reported as SearchRange::zero() = (1,0). */
int awry_search_batch(const awry_index *index, const uint8_t *qbytes, const uint64_t *qoff,
                      uint64_t nq, awry_range *ranges);

enum {
  AWRY_LOCATE_BWT_ORDER = 0, /* per-query hits in BWT-row order, exactly the reference's
                                push order (fm_index.rs:521) */
  AWRY_LOCATE_SORTED = 1     /* per-query hits sorted ascending by (seq_idx, local_pos) */
};

/* FmIndex::parallel_locate (fm_index.rs:479-487); locate_string (:516-544) is a batch of one.
 * hit_off (caller-owned, nq+1 entries) is the CSR offset array; *hits is library-owned
 * (release with awry_hits_free) and holds *n_hits entries. */
int awry_locate_batch(const awry_index *index, const uint8_t *qbytes, const uint64_t *qoff,
                      uint64_t nq, uint32_t flags, uint64_t *hit_off, awry_hit **hits,
                      uint64_t *n_hits);
void awry_hits_free(awry_hit *hits);

/* Same, with caller-owned output like `counts` above: up to `capacity` hits are written to `hits`.
 * *n_hits is always the total found; if it exceeds `capacity` the call returns AWRY_ERR_CAPACITY
 * (hit_off is complete, hits is not) and can be repeated with a larger buffer.  capacity = 0 just fills
 * hit_off / *n_hits.  With `hits` in page-locked memory (cudaHostAlloc / cudaHostRegister), BWT order and
 * the unsampled suffix array present, the two passes run without a host round trip: the device keeps the
 * running hit total and the gather kernel writes the hits straight into `hits`. */
int awry_locate_batch_into(const awry_index *index, const uint8_t *qbytes, const uint64_t *qoff,
                           uint64_t nq, uint32_t flags, uint64_t *hit_off, awry_hit *hits,
                           uint64_t capacity, uint64_t *n_hits);

/* ------------------------------------------------------------------ batched search on pre-packed reads
 * The reference's callers hold `&str`s (fm_index.rs:455-487), so the calls above take ASCII and the
 * library packs it to 2 bits per base on the host cores before the PCIe copy.  A caller that searches the
 * same reads more than once, or stores them packed, can hand the 2-bit form over and skip that pass: a
 * quarter of the bytes are read from host memory and nothing is computed on the host.  Nucleotide only.
 *   crumbs      code of query byte p (p counted as in qoff) = (ascii >> 1) & 3  (A0 C1 T2 G3, either case)
 *               at bits 2*(p%4) of crumbs[p/4]; the array holds ceil(qoff[nq]/4) bytes
 *               (awry_host_pack_dna produces exactly this)
 *   exceptions  every byte outside ACGTacgt (N, IUPAC codes, '$'...) as (p << 8) | ascii byte, strictly
 *               ascending by p; its crumb is ignored
 * Results are those of awry_count_batch / awry_locate_batch_into on the ASCII the codes stand for. */
int awry_count_batch_packed2(const awry_index *index, const uint8_t *crumbs, const uint64_t *qoff,
                             uint64_t nq, const uint64_t *exceptions, uint64_t n_exc, uint64_t *counts);
int awry_locate_batch_packed2(const awry_index *index, const uint8_t *crumbs, const uint64_t *qoff,
                              uint64_t nq, const uint64_t *exceptions, uint64_t n_exc, uint32_t flags,
                              uint64_t *hit_off, awry_hit *hits, uint64_t capacity, uint64_t *n_hits);

/* ------------------------------------------------------------------ Hamming search (<= k substitutions, no indels)
 * The reference answers one question, where a query occurs EXACTLY (get_search_range_for_string, fm_index.rs:402-438,
 * one update_range_with_symbol step per symbol, :559-582).  These calls extend it to windows of the text within
 * Hamming distance k (Bowtie's `-v k`), nucleotide only.  Insertions and deletions: the edit-distance block below.
 *   text      the text the index holds: records joined by 'N', n = bwt_len - 1 symbols, no '$' (fm_index.rs:148-153).
 *             A window is text[s .. s+L) for 0 <= s <= n - L; windows may cross record delimiters, where the 'N' is
 *             an ordinary symbol, as for exact search.
 *   distance  the number of positions whose symbols differ, query bytes mapped as for exact search (either case,
 *             U = T, any other byte = N): a query N matches a text N and mismatches A / C / G / T.
 *   count     counts[q * (k+1) + d] = the number of windows at distance exactly d, d = 0 .. k (caller-owned,
 *             nq * (k+1) entries).  For k = 0 this equals awry_count_batch.
 *   locate    every window at distance <= k, once each, per query in ascending text position, i.e. ascending
 *             (seq_idx, local_pos) of the window start.  hit_mismatches (NULL or `capacity` entries) receives each
 *             hit's distance.  capacity / AWRY_ERR_CAPACITY as in awry_locate_batch_into: hit_off (nq+1) and
 *             *n_hits are complete even when `hits` is not.
 *   errors    k > AWRY_HAMMING_MAX -> AWRY_ERR_INVALID_ARG; an empty query or one with '$' / '#', and a query of
 *             length L <= k (every window would match) -> AWRY_ERR_INVALID_QUERY; a protein index, or one without
 *             the unsampled suffix array and the text on the device (AWRY_B200_FULL_SA=0, AWRY_B200_TEXT=0,
 *             AWRY_B200_PAIR_INDEX=0, a file that samples every suffix array entry (ratio 1), not enough device
 *             memory, 64-bit row pointers) -> AWRY_ERR_UNSUPPORTED.  Locate works through chunks of queries (at most
 *             512 k queries and 64 MB, as awry_locate_batch) and, as awry_locate_device_hamming, holds a chunk's hits
 *             on the device: when they do not fit, or one query has 2^31 hits or more -> AWRY_ERR_NOMEM, naming the
 *             hit total.
 * Scheme (pigeonhole): the query is cut into k+1 pieces, piece j = bytes [a_j, a_{j+1}), a_j = floor(j L / (k+1));
 * each piece is searched exactly, an occurrence of piece j at text position p names the window s = p - a_j, and the
 * window is verified against the text on the device.  It is kept iff its distance is <= k and j is the smallest piece
 * it matches exactly, so no window is reported twice.  Cost: about one exact search per piece plus one verification
 * per candidate, and the candidates are about the sum over pieces of n / 4^(piece length): short queries at high k
 * (12 bp at k = 3: 3-bp pieces) are legal but expensive. */
enum { AWRY_HAMMING_MAX = 3 };
int awry_count_batch_hamming(const awry_index *index, const uint8_t *qbytes, const uint64_t *qoff, uint64_t nq,
                             uint32_t max_mismatches, uint64_t *counts /* nq * (max_mismatches + 1) */);
int awry_locate_batch_hamming(const awry_index *index, const uint8_t *qbytes, const uint64_t *qoff, uint64_t nq,
                              uint32_t max_mismatches, uint64_t *hit_off /* nq + 1 */, awry_hit *hits,
                              uint8_t *hit_mismatches /* NULL or capacity entries */, uint64_t capacity,
                              uint64_t *n_hits);
/* awry_count_batch_hamming on device-resident queries (see awry_count_device below): pointers on replica `replica`'s
 * device, work enqueued on `cuda_stream`.  It synchronises that stream once, after the pieces are searched (the
 * candidate total sizes the verification), and returns without waiting for the verification.  An empty / sentinel /
 * L <= k query is latched and reported by awry_device_check; its counts are 0. */
int awry_count_device_hamming(const awry_index *index, int replica, const uint8_t *d_qbytes, const uint64_t *d_qoff,
                              uint64_t nq, uint32_t max_mismatches, uint64_t *d_counts, void *cuda_stream);
/* awry_locate_batch_hamming on device-resident queries (see awry_locate_device below).  No per-read data goes to the
 * host.
 *   results   bit for bit those of awry_locate_batch_hamming on the same reads: d_hit_off (nq + 1, device), the hits
 *             of each query in ascending text position as (seq_idx, local_pos), and each hit's distance.
 *   output    *d_hits and *d_hit_mismatches are device allocations from the library's stream-ordered pool, released
 *             with awry_device_free.  d_hit_mismatches == NULL: no distances are produced.  No hits: *n_hits = 0 and
 *             both pointers NULL.  nq = 0 behaves as awry_locate_device.
 *   sync      besides the read-back of the batch's first and last offset, the call synchronises `cuda_stream` twice:
 *             after the pieces are searched (the candidate total, as awry_count_device_hamming) and after a count pass
 *             over the candidates (the hit total sizes the output).  It returns without waiting for the last kernels;
 *             the results are valid in stream order.
 *   refused   an empty / sentinel / L <= k query, or one whose offsets leave the batch, is latched for
 *             awry_device_check as by awry_count_device_hamming, and gets the hit range that call's counts give it.
 *   errors    those of awry_count_device_hamming (k, replica, null pointers, 2 nq (k+1) >= 2^31 pieces ->
 *             AWRY_ERR_INVALID_ARG; the index -> AWRY_ERR_UNSUPPORTED); the hits do not fit the device, or one query
 *             has 2^31 hits or more -> AWRY_ERR_NOMEM, naming the hit total.
 * Scheme (DESIGN.md §1e): a count pass verifies every candidate and sizes each query's range, a place pass verifies them
 * again and writes each accepted window into its query's range, and a segmented sort puts each range in text order. */
int awry_locate_device_hamming(const awry_index *index, int replica, const uint8_t *d_qbytes, const uint64_t *d_qoff,
                               uint64_t nq, uint32_t max_mismatches, uint64_t *d_hit_off /* nq + 1 */,
                               awry_hit **d_hits, uint8_t **d_hit_mismatches /* NULL: not wanted */, uint64_t *n_hits,
                               void *cuda_stream);

/* ------------------------------------------------------------------ both strands (query and reverse complement)
 * A read comes from either strand of the DNA; the index holds one.  These calls search every query together with its
 * reverse complement, nucleotide only (a protein index -> AWRY_ERR_UNSUPPORTED).
 *   rc(q)      the query's bytes mapped as for exact search (either case, U = T, any other byte except '$' / '#' =
 *              N), complemented (A <-> T, C <-> G, N = N) and reversed.
 *   virtual    query q of a batch stands for two searches: v = 2q (the query) and v = 2q + 1 (rc(q)).  Every result
 *              for v = 2q + 1 is bit for bit what awry_count_batch / awry_locate_batch_into return for the ASCII
 *              string rc(q) over ACGTN, BWT-row order under AWRY_LOCATE_BWT_ORDER included; v = 2q is q itself.
 *   hits       a reverse-strand hit is the (seq_idx, local_pos) of the start of the window of the indexed text that
 *              equals rc(q) (the usual leftmost coordinate); windows may cross record delimiters, as for exact
 *              search.  A query equal to its reverse complement reports the same windows on both strands (nothing is
 *              deduplicated).
 *   counts     counts[2q] forward, counts[2q + 1] reverse complement (2 nq entries).
 *   locate     hit_off is the CSR over the virtual queries (2 nq + 1 entries): query q's forward hits are
 *              [hit_off[2q], hit_off[2q+1]), its reverse-strand hits [hit_off[2q+1], hit_off[2q+2]).  `flags` orders
 *              the hits within each strand; capacity / AWRY_ERR_CAPACITY as in awry_locate_batch_into.
 *   errors     an empty query or one with '$' / '#' -> AWRY_ERR_INVALID_QUERY, naming the caller's query index q;
 *              non-monotone offsets -> AWRY_ERR_INVALID_ARG.  The device calls latch refused queries for
 *              awry_device_check as awry_count_device does, and refuse (AWRY_ERR_INVALID_ARG) a batch whose 2 nq
 *              virtual queries would not fit the kernels' 32-bit query counters (2 nq >= 2^32 - 2^24).
 * Device hits (*d_hits) are released with awry_device_free. */
int awry_count_batch_strands(const awry_index *index, const uint8_t *qbytes, const uint64_t *qoff, uint64_t nq,
                             uint64_t *counts /* 2*nq: [2q] forward, [2q+1] reverse complement */);
int awry_locate_batch_strands(const awry_index *index, const uint8_t *qbytes, const uint64_t *qoff, uint64_t nq,
                              uint32_t flags, uint64_t *hit_off /* 2*nq + 1 */, awry_hit *hits, uint64_t capacity,
                              uint64_t *n_hits);
int awry_count_device_strands(const awry_index *index, int replica, const uint8_t *d_qbytes, const uint64_t *d_qoff,
                              uint64_t nq, uint64_t *d_counts /* 2*nq */, void *cuda_stream);
int awry_locate_device_strands(const awry_index *index, int replica, const uint8_t *d_qbytes, const uint64_t *d_qoff,
                               uint64_t nq, uint32_t flags, uint64_t *d_hit_off /* 2*nq + 1 */, awry_hit **d_hits,
                               uint64_t *n_hits, void *cuda_stream);

/* ------------------------------------------------------------------ Hamming search on both strands
 * The two blocks above together: every query and its reverse complement, each with up to k substitutions.
 *   virtual    query q stands for v = 2q (q) and v = 2q + 1 (rc(q), as in the both-strands block).  Every result for
 *              v = 2q + 1 is bit for bit what awry_count_batch_hamming / awry_locate_batch_hamming return for the
 *              ASCII string rc(q): counts per distance, the hits in ascending text position and each hit's distance;
 *              v = 2q is q itself.  A query equal to its reverse complement reports the same windows on both strands.
 *   counts     counts[(2q + s) * (k+1) + d], s = 0 forward, s = 1 reverse complement (2 nq (k+1) entries).
 *   locate     hit_off is the CSR over the virtual queries (2 nq + 1 entries); capacity / AWRY_ERR_CAPACITY, and
 *              hit_mismatches, as in awry_locate_batch_hamming.
 *   errors     those of both blocks: k > AWRY_HAMMING_MAX -> AWRY_ERR_INVALID_ARG; an empty query, one with '$' / '#'
 *              or one of length L <= k -> AWRY_ERR_INVALID_QUERY, naming the caller's query index q; a protein index
 *              or one without the unsampled suffix array and the text -> AWRY_ERR_UNSUPPORTED.
 * The device count behaves as awry_count_device_hamming (one synchronisation, refused queries latched for
 * awry_device_check with counts 0) and refuses (AWRY_ERR_INVALID_ARG) a batch with 2 nq (k+1) >= 2^31 pieces.  The
 * device locate behaves as awry_locate_device_hamming over the 2 nq virtual queries (d_hit_off: 2 nq + 1 entries);
 * its results are bit for bit those of awry_locate_batch_hamming_strands. */
int awry_count_batch_hamming_strands(const awry_index *index, const uint8_t *qbytes, const uint64_t *qoff, uint64_t nq,
                                     uint32_t max_mismatches, uint64_t *counts /* 2*nq * (max_mismatches + 1) */);
int awry_locate_batch_hamming_strands(const awry_index *index, const uint8_t *qbytes, const uint64_t *qoff, uint64_t nq,
                                      uint32_t max_mismatches, uint64_t *hit_off /* 2*nq + 1 */, awry_hit *hits,
                                      uint8_t *hit_mismatches /* NULL or capacity entries */, uint64_t capacity,
                                      uint64_t *n_hits);
int awry_count_device_hamming_strands(const awry_index *index, int replica, const uint8_t *d_qbytes,
                                      const uint64_t *d_qoff, uint64_t nq, uint32_t max_mismatches,
                                      uint64_t *d_counts /* 2*nq * (max_mismatches + 1) */, void *cuda_stream);
int awry_locate_device_hamming_strands(const awry_index *index, int replica, const uint8_t *d_qbytes,
                                       const uint64_t *d_qoff, uint64_t nq, uint32_t max_mismatches,
                                       uint64_t *d_hit_off /* 2*nq + 1 */, awry_hit **d_hits,
                                       uint8_t **d_hit_mismatches /* NULL: not wanted */, uint64_t *n_hits,
                                       void *cuda_stream);

/* ------------------------------------------------------------------ edit-distance search (<= k substitutions,
 * insertions and deletions).  The Hamming block above with indels: a read with a one-base insertion or deletion
 * (homopolymer runs, a guide with a bulge) is found.  Nucleotide only.
 *   text      as in the Hamming block: n = bwt_len - 1 symbols, records joined by 'N'; an alignment may cross record
 *             delimiters.  Query bytes are mapped as for exact search, so a query N equals a text N.
 *   distance  Levenshtein distance (substitution, insertion, deletion: 1 each).  For a start position s (0 <= s < n),
 *             d(s) = min over l >= 0 with s + l <= n of ed(query, text[s .. s+l)).  An occurrence is a start s with
 *             d(s) <= k, reported once, with d(s).
 *   neighbouring starts  an occurrence is a START, not a locus: an exact occurrence at s also makes s - 1 .. s - k
 *             and s + 1 .. s + k occurrences at distances 1 .. k (insert text symbols in front of the query, or delete
 *             its leading symbols), and all of them are reported.  Nothing merges them into one locus.
 *             awry_*_edit_loci (the next block) report each locus once.
 *   count     counts[q * (k+1) + d] = the number of starts with d(s) = d (nq * (k+1) entries).  For k = 0 this equals
 *             awry_count_batch; for every k the d = 0 column equals that of the Hamming calls.
 *   locate    every start with d(s) <= k, once each, per query in ascending text position, as (seq_idx, local_pos) of
 *             s.  hit_edits (NULL or `capacity` entries) receives d(s).  capacity / AWRY_ERR_CAPACITY and hit_off (nq+1)
 *             as in awry_locate_batch_hamming.
 *   errors    k > AWRY_EDIT_MAX -> AWRY_ERR_INVALID_ARG; an empty query, one with '$' / '#' or one of length L <= k ->
 *             AWRY_ERR_INVALID_QUERY naming the caller's query; a protein index, or one without the unsampled suffix
 *             array and the text on the device -> AWRY_ERR_UNSUPPORTED.  The device calls latch refused queries for
 *             awry_device_check, and their counts are 0.
 * Scheme: the pieces, their exact search and the candidates are those of the Hamming calls.  An exact occurrence of
 * piece j at p names the starts [s0 - k, s0 + k], s0 = p - a_j, and each start's d(s) comes from one banded DP on the
 * device (4k + 1 diagonals).  A start is reported by the smallest (piece, position) occurrence within k of it, so
 * nothing is deduplicated globally.
 * The _strands calls search both strands, as the Hamming-on-both-strands block: v = 2q is q, v = 2q + 1 is rc(q),
 * counts[(2q + s) * (k+1) + d], hit_off over the 2 nq virtual queries; every v = 2q + 1 result is bit for bit that
 * of the single-strand call on rc(q).  The device counts behave as awry_count_device_hamming: one synchronisation,
 * after the pieces are searched.  The device locates behave as awry_locate_device_hamming (d_hit_edits receives d(s));
 * their results are bit for bit those of awry_locate_batch_edit and awry_locate_batch_edit_strands. */
enum { AWRY_EDIT_MAX = 3 };
int awry_count_batch_edit(const awry_index *index, const uint8_t *qbytes, const uint64_t *qoff, uint64_t nq,
                          uint32_t max_edits, uint64_t *counts /* nq * (max_edits + 1) */);
int awry_locate_batch_edit(const awry_index *index, const uint8_t *qbytes, const uint64_t *qoff, uint64_t nq,
                           uint32_t max_edits, uint64_t *hit_off /* nq + 1 */, awry_hit *hits,
                           uint8_t *hit_edits /* NULL or capacity entries */, uint64_t capacity, uint64_t *n_hits);
int awry_count_device_edit(const awry_index *index, int replica, const uint8_t *d_qbytes, const uint64_t *d_qoff,
                           uint64_t nq, uint32_t max_edits, uint64_t *d_counts /* nq * (max_edits + 1) */,
                           void *cuda_stream);
int awry_count_batch_edit_strands(const awry_index *index, const uint8_t *qbytes, const uint64_t *qoff, uint64_t nq,
                                  uint32_t max_edits, uint64_t *counts /* 2*nq * (max_edits + 1) */);
int awry_locate_batch_edit_strands(const awry_index *index, const uint8_t *qbytes, const uint64_t *qoff, uint64_t nq,
                                   uint32_t max_edits, uint64_t *hit_off /* 2*nq + 1 */, awry_hit *hits,
                                   uint8_t *hit_edits /* NULL or capacity entries */, uint64_t capacity,
                                   uint64_t *n_hits);
int awry_count_device_edit_strands(const awry_index *index, int replica, const uint8_t *d_qbytes,
                                   const uint64_t *d_qoff, uint64_t nq, uint32_t max_edits,
                                   uint64_t *d_counts /* 2*nq * (max_edits + 1) */, void *cuda_stream);
int awry_locate_device_edit(const awry_index *index, int replica, const uint8_t *d_qbytes, const uint64_t *d_qoff,
                            uint64_t nq, uint32_t max_edits, uint64_t *d_hit_off /* nq + 1 */, awry_hit **d_hits,
                            uint8_t **d_hit_edits /* NULL: not wanted */, uint64_t *n_hits, void *cuda_stream);
int awry_locate_device_edit_strands(const awry_index *index, int replica, const uint8_t *d_qbytes,
                                    const uint64_t *d_qoff, uint64_t nq, uint32_t max_edits,
                                    uint64_t *d_hit_off /* 2*nq + 1 */, awry_hit **d_hits,
                                    uint8_t **d_hit_edits /* NULL: not wanted */, uint64_t *n_hits, void *cuda_stream);

/* ------------------------------------------------------------------ edit-distance search by locus
 * The edit-distance block above reports starts: one occurrence comes back as up to 2k + 1 neighbouring starts.  These
 * calls report each locus once, so a read maps to one hit per place and per-distance counts count sites.
 *   virtual   v = q (strands = 0), or v = 2q (q) and v = 2q + 1 (rc(q)) (strands = 1), as in the blocks above.
 *   H         exactly the starts awry_locate_batch_edit[_strands] returns for v at that k, each with its distance d(s);
 *             s is the global start seq_starts[seq_idx] + local_pos.
 *   locus     a start s in H such that both hold:
 *             (a) no s' in H with 0 < |s' - s| <= k has d(s') < d(s) (a start within k of a strictly better one is a
 *                 shifted copy of it);
 *             (b) if d(s) >= 1, s - 1 is not in H with d(s - 1) = d(s) (a run of adjacent starts at one nonzero
 *                 distance is one locus, reported at its leftmost start).  Exact occurrences (d = 0) are never merged:
 *                 adjacent exact occurrences in a homopolymer all stay, as in exact search.
 *   so        k = 0: the loci are the hits of awry_locate_batch[_strands] with AWRY_LOCATE_SORTED.  The d = 0 loci are the
 *             exact occurrences (that column of the counts equals awry_count_batch[_strands]).  The loci are a subset
 *             of H with the same distances, in the same order.  The leftmost hit at a query's smallest distance is a
 *             locus, so the best distance per query is unchanged.  Different virtual queries never interact (forward
 *             and reverse-complement loci are decided separately).  Two occurrences more than k apart are both kept;
 *             so are two of equal distance within k unless they are adjacent (b).  A plateau's locus is its leftmost
 *             start: one optimal start, not necessarily the one a scoring aligner would prefer.
 *   count     counts[v * (k+1) + d] = the number of loci of v at distance d ((nq << strands) * (k+1) entries).
 *   locate    the loci of each v in ascending text position, as (seq_idx, local_pos), hit_off over the nq << strands
 *             virtual queries; hit_edits (NULL or `capacity` entries) receives d(s); capacity / AWRY_ERR_CAPACITY as
 *             in awry_locate_batch_edit.  awry_align_* aligns the loci as any edit-distance hit.
 *   errors    strands > 1 -> AWRY_ERR_INVALID_ARG; otherwise exactly those of the matching edit calls (k > 3, null
 *             pointers, a bad replica -> AWRY_ERR_INVALID_ARG; a refused query -> AWRY_ERR_INVALID_QUERY naming it in the
 *             host calls, latched for awry_device_check by the device calls; an unsupported index ->
 *             AWRY_ERR_UNSUPPORTED).  A refused query's device result is the filter applied to the range the device
 *             edit locate gives it.
 *   device    bit for bit the host calls' results.  The device locate synchronises three times (the candidate total,
 *             the hit total, the locus total that sizes the outputs); its outputs come from the stream-ordered pool and
 *             are released with awry_device_free.  The device count runs the place pass and the sort of the device
 *             locate and synchronises twice: it costs about a device locate, not a count.  Where starts will do,
 *             awry_count_device_edit is the cheaper call.
 * Scheme (DESIGN.md §1g): the hits of each query are sorted by text position; one thread per hit reads at most k
 * neighbours on each side, and the loci are compacted by a scan of the keep flags. */
int awry_count_batch_edit_loci(const awry_index *index, const uint8_t *qbytes, const uint64_t *qoff, uint64_t nq,
                               uint32_t strands /* 0 or 1 */, uint32_t max_edits,
                               uint64_t *counts /* (nq << strands) * (max_edits + 1) */);
int awry_locate_batch_edit_loci(const awry_index *index, const uint8_t *qbytes, const uint64_t *qoff, uint64_t nq,
                                uint32_t strands, uint32_t max_edits, uint64_t *hit_off /* (nq << strands) + 1 */,
                                awry_hit *hits, uint8_t *hit_edits /* NULL or capacity */, uint64_t capacity,
                                uint64_t *n_hits);
int awry_count_device_edit_loci(const awry_index *index, int replica, const uint8_t *d_qbytes, const uint64_t *d_qoff,
                                uint64_t nq, uint32_t strands, uint32_t max_edits, uint64_t *d_counts, void *cuda_stream);
int awry_locate_device_edit_loci(const awry_index *index, int replica, const uint8_t *d_qbytes, const uint64_t *d_qoff,
                                 uint64_t nq, uint32_t strands, uint32_t max_edits, uint64_t *d_hit_off,
                                 awry_hit **d_hits, uint8_t **d_hit_edits /* NULL: not wanted */, uint64_t *n_hits,
                                 void *cuda_stream);

/* ------------------------------------------------------------------ alignment of Hamming and edit-distance hits
 * The locate calls above say where a query matches and at what distance; these calls say what matched: the end of
 * each hit's alignment and its edit operations (a CIGAR), nucleotide only.  Text, query bytes, n and the virtual
 * queries of both-strand search are as in the blocks above.
 *   Q         the searched string: query q (single strand, or v = 2q), rc(q) for v = 2q + 1; L = its length.
 *   s         the hit's global start, seq_starts[seq_idx] + local_pos; T = the text.
 *   Hamming   window T[s .. s+L) inside the text with <= k mismatches: text_len = L, distance = the mismatches, one
 *             'X' op per mismatching position, ascending.
 *   edit      d(s) as in the edit-distance block (start fixed, end free, only T[s .. n) used).  If d(s) <= k the
 *             alignment is the lexicographically smallest op string (order '=' < 'X' < 'I' < 'D') among all
 *             alignments of Q against some T[s .. s+l) of cost d(s); text_len = l.  Equivalently: walk from cell (0, 0),
 *             take a match whenever the symbols are equal, otherwise the first of X, I, D after which cost d(s) is
 *             still reachable, and stop once all L query symbols are used (never a trailing D).  At s + j = n only I
 *             is possible.
 *   none      otherwise, and for a hit of a refused query, a hit with seq_idx >= n_sequences or s >= n: "no alignment
 *             within k": distance = k + 1, n_ops = 0, text_len = 0.
 *   ops       SAM conventions: I = a query symbol against nothing, D = a text symbol against nothing.  A reverse-strand
 *             hit is reported in rc(q) coordinates, as SAM stores a reverse-strand record, so the ops read in
 *             reference order.  Unused ops and every pad byte are 0.
 *   promise   for every hit a locate call returns, with that call's query, metric, strands and k (edit for the loci): distance = the
 *             call's distance of the hit, n_ops = distance, and applying the ops to Q gives exactly T[s .. s+text_len).
 *   inputs    hit_off / hits exactly as the locate calls produce them (awry_locate_{batch,device}_{hamming,edit}
 *             [_strands], awry_locate_{batch,device}_edit_loci): hit_off has nv + 1 entries, nv = nq << strands, and hit_off[0] = 0; hits may be in any order
 *             within their query's range and each is aligned on its own.  out[h] belongs to hits[h].
 *   errors    k > 3, an unknown metric, strands > 1, a null pointer, hit_off not starting at 0 or not monotone (host
 *             call) -> AWRY_ERR_INVALID_ARG; a protein index or one without the text on the device (as the approximate
 *             calls) -> AWRY_ERR_UNSUPPORTED; the host call: an empty query, one with '$' / '#' or with L <= k ->
 *             AWRY_ERR_INVALID_QUERY naming q.  The device call latches such queries for awry_device_check and their
 *             hits get "no alignment".
 *   device    awry_align_device reads back the batch's first and last query offset (one synchronisation) and returns
 *             without waiting; it trusts d_hit_off[nv] == n_hits (the bounds-checked build asserts it).  All pointers
 *             are on replica `replica`'s device.
 * Scheme (DESIGN.md §1f): one thread per hit reads the packed query against the text on the device: Hamming compares 8
 * symbols per step, edit distance runs an iterative-deepening search over budgets 0 .. k that extends matches 8
 * symbols at a time and tries X, I, D at a mismatch. */
enum { AWRY_METRIC_HAMMING = 0, AWRY_METRIC_EDIT = 1 };
typedef struct awry_edit_op {
  uint32_t qpos;     /* index into Q of the op's query symbol (I, X), or of the symbol it precedes (D) */
  uint32_t tpos;     /* offset into the window: text[s + tpos] (X, D), or the text offset it precedes (I) */
  uint8_t op;        /* 'X', 'I', 'D' */
  uint8_t query_sym; /* 'A', 'C', 'G', 'T', 'N' of Q (0 for D) */
  uint8_t text_sym;  /* 'A', 'C', 'G', 'T', 'N' of the text (0 for I) */
  uint8_t pad;
} awry_edit_op;
typedef struct awry_alignment {
  uint32_t text_len; /* l: the window is text[s .. s+l) */
  uint8_t distance;  /* k + 1: no alignment within k */
  uint8_t n_ops;     /* == distance when aligned */
  uint8_t pad[2];
  awry_edit_op ops[AWRY_EDIT_MAX]; /* the first n_ops are valid, ascending by qpos */
} awry_alignment;
typedef char awry_edit_op_is_12_bytes[sizeof(awry_edit_op) == 12 ? 1 : -1];
typedef char awry_alignment_is_44_bytes[sizeof(awry_alignment) == 44 ? 1 : -1];
int awry_align_batch(const awry_index *index, const uint8_t *qbytes, const uint64_t *qoff, uint64_t nq, uint32_t metric,
                     uint32_t strands /* 0 or 1 */, uint32_t k, const uint64_t *hit_off /* nv + 1, nv = nq << strands */,
                     const awry_hit *hits, awry_alignment *out /* hit_off[nv] entries */);
int awry_align_device(const awry_index *index, int replica, const uint8_t *d_qbytes, const uint64_t *d_qoff, uint64_t nq,
                      uint32_t metric, uint32_t strands, uint32_t k, const uint64_t *d_hit_off, const awry_hit *d_hits,
                      uint64_t n_hits, awry_alignment *d_out, void *cuda_stream);
/* Host only, no device: the extended CIGAR (op letters =, X, I, D; e.g. "47=1X102=") of one alignment of a query of
 * length L = query_len.  Writes at most cap bytes including the NUL; *needed (may be NULL) = full length + 1.
 * AWRY_ERR_CAPACITY if it did not fit (buf then holds nothing useful); AWRY_ERR_INVALID_ARG for a "no alignment"
 * record, n_ops > 3, or ops that are out of order or do not fit L. */
int awry_alignment_cigar(const awry_alignment *a, uint32_t query_len, char *buf, size_t cap, size_t *needed);

/* ------------------------------------------------------------------ read mapping: the best locus per read
 * The calls above return every hit within k; a read mapper wants one answer per read: its best locus over the searched
 * strands, whether that locus is unique, how far the runner-up is, and its alignment.  These calls give that record
 * for one batch, metric AWRY_METRIC_HAMMING or AWRY_METRIC_EDIT, strands 0 or 1, k <= 3.  Virtual queries (v = q, or
 * v = 2q for q and v = 2q + 1 for rc(q)), text, n and global starts are as in the blocks above.
 *   H_v       Hamming: exactly the windows awry_locate_batch_hamming[_strands] returns for v; edit: exactly the loci
 *             awry_locate_batch_edit_loci(strands) returns for v (mapping by start, with its shifted copies, would
 *             only inflate the counts).  d_v(s) is the distance of start s in H_v.
 *   per read  q's virtual queries merged by global start s: D(s) = min of d_v(s) over the v with s in H_v; strand(s) =
 *             the smaller strand attaining it.  A start found on both strands at one distance (a palindromic window)
 *             counts once, on strand 0.
 *   best      best = min D(s); B = {s : D(s) = best} in ascending s.  n_best = |B|; n_second = |{s : D(s) = best + 1}|
 *             if best < k, else 0 (that stratum was not searched).
 *   primary   B[h mod n_best], with h a hash of the read's own content: c_i = the code of read byte i as exact search
 *             maps it (A/a 0, C/c 1, G/g 2, T/t/U/u 3, any other byte 4), taken on the read as given, never on rc(q);
 *             h0 = FNV-1a-64 over the bytes c_0 .. c_{L-1} (basis 0xcbf29ce484222325, prime 0x100000001b3); h =
 *             fmix64(h0): x ^= x >> 33; x *= 0xff51afd7ed558ccd; x ^= x >> 33; x *= 0xc4ceb9fe1a85ec53; x ^= x >> 33.
 *             So equal loci (the copies of a repeat) share the reads between them, and the choice depends on the read
 *             alone: the same for every batch split, chunk size, replica, host or device call.  There is no seed.
 *   mapq      this project's definition, shaped after the approximate mapping quality of backtracking short-read
 *             mappers with c1 = n_best, c2 = n_second: 0 if the read is unmapped or n_best >= 2; 25 if best = k
 *             (uniqueness beyond k is unknown); otherwise AWRY_MAPQ_SECOND[min(n_second, 255)]: 37 for n_second = 0,
 *             else max(0, 23 - g(n_second)) with g(n) = floor(4.343 ln n + 0.5).
 *   aln       NULL: not made.  Otherwise, for a mapped read, aln[q] is exactly what awry_align_batch(metric, strands, k)
 *             returns for the single hit `hit` of v = (q << strands) | strand (ops in rc(q) coordinates on strand 1);
 *             for an unmapped read the "no alignment" record (distance k + 1, n_ops 0, text_len 0).
 *   refused   an empty read, one with '$' / '#', with L <= k or with offsets outside the batch: the host call fails with
 *             AWRY_ERR_INVALID_QUERY naming it; the device call latches it for awry_device_check and its record is
 *             AWRY_MAP_UNMAPPED | AWRY_MAP_REFUSED (whatever the search made of its bytes).
 *   errors    metric > 1, strands > 1, k > 3, a null pointer or a bad replica -> AWRY_ERR_INVALID_ARG; a protein index
 *             or one without the unsampled suffix array and the text -> AWRY_ERR_UNSUPPORTED; a batch too large for one
 *             approximate run -> the Hamming block's error; more than 2^31 hits within best + 1 in one batch ->
 *             AWRY_ERR_NOMEM (split the batch).
 *   device    outputs are the caller's (nq entries, sizes known up front): nothing to release.  awry_map_device
 *             synchronises as the device locates do (the offsets read-back, the candidate total, the hit total within
 *             the bound) and returns without waiting for its last kernels; results are bit for bit the host call's.
 * Scheme (DESIGN.md §1h): the count pass of the locate gives each read's best distance; only hits within best + 1 are
 * placed, sorted, filtered to loci (edit) and merged per read by one segmented sort; one thread per hit marks each
 * start's first entry, a scan ranks the best ones, and one thread per read writes its record. */
enum { AWRY_MAP_UNMAPPED = 1, AWRY_MAP_REFUSED = 2 };
typedef struct awry_mapping {
  awry_hit hit;      /* primary locus (seq_idx, local_pos); both ~0 when unmapped */
  uint32_t n_best;   /* distinct starts at `distance` over the searched strands; 0 when unmapped */
  uint32_t n_second; /* distinct starts at distance + 1; 0 when distance == k or unmapped */
  uint8_t distance;  /* best; k + 1 when unmapped */
  uint8_t strand;    /* 0: q, 1: rc(q) */
  uint8_t mapq;
  uint8_t flags;     /* AWRY_MAP_UNMAPPED (no locus <= k), AWRY_MAP_REFUSED (also unmapped) */
  uint32_t pad;      /* 0 */
} awry_mapping;
typedef char awry_mapping_is_32_bytes[sizeof(awry_mapping) == 32 ? 1 : -1];
/* mapq of a unique read with best < k, by min(n_second, 255) */
#define AWRY_MAPQ_SECOND \
  {37, 23, 20, 18, 17, 16, 15, 15, 14, 13, 13, 13, 12, 12, 12, 11, 11, 11, 10, 10, 10, 10, 10, 9, 9, 9, 9, 9, 9, 8, 8, 8,  \
   8, 8, 8, 8, 7, 7, 7, 7, 7, 7, 7, 7, 7, 6, 6, 6, 6, 6, 6, 6, 6, 6, 6, 6, 6, 5, 5, 5, 5, 5, 5, 5,  \
   5, 5, 5, 5, 5, 5, 5, 4, 4, 4, 4, 4, 4, 4, 4, 4, 4, 4, 4, 4, 4, 4, 4, 4, 4, 4, 3, 3, 3, 3, 3, 3,  \
   3, 3, 3, 3, 3, 3, 3, 3, 3, 3, 3, 3, 3, 3, 3, 3, 3, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2,  \
   2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1,  \
   1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0,  \
   0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0,  \
   0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0}
int awry_map_batch(const awry_index *index, const uint8_t *qbytes, const uint64_t *qoff, uint64_t nq, uint32_t metric,
                   uint32_t strands /* 0 or 1 */, uint32_t k, awry_mapping *out /* nq */,
                   awry_alignment *aln /* NULL or nq */);
int awry_map_device(const awry_index *index, int replica, const uint8_t *d_qbytes, const uint64_t *d_qoff, uint64_t nq,
                    uint32_t metric, uint32_t strands, uint32_t k, awry_mapping *d_out /* nq */,
                    awry_alignment *d_aln /* NULL or nq */, void *cuda_stream);

/* ------------------------------------------------------------------ streaming reads-file front-end
 * SURVEY.md 8(f) rank 4.  The reference's users parse their reads on the CPU and pass `&str`s to
 * parallel_count / parallel_locate (fm_index.rs:455-487); these entry points take the FASTQ ('@') or
 * FASTA ('>', sequences may span lines) file itself, plain or gzip-compressed: raw chunks are uploaded
 * from pinned memory while a reader thread fetches (or inflates) the next ones, and the records are split
 * on the device.  Read i of the file is query i.  Results are library-owned; release each pointer with awry_buffer_free
 * (hits: awry_hits_free).  On a handle with several replicas a plain file is cut into one segment per replica at
 * record starts found on the host and every replica parses and searches its own segment (a gzip stream cannot be
 * entered in the middle and stays on replica 0). */
int awry_count_reads_file(const awry_index *index, const char *path, uint64_t **counts,
                          uint64_t *n_reads);
int awry_locate_reads_file(const awry_index *index, const char *path, uint32_t flags,
                           uint64_t **hit_off /* n_reads + 1 */, awry_hit **hits, uint64_t *n_reads,
                           uint64_t *n_hits);
void awry_buffer_free(void *p);

/* ------------------------------------------------------------------ single steps (public in the reference) */

/* SearchRange::new / FmIndex::initial_search_range (search.rs:43-48, fm_index.rs:383) */
int awry_initial_range(const awry_index *index, uint8_t ascii_symbol, awry_range *out);
/* FmIndex::update_range_with_symbol (fm_index.rs:559-582); one-thread kernel launch */
int awry_update_range(const awry_index *index, awry_range range, uint8_t ascii_symbol,
                      awry_range *out);
/* FmIndex::backstep (fm_index.rs:585-593); one-thread kernel launch */
int awry_backstep(const awry_index *index, uint64_t bwt_row, uint64_t *out);

/* ------------------------------------------------------------------ device-resident entry points
 * Same kernels as the *_batch calls, for callers that already hold the queries in HBM
 * (bench.py's kernel-only figure).  Pointers are device pointers on replica `replica`'s
 * device; `cuda_stream` is a cudaStream_t (NULL = default stream).  The kernels are enqueued on that
 * stream and the call returns without waiting for them; it does read the first and last query offset
 * back first (16 bytes, one stream synchronisation) to size its scratch, so it is not capturable in a
 * CUDA graph. */
int awry_count_device(const awry_index *index, int replica, const uint8_t *d_qbytes,
                      const uint64_t *d_qoff, uint64_t nq, uint64_t *d_counts, void *cuda_stream);
/* two-pass locate on device-resident queries; results stay on the device.  Synchronises once
 * (the hit total sizes the output).  d_hit_off: nq+1 u64.  *d_hits is a device allocation
 * released with awry_device_free. */
int awry_locate_device(const awry_index *index, int replica, const uint8_t *d_qbytes,
                       const uint64_t *d_qoff, uint64_t nq, uint32_t flags, uint64_t *d_hit_off,
                       awry_hit **d_hits, uint64_t *n_hits, void *cuda_stream);
/* d_ptr came from the library's stream-ordered pool; the caller must have synchronised the stream that last
 * used it (the release itself is not ordered against the caller's streams). */
int awry_device_free(const awry_index *index, int replica, void *d_ptr);
/* The *_device calls are asynchronous, so an empty / sentinel-carrying query cannot be reported
 * by them; it is latched per replica.  This synchronises `cuda_stream`, returns
 * AWRY_ERR_INVALID_QUERY if any device batch since the last check held such a query (its result
 * slot is then 0 / SearchRange::zero()), and clears the latch. */
int awry_device_check(const awry_index *index, int replica, void *cuda_stream);

/* ------------------------------------------------------------------ instrumentation */

/* Per-kernel accounting kept by the library (CUDA events on the launching stream when
 * profiling is enabled): launches = number of this library's kernels launched since the last
 * reset; *_ms = summed device time of the dominant kernels. */
typedef struct awry_profile {
  uint64_t launches;
  uint64_t search_launches;
  double search_ms; /* backward-search kernel */
  uint64_t walk_launches;
  double walk_ms;   /* locate LF-walk kernel */
  uint64_t pack_launches;
  double pack_ms;   /* ASCII -> packed-symbol prepass */
  uint64_t h2d_bytes;
  uint64_t d2h_bytes;
} awry_profile;
int awry_profile_enable(int on);       /* event timing costs a sync per call: off by default */
int awry_profile_reset(void);
int awry_profile_get(awry_profile *out);

/* Random-gather roofline microbenchmark (SURVEY.md 8(d)): n_reads independent, uniformly random,
 * `granule`-byte aligned reads of `granule` bytes (32, 64 or 128) over a buffer of
 * `footprint_bytes`, `lanes` consecutive lanes cooperating on one granule (1, 2, 4 or 8).
 * Returns achieved reads/s and GB/s. */
int awry_bench_random_gather(int device, uint64_t footprint_bytes, uint32_t granule, uint32_t lanes,
                             uint64_t n_reads, int iters, double *reads_per_s, double *gb_per_s);

/* Tuning knob for experiments: selects the search-kernel variant.  lanes_per_query: 1/2/4 =
 * that many lanes on the one-symbol blocks, 8 = the two-symbol (pair index) kernels, -1 = scalar
 * kernel, 0 = default (pair index when it exists: the wave kernel where one-row intervals are finished in the
 * text -- see awry_set_count_variant -- else the refilling kernel); 80 = the refilling pair kernel (lane groups
 * draw a new query as soon as theirs ends), 81 / 82 (83 / 84: lower residency) = the same as a state machine
 * with 1 / 2 query slots per lane group.  blocks_per_sm caps residency (and selects the refilling kernel). */
int awry_set_search_variant(int lanes_per_query, int threads_per_block, int blocks_per_sm);

/* Count and locate pass 1, nucleotide.  Once backward search (fm_index.rs:402-438) has narrowed the interval to ONE row, the rest of
 * the query can only keep that row or empty the interval, and which of the two is decided by the text in front
 * of the occurrence.  When the index holds the unsampled suffix array and the text (4 bits per symbol, read back
 * out of BWT + suffix array at load time: bwt_len / 2 bytes, AWRY_B200_TEXT=0 never), the count kernel looks the
 * row's position up and compares the remaining symbols with the text -- 2-3 memory requests instead of one per
 * two symbols; counts are identical.  Locate does the same when its pass 2 is the gather from the unsampled array:
 * the hit of such a query is the text position itself.  variant 0 = do so when the arrays are present (default),
 * 1 = backward search to the last symbol. */
int awry_set_count_variant(int variant);

/* Locate pass 2.  Three ways to turn a BWT row into a text position, identical results:
 *   (a) the UNSAMPLED suffix array, rebuilt on the device at load time from the file's sampled one
 *       (compressed_suffix_array.rs:109-111) with one LF step per BWT row: a hit is one read of SA[row]
 *       instead of the LF-walk of fm_index.rs:521-537.  32 bits per row; kept when it takes < 1/3 of the free
 *       memory (AWRY_B200_FULL_SA=0 never, =1 whenever it fits);
 *   (b) nucleotide, when (a) is absent (or AWRY_B200_LEAN_SA=1): the suffix array sampled by TEXT POSITION
 *       (SA[row] % r == 0) with a mark bit per row, both derived at load time: an LF-walk of at most r - 1
 *       steps, 4.57 + 32/r bits per row (SURVEY 8(f) rank 3, without a new file format).  Being derived, r is
 *       the library's choice, not the file's: min(file ratio, 4), doubled until the arrays fit a third of the
 *       free device memory (AWRY_B200_LEAN_RATIO overrides);
 *   (c) the reference's own scheme: LF-walk to the next ROW the file sampled (geometric walk lengths).
 * variant 0 = the best one present (default), 1 = always (c), 2 = (b) if present, else (c). */
int awry_set_locate_variant(int variant);

/* Host-side query packing (nucleotide): the *_batch calls turn ASCII bases into 2-bit codes on the host
 * cores (AVX2/BMI2 or AVX-512BW, a process-wide thread pool: AWRY_B200_HOST_THREADS) while earlier
 * chunks are in flight, so a quarter of the bytes cross PCIe; bytes outside ACGT travel as a side list.
 * mode -1 = auto (on when the CPU supports it and the pool has >= 4 threads; AWRY_B200_HOST_PACK=0/1
 * overrides), 0 = always send ASCII, 1 = always pack. */
int awry_set_host_pack(int mode);
/* Threads the host-side packer may use (a process-wide pool shared by all calls and replicas; it grows on
 * demand).  Default: AWRY_B200_HOST_THREADS, else min(16, cores / LOCAL_WORLD_SIZE) -- one process per GPU
 * under torchrun shares the host; a process that drives several replicas itself should raise it to the
 * cores it owns.  n = 0 restores the default. */
int awry_set_host_threads(int n);
int awry_host_threads(void);
/* The packer itself (the producer of awry_*_batch_packed2's input): dst gets ceil(n/4) bytes, crumb i =
 * (src[i] >> 1) & 3 at bits 2*(i%4) of dst[i/4]; exceptions (up to exc_cap, ascending by i) receive
 * (i << 8) | src[i] for bytes outside ACGTacgt; *n_exc is their total number. */
int awry_host_pack_dna(const uint8_t *src, uint64_t n, uint8_t *dst, uint64_t *exceptions,
                       uint64_t exc_cap, uint64_t *n_exc);

const char *awry_last_error(void);
const char *awry_version(void);

#ifdef __cplusplus
}
#endif
#endif /* AWRY_B200_H */
