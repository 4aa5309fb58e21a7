// awry_b200.hpp -- header-only C++17 host mirror of the reference's Rust API over the C ABI.
//
// The reference is a Rust crate; no Rust toolchain exists in the build image, so this is the
// compiled-language host side that sits above include/awry_b200.h (the Rust facade under rust/
// is the same thing in the reference's own language).  Names, argument meaning and error
// behaviour follow /root/reference/src/fm_index.rs: where the reference returns io::Error this
// throws awry::Error; where it panics (empty query, sentinel in a query) this throws too.
#pragma once
#include <array>
#include <cstdint>
#include <stdexcept>
#include <string>
#include <string_view>
#include <utility>
#include <vector>

#include "awry_b200.h"

namespace awry {

struct Error : std::runtime_error {
  int code;
  Error(int c, const char* msg) : std::runtime_error(msg), code(c) {}
};

enum class SymbolAlphabet : uint32_t { Nucleotide = AWRY_NUCLEOTIDE, Amino = AWRY_AMINO };  // alphabet.rs:28-31

struct SearchRange {  // search.rs:25-81
  uint64_t start_ptr = 1, end_ptr = 0;
  static SearchRange zero() { return {1, 0}; }
  bool is_empty() const { return start_ptr > end_ptr; }
  uint64_t len() const { return is_empty() ? 0 : end_ptr - start_ptr + 1; }
};

struct LocalizedSequencePosition {  // sequence_index.rs:32-78
  uint64_t sequence_idx_ = 0, local_position_ = 0;
  uint64_t sequence_idx() const { return sequence_idx_; }
  uint64_t local_position() const { return local_position_; }
  bool operator==(const LocalizedSequencePosition& o) const {
    return sequence_idx_ == o.sequence_idx_ && local_position_ == o.local_position_;
  }
  bool operator<(const LocalizedSequencePosition& o) const {
    return sequence_idx_ != o.sequence_idx_ ? sequence_idx_ < o.sequence_idx_ : local_position_ < o.local_position_;
  }
};

struct FmBuildArgs {  // fm_index.rs:78-96; 0 = the reference's default (ratio 8, k 10 / 4)
  std::string input_file_src;
  uint64_t suffix_array_compression_ratio = 0;
  uint32_t lookup_table_kmer_len = 0;
  SymbolAlphabet alphabet = SymbolAlphabet::Nucleotide;
};

class FmIndex {
 public:
  // FmIndex::load (fm_index_file.rs:132)
  static FmIndex load(const std::string& path, const std::vector<int>& devices = {}) {
    awry_index* h = nullptr;
    check(awry_index_load(path.c_str(), devices.empty() ? nullptr : devices.data(), int(devices.size()), &h));
    return FmIndex(h);
  }
  // FmIndex::new (fm_index.rs:142-268) on the GPU; `save_to` non-empty = also FmIndex::save
  static FmIndex build(const FmBuildArgs& args, const std::vector<int>& devices = {}, const std::string& save_to = "") {
    awry_build_args a{};
    a.input_file_src = args.input_file_src.c_str();
    a.output_file_src = save_to.empty() ? nullptr : save_to.c_str();
    a.alphabet = uint32_t(args.alphabet);
    a.lookup_table_kmer_len = args.lookup_table_kmer_len;
    a.suffix_array_compression_ratio = args.suffix_array_compression_ratio;
    a.device = devices.empty() ? 0 : devices[0];
    awry_index* h = nullptr;
    check(awry_index_build(&a, devices.empty() ? nullptr : devices.data(), int(devices.size()), &h));
    return FmIndex(h);
  }
  // hand-over from the reference's CPU construction (FmIndex::new, fm_index.rs:142-268)
  static FmIndex from_parts(const awry_parts& parts, const std::vector<int>& devices = {}) {
    awry_index* h = nullptr;
    check(awry_index_from_parts(&parts, devices.empty() ? nullptr : devices.data(), int(devices.size()), &h));
    return FmIndex(h);
  }
  // FmIndex::save (fm_index_file.rs:42-106)
  void save(const std::string& path) const { check(awry_index_save(h_, path.c_str())); }
  FmIndex(FmIndex&& o) noexcept : h_(std::exchange(o.h_, nullptr)), info_(o.info_) {}
  FmIndex& operator=(FmIndex&& o) noexcept {
    if (this != &o) {
      awry_index_free(h_);
      h_ = std::exchange(o.h_, nullptr);
      info_ = o.info_;
    }
    return *this;
  }
  FmIndex(const FmIndex&) = delete;
  FmIndex& operator=(const FmIndex&) = delete;
  ~FmIndex() { awry_index_free(h_); }

  // getters (fm_index.rs:302-368)
  SymbolAlphabet alphabet() const { return SymbolAlphabet(info_.alphabet); }
  uint64_t suffix_array_compression_ratio() const { return info_.sa_ratio; }
  uint64_t bwt_len() const { return info_.bwt_len; }
  uint64_t version_number() const { return info_.version; }
  std::vector<uint64_t> prefix_sums() const {
    return std::vector<uint64_t>(info_.prefix_sums, info_.prefix_sums + info_.n_prefix_sums);
  }

  // fm_index.rs:383, :559-593
  SearchRange initial_search_range(char symbol) const {
    awry_range r;
    check(awry_initial_range(h_, uint8_t(symbol), &r));
    return {r.start_ptr, r.end_ptr};
  }
  SearchRange update_range_with_symbol(SearchRange range, char symbol) const {
    awry_range r;
    check(awry_update_range(h_, awry_range{range.start_ptr, range.end_ptr}, uint8_t(symbol), &r));
    return {r.start_ptr, r.end_ptr};
  }
  uint64_t backstep(uint64_t search_pointer) const {
    uint64_t out = 0;
    check(awry_backstep(h_, search_pointer, &out));
    return out;
  }

  // fm_index.rs:499-501, :516-544: batches of one
  uint64_t count_string(std::string_view query) const { return parallel_count({query})[0]; }
  std::vector<LocalizedSequencePosition> locate_string(std::string_view query) const {
    return parallel_locate({query})[0];
  }

  // fm_index.rs:455-460; input order preserved
  std::vector<uint64_t> parallel_count(const std::vector<std::string_view>& queries) const {
    std::vector<uint8_t> bytes;
    std::vector<uint64_t> off;
    pack(queries, bytes, off);
    std::vector<uint64_t> counts(queries.size());
    check(awry_count_batch(h_, bytes.data(), off.data(), queries.size(), counts.data()));
    return counts;
  }
  // fm_index.rs:479-487; per-query hits in BWT-row order (or sorted ascending)
  std::vector<std::vector<LocalizedSequencePosition>> parallel_locate(
      const std::vector<std::string_view>& queries, bool sorted = false) const {
    std::vector<uint8_t> bytes;
    std::vector<uint64_t> off;
    pack(queries, bytes, off);
    std::vector<uint64_t> hit_off(queries.size() + 1);
    awry_hit* hits = nullptr;
    uint64_t n = 0;
    check(awry_locate_batch(h_, bytes.data(), off.data(), queries.size(),
                            sorted ? AWRY_LOCATE_SORTED : AWRY_LOCATE_BWT_ORDER, hit_off.data(), &hits, &n));
    std::vector<std::vector<LocalizedSequencePosition>> out(queries.size());
    for (size_t q = 0; q < queries.size(); q++)
      for (uint64_t i = hit_off[q]; i < hit_off[q + 1]; i++) out[q].push_back({hits[i].seq_idx, hits[i].local_pos});
    awry_hits_free(hits);
    return out;
  }
  // Hamming search (no counterpart in the reference): windows within max_mismatches <= AWRY_HAMMING_MAX substitutions.
  // counts[q][d] = windows of query q at distance exactly d
  std::vector<std::vector<uint64_t>> parallel_count_hamming(const std::vector<std::string_view>& queries,
                                                            uint32_t max_mismatches) const {
    std::vector<uint8_t> bytes;
    std::vector<uint64_t> off;
    pack(queries, bytes, off);
    std::vector<uint64_t> flat(queries.size() * (size_t(max_mismatches) + 1));
    check(awry_count_batch_hamming(h_, bytes.data(), off.data(), queries.size(), max_mismatches, flat.data()));
    std::vector<std::vector<uint64_t>> out(queries.size());
    for (size_t q = 0; q < queries.size(); q++)
      out[q].assign(flat.begin() + q * (max_mismatches + 1), flat.begin() + (q + 1) * (max_mismatches + 1));
    return out;
  }
  // per query: (window start, distance), ascending by position
  std::vector<std::vector<std::pair<LocalizedSequencePosition, uint32_t>>> parallel_locate_hamming(
      const std::vector<std::string_view>& queries, uint32_t max_mismatches) const {
    std::vector<uint8_t> bytes;
    std::vector<uint64_t> off;
    pack(queries, bytes, off);
    std::vector<uint64_t> hit_off(queries.size() + 1);
    std::vector<awry_hit> hits(queries.size() + 1);
    std::vector<uint8_t> dist(hits.size());
    uint64_t n = 0;
    int rc = awry_locate_batch_hamming(h_, bytes.data(), off.data(), queries.size(), max_mismatches, hit_off.data(),
                                       hits.data(), dist.data(), hits.size(), &n);
    if (rc == AWRY_ERR_CAPACITY) {  // the total is known now: once more with room for every hit
      hits.resize(n);
      dist.resize(n);
      rc = awry_locate_batch_hamming(h_, bytes.data(), off.data(), queries.size(), max_mismatches, hit_off.data(),
                                     hits.data(), dist.data(), hits.size(), &n);
    }
    check(rc);
    std::vector<std::vector<std::pair<LocalizedSequencePosition, uint32_t>>> out(queries.size());
    for (size_t q = 0; q < queries.size(); q++)
      for (uint64_t i = hit_off[q]; i < hit_off[q + 1]; i++)
        out[q].push_back({{hits[i].seq_idx, hits[i].local_pos}, uint32_t(dist[i])});
    return out;
  }
  // Both strands (no counterpart in the reference): every query and its reverse complement.
  // counts[q] = {forward count, reverse-complement count}
  std::vector<std::array<uint64_t, 2>> parallel_count_strands(const std::vector<std::string_view>& queries) const {
    std::vector<uint8_t> bytes;
    std::vector<uint64_t> off;
    pack(queries, bytes, off);
    std::vector<std::array<uint64_t, 2>> out(queries.size());
    check(awry_count_batch_strands(h_, bytes.data(), off.data(), queries.size(), out.empty() ? nullptr : out[0].data()));
    return out;
  }
  // per query: {forward hits, reverse-strand hits (start of the window equal to the reverse complement)}, each in
  // BWT-row order (or sorted ascending)
  std::vector<std::array<std::vector<LocalizedSequencePosition>, 2>> parallel_locate_strands(
      const std::vector<std::string_view>& queries, bool sorted = false) const {
    std::vector<uint8_t> bytes;
    std::vector<uint64_t> off;
    pack(queries, bytes, off);
    const uint32_t flags = sorted ? AWRY_LOCATE_SORTED : AWRY_LOCATE_BWT_ORDER;
    std::vector<uint64_t> hit_off(2 * queries.size() + 1);
    std::vector<awry_hit> hits(2 * queries.size() + 1);
    uint64_t n = 0;
    int rc = awry_locate_batch_strands(h_, bytes.data(), off.data(), queries.size(), flags, hit_off.data(), hits.data(),
                                       hits.size(), &n);
    if (rc == AWRY_ERR_CAPACITY) {  // the total is known now: once more with room for every hit
      hits.resize(n);
      rc = awry_locate_batch_strands(h_, bytes.data(), off.data(), queries.size(), flags, hit_off.data(), hits.data(),
                                     hits.size(), &n);
    }
    check(rc);
    std::vector<std::array<std::vector<LocalizedSequencePosition>, 2>> out(queries.size());
    for (size_t v = 0; v < 2 * queries.size(); v++)
      for (uint64_t i = hit_off[v]; i < hit_off[v + 1]; i++) out[v / 2][v % 2].push_back({hits[i].seq_idx, hits[i].local_pos});
    return out;
  }
  // Hamming search on both strands: counts[q][s][d] = windows at distance exactly d from query q (s = 0) or from its
  // reverse complement (s = 1)
  std::vector<std::array<std::vector<uint64_t>, 2>> parallel_count_hamming_strands(
      const std::vector<std::string_view>& queries, uint32_t max_mismatches) const {
    std::vector<uint8_t> bytes;
    std::vector<uint64_t> off;
    pack(queries, bytes, off);
    const size_t P = size_t(max_mismatches) + 1;
    std::vector<uint64_t> flat(2 * queries.size() * P);
    check(awry_count_batch_hamming_strands(h_, bytes.data(), off.data(), queries.size(), max_mismatches, flat.data()));
    std::vector<std::array<std::vector<uint64_t>, 2>> out(queries.size());
    for (size_t v = 0; v < 2 * queries.size(); v++) out[v / 2][v % 2].assign(flat.begin() + v * P, flat.begin() + (v + 1) * P);
    return out;
  }
  // per query: {forward hits, reverse-strand hits}, each (window start, distance) ascending by position
  std::vector<std::array<std::vector<std::pair<LocalizedSequencePosition, uint32_t>>, 2>> parallel_locate_hamming_strands(
      const std::vector<std::string_view>& queries, uint32_t max_mismatches) const {
    std::vector<uint8_t> bytes;
    std::vector<uint64_t> off;
    pack(queries, bytes, off);
    std::vector<uint64_t> hit_off(2 * queries.size() + 1);
    std::vector<awry_hit> hits(2 * queries.size() + 1);
    std::vector<uint8_t> dist(hits.size());
    uint64_t n = 0;
    int rc = awry_locate_batch_hamming_strands(h_, bytes.data(), off.data(), queries.size(), max_mismatches,
                                               hit_off.data(), hits.data(), dist.data(), hits.size(), &n);
    if (rc == AWRY_ERR_CAPACITY) {  // the total is known now: once more with room for every hit
      hits.resize(n);
      dist.resize(n);
      rc = awry_locate_batch_hamming_strands(h_, bytes.data(), off.data(), queries.size(), max_mismatches,
                                             hit_off.data(), hits.data(), dist.data(), hits.size(), &n);
    }
    check(rc);
    std::vector<std::array<std::vector<std::pair<LocalizedSequencePosition, uint32_t>>, 2>> out(queries.size());
    for (size_t v = 0; v < 2 * queries.size(); v++)
      for (uint64_t i = hit_off[v]; i < hit_off[v + 1]; i++)
        out[v / 2][v % 2].push_back({{hits[i].seq_idx, hits[i].local_pos}, uint32_t(dist[i])});
    return out;
  }
  // Edit-distance search (no counterpart in the reference): text starts within max_edits <= AWRY_EDIT_MAX
  // substitutions, insertions and deletions.  counts[q][d] = starts of query q at distance exactly d
  std::vector<std::vector<uint64_t>> parallel_count_edit(const std::vector<std::string_view>& queries,
                                                         uint32_t max_edits) const {
    const size_t P = size_t(max_edits) + 1;
    const std::vector<uint64_t> flat = count_edit_flat(queries, max_edits, false);
    std::vector<std::vector<uint64_t>> out(queries.size());
    for (size_t q = 0; q < queries.size(); q++) out[q].assign(flat.begin() + q * P, flat.begin() + (q + 1) * P);
    return out;
  }
  // per query: (start, distance), ascending by position; the neighbouring starts of one locus are all there
  std::vector<std::vector<std::pair<LocalizedSequencePosition, uint32_t>>> parallel_locate_edit(
      const std::vector<std::string_view>& queries, uint32_t max_edits) const {
    return locate_edit_flat(queries, max_edits, false);
  }
  // both strands: counts[q][s][d] = starts at distance exactly d from query q (s = 0) or its reverse complement (s = 1)
  std::vector<std::array<std::vector<uint64_t>, 2>> parallel_count_edit_strands(
      const std::vector<std::string_view>& queries, uint32_t max_edits) const {
    const size_t P = size_t(max_edits) + 1;
    const std::vector<uint64_t> flat = count_edit_flat(queries, max_edits, true);
    std::vector<std::array<std::vector<uint64_t>, 2>> out(queries.size());
    for (size_t v = 0; v < 2 * queries.size(); v++) out[v / 2][v % 2].assign(flat.begin() + v * P, flat.begin() + (v + 1) * P);
    return out;
  }
  // per query: {forward hits, reverse-strand hits}, each (start, distance) ascending by position
  std::vector<std::array<std::vector<std::pair<LocalizedSequencePosition, uint32_t>>, 2>> parallel_locate_edit_strands(
      const std::vector<std::string_view>& queries, uint32_t max_edits) const {
    const auto flat = locate_edit_flat(queries, max_edits, true);
    std::vector<std::array<std::vector<std::pair<LocalizedSequencePosition, uint32_t>>, 2>> out(queries.size());
    for (size_t v = 0; v < flat.size(); v++) out[v / 2][v % 2] = flat[v];
    return out;
  }
  // Edit-distance loci (no counterpart in the reference): as the four calls above, but each occurrence once, at its
  // locus (include/awry_b200.h), not at every neighbouring start
  std::vector<std::vector<uint64_t>> parallel_count_edit_loci(const std::vector<std::string_view>& queries,
                                                              uint32_t max_edits) const {
    const size_t P = size_t(max_edits) + 1;
    const std::vector<uint64_t> flat = count_edit_flat(queries, max_edits, false, true);
    std::vector<std::vector<uint64_t>> out(queries.size());
    for (size_t q = 0; q < queries.size(); q++) out[q].assign(flat.begin() + q * P, flat.begin() + (q + 1) * P);
    return out;
  }
  std::vector<std::vector<std::pair<LocalizedSequencePosition, uint32_t>>> parallel_locate_edit_loci(
      const std::vector<std::string_view>& queries, uint32_t max_edits) const {
    return locate_edit_flat(queries, max_edits, false, true);
  }
  std::vector<std::array<std::vector<uint64_t>, 2>> parallel_count_edit_loci_strands(
      const std::vector<std::string_view>& queries, uint32_t max_edits) const {
    const size_t P = size_t(max_edits) + 1;
    const std::vector<uint64_t> flat = count_edit_flat(queries, max_edits, true, true);
    std::vector<std::array<std::vector<uint64_t>, 2>> out(queries.size());
    for (size_t v = 0; v < 2 * queries.size(); v++) out[v / 2][v % 2].assign(flat.begin() + v * P, flat.begin() + (v + 1) * P);
    return out;
  }
  std::vector<std::array<std::vector<std::pair<LocalizedSequencePosition, uint32_t>>, 2>> parallel_locate_edit_loci_strands(
      const std::vector<std::string_view>& queries, uint32_t max_edits) const {
    const auto flat = locate_edit_flat(queries, max_edits, true, true);
    std::vector<std::array<std::vector<std::pair<LocalizedSequencePosition, uint32_t>>, 2>> out(queries.size());
    for (size_t v = 0; v < flat.size(); v++) out[v / 2][v % 2] = flat[v];
    return out;
  }
  // Alignment of located hits (no counterpart in the reference): hit_off / hits as a locate_{hamming,edit}[_strands]
  // call with the same queries, metric (AWRY_METRIC_HAMMING / AWRY_METRIC_EDIT) and k returned them; one alignment per
  // hit (text_len, distance, the ops: see cigar)
  std::vector<awry_alignment> align_hits(const std::vector<std::string_view>& queries, uint32_t metric, uint32_t k,
                                         const std::vector<uint64_t>& hit_off, const std::vector<awry_hit>& hits,
                                         bool strands = false) const {
    std::vector<uint8_t> bytes;
    std::vector<uint64_t> off;
    pack(queries, bytes, off);
    std::vector<awry_alignment> out(hits.size());
    check(awry_align_batch(h_, bytes.data(), off.data(), queries.size(), metric, strands ? 1 : 0, k, hit_off.data(),
                           hits.data(), out.data()));
    return out;
  }
  // Read mapping (no counterpart in the reference): each query's best locus within k under `metric`, over both strands
  // or the query as given, with its uniqueness, mapping quality and (align) its alignment; second is empty unless align
  std::pair<std::vector<awry_mapping>, std::vector<awry_alignment>> parallel_map(const std::vector<std::string_view>& queries,
                                                                               uint32_t metric, uint32_t k,
                                                                               bool strands = true,
                                                                               bool align = true) const {
    std::vector<uint8_t> bytes;
    std::vector<uint64_t> off;
    pack(queries, bytes, off);
    std::pair<std::vector<awry_mapping>, std::vector<awry_alignment>> out;
    out.first.resize(queries.size());
    if (align) out.second.resize(queries.size());
    check(awry_map_batch(h_, bytes.data(), off.data(), queries.size(), metric, strands ? 1 : 0, k, out.first.data(),
                         align ? out.second.data() : nullptr));
    return out;
  }
  // the extended CIGAR (=, X, I, D) of one alignment of a query of length query_len, e.g. "47=1X102="
  static std::string cigar(const awry_alignment& a, uint32_t query_len) {
    size_t need = 0;
    const int rc = awry_alignment_cigar(&a, query_len, nullptr, 0, &need);
    if (rc != AWRY_ERR_CAPACITY) check(rc);
    std::string s(need, '\0');
    check(awry_alignment_cigar(&a, query_len, &s[0], s.size(), &need));
    s.resize(need - 1);
    return s;
  }
  awry_index* handle() const { return h_; }

 private:
  explicit FmIndex(awry_index* h) : h_(h) { check(awry_index_info(h_, &info_)); }
  // the edit calls' flat results: counts (nq or 2 nq) x (k+1), and the hits of each (virtual) query; `loci`: the
  // awry_*_edit_loci calls
  std::vector<uint64_t> count_edit_flat(const std::vector<std::string_view>& queries, uint32_t max_edits,
                                        bool strands, bool loci = false) const {
    std::vector<uint8_t> bytes;
    std::vector<uint64_t> off;
    pack(queries, bytes, off);
    std::vector<uint64_t> flat((strands ? 2 : 1) * queries.size() * (size_t(max_edits) + 1));
    if (loci)
      check(awry_count_batch_edit_loci(h_, bytes.data(), off.data(), queries.size(), strands ? 1 : 0, max_edits,
                                       flat.data()));
    else
      check((strands ? awry_count_batch_edit_strands : awry_count_batch_edit)(h_, bytes.data(), off.data(),
                                                                              queries.size(), max_edits, flat.data()));
    return flat;
  }
  std::vector<std::vector<std::pair<LocalizedSequencePosition, uint32_t>>> locate_edit_flat(
      const std::vector<std::string_view>& queries, uint32_t max_edits, bool strands, bool loci = false) const {
    std::vector<uint8_t> bytes;
    std::vector<uint64_t> off;
    pack(queries, bytes, off);
    const size_t nv = (strands ? 2 : 1) * queries.size();
    auto edit = strands ? awry_locate_batch_edit_strands : awry_locate_batch_edit;
    auto call = [&](const awry_index* h, const uint8_t* b, const uint64_t* o, uint64_t nq, uint32_t k, uint64_t* ho,
                    awry_hit* hs, uint8_t* d, uint64_t cap, uint64_t* n) {
      return loci ? awry_locate_batch_edit_loci(h, b, o, nq, strands ? 1 : 0, k, ho, hs, d, cap, n)
                  : edit(h, b, o, nq, k, ho, hs, d, cap, n);
    };
    std::vector<uint64_t> hit_off(nv + 1);
    std::vector<awry_hit> hits(nv + 1);
    std::vector<uint8_t> dist(hits.size());
    uint64_t n = 0;
    int rc = call(h_, bytes.data(), off.data(), queries.size(), max_edits, hit_off.data(), hits.data(), dist.data(),
                  hits.size(), &n);
    if (rc == AWRY_ERR_CAPACITY) {  // the total is known now: once more with room for every hit
      hits.resize(n);
      dist.resize(n);
      rc = call(h_, bytes.data(), off.data(), queries.size(), max_edits, hit_off.data(), hits.data(), dist.data(),
                hits.size(), &n);
    }
    check(rc);
    std::vector<std::vector<std::pair<LocalizedSequencePosition, uint32_t>>> out(nv);
    for (size_t v = 0; v < nv; v++)
      for (uint64_t i = hit_off[v]; i < hit_off[v + 1]; i++)
        out[v].push_back({{hits[i].seq_idx, hits[i].local_pos}, uint32_t(dist[i])});
    return out;
  }
  static void check(int rc) {
    if (rc != AWRY_OK) throw Error(rc, awry_last_error());
  }
  static void pack(const std::vector<std::string_view>& qs, std::vector<uint8_t>& bytes, std::vector<uint64_t>& off) {
    off.assign(1, 0);
    for (auto q : qs) {
      bytes.insert(bytes.end(), q.begin(), q.end());
      off.push_back(bytes.size());
    }
    if (bytes.empty()) bytes.push_back(0);
  }
  awry_index* h_ = nullptr;
  awry_info info_{};
};

}  // namespace awry
