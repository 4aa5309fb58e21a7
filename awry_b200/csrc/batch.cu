// batch.cu -- the batched count / locate pipelines of libawry_b200 and their entry points:
// parallel_count / parallel_locate (rayon map over queries, /root/reference/src/fm_index.rs:455-487) as
// chunked host -> device -> host pipelines per replica, plus the device-resident variants.
#include "host.hpp"

using namespace awry;
using namespace awry::host;

namespace awry {
namespace host {

// ------------------------------------------------------------------ batched pipelines

// AWRY_B200_TRACE=1: host-side stage times of the batched pipelines on stderr (scripts/locate_trace.py)
static bool trace_on() {
  static const bool on = getenv("AWRY_B200_TRACE") != nullptr;
  return on;
}
static void trace_mark(const char* what, long long i = -1) {
  if (!trace_on()) return;
  static const auto t_origin = std::chrono::steady_clock::now();
  fprintf(stderr, "[trace] %10.3f ms  %s %lld\n",
          std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_origin).count(), what, i);
}
// device-side timeline of a traced call: events recorded on the chunk streams, printed relative to the first
struct GpuTrace {
  struct Ev {
    cudaEvent_t e;
    const char* what;
    long long i;
  };
  std::vector<Ev> evs;
  void mark(cudaStream_t st, const char* what, long long i) {
    if (!trace_on()) return;
    cudaEvent_t e;
    if (cudaEventCreate(&e) != cudaSuccess) return;
    cudaEventRecord(e, st);
    evs.push_back(Ev{e, what, i});
  }
  void dump() {
    if (evs.empty()) return;
    for (auto& v : evs) cudaEventSynchronize(v.e);
    for (auto& v : evs) {
      float ms = 0;
      cudaEventElapsedTime(&ms, evs[0].e, v.e);
      fprintf(stderr, "[gpu]   %10.3f ms  %s %lld\n", ms, v.what, v.i);
    }
    for (auto& v : evs) cudaEventDestroy(v.e);
    evs.clear();
  }
};
static thread_local GpuTrace* g_gpu_trace = nullptr;
static void gpu_mark(cudaStream_t st, const char* what, long long i) {
  if (g_gpu_trace) g_gpu_trace->mark(st, what, i);
}

bool is_pinned(const void* p) {
  cudaPointerAttributes a;
  if (cudaPointerGetAttributes(&a, p) != cudaSuccess) {
    cudaGetLastError();
    return false;
  }
  return a.type == cudaMemoryTypeHost;
}

void parallel_memcpy(void* dst, const void* src, size_t n) {
  const size_t MIN_PER_THREAD = 8u << 20;
  unsigned hw = std::max(1u, std::thread::hardware_concurrency());
  unsigned nt = unsigned(std::min<size_t>(std::min(hw, 16u), n / MIN_PER_THREAD));
  if (nt <= 1) {
    memcpy(dst, src, n);
    return;
  }
  std::vector<std::thread> th;
  for (unsigned t = 0; t < nt; t++) {
    size_t lo = n * t / nt, hi = n * (t + 1) / nt;
    th.emplace_back([=] { memcpy(static_cast<char*>(dst) + lo, static_cast<const char*>(src) + lo, hi - lo); });
  }
  for (auto& x : th) x.join();
}

// Pipeline chunk: small enough that the exposed first upload / last kernel are a few percent of a
// 10 M-read batch, large enough (~0.9 M reads) to keep the persistent search grid busy.
constexpr uint64_t CHUNK_MAX_Q = 1u << 20;  // queries per pipeline chunk
uint64_t chunk_max_bytes() {                 // query bytes per pipeline chunk (AWRY_B200_CHUNK_MB, default 128)
  static const uint64_t v = [] {
    uint64_t mb = 128;
    if (const char* e = getenv("AWRY_B200_CHUNK_MB")) mb = std::min<uint64_t>(1024, std::max<uint64_t>(1, strtoull(e, nullptr, 10)));
    return mb << 20;
  }();
  return v;
}

struct Chunk {
  uint64_t q0, q1, b0, b1;
};

// `ramp_from` > 0: the first chunk holds about that many bytes and every following one up to 1.4 x its
// predecessor, until max_bytes is reached (see shaped_chunks).
std::vector<Chunk> make_chunks(const uint64_t* qoff, uint64_t q_lo, uint64_t q_hi, uint64_t max_q, uint64_t max_bytes,
                               uint64_t ramp_from = 0) {
  std::vector<Chunk> out;
  uint64_t q = q_lo;
  double cap = ramp_from ? double(std::min(ramp_from, max_bytes)) : double(max_bytes);
  while (q < q_hi) {
    const uint64_t cap_bytes = uint64_t(cap);
    uint64_t hi = std::min(q_hi, q + max_q);
    // largest hi with qoff[hi] - qoff[q] <= cap_bytes (at least one query)
    if (qoff[hi] - qoff[q] > cap_bytes) {
      uint64_t lo2 = q + 1, hi2 = hi;
      while (lo2 < hi2) {
        uint64_t mid = (lo2 + hi2 + 1) / 2;
        if (qoff[mid] - qoff[q] <= cap_bytes)
          lo2 = mid;
        else
          hi2 = mid - 1;
      }
      hi = lo2;
    }
    out.push_back(Chunk{q, hi, qoff[q], qoff[hi]});
    q = hi;
    cap = std::min(double(max_bytes), cap * 1.4);
  }
  return out;
}

// Pipeline fill and drain: the device idles while the host prepares the first chunk, and the host idles while the
// device works on the last one.  ASCII input (the host packs every chunk before its copy): the first chunk is split
// into 1/4 + 3/4 and the last into 1/2 + 1/4 + 1/4 (by queries).  A finer ramp -- 16 MB first, every chunk 1.4 x its
// predecessor -- was measured and LOSES there (21.0-21.5 against 19.9 ms per 10 M reads,
// profiles/r02_s6_count_e2e_trace.log): packing and copying chunk i + 1 one after the other takes longer than
// searching chunk i, so the device waits a little at every step of the ramp instead of once, and chunks of 0.1-0.4 M
// reads run the persistent search kernel at 2.0-2.4 ms per M reads instead of 1.8.  Pre-packed input has no host
// pass; there the ramp wins (19.0-19.3 -> 18.5 ms) and is used (`ramp`).
std::vector<Chunk> shaped_chunks(const uint64_t* qoff, uint64_t q_lo, uint64_t q_hi, uint64_t max_q, uint64_t max_bytes,
                                 bool ramp) {
  const uint64_t total = qoff[q_hi] >= qoff[q_lo] ? qoff[q_hi] - qoff[q_lo] : 0;
  const uint64_t RAMP_FROM = 16u << 20, MIN_SPLIT = 64u << 20;  // (only chunks worth splitting are split)
  std::vector<Chunk> in = make_chunks(qoff, q_lo, q_hi, max_q, max_bytes, ramp && total >= 3 * RAMP_FROM ? RAMP_FROM : 0);
  if (in.size() < 3) return in;
  auto split = [&](const Chunk& c, std::initializer_list<double> cuts, std::vector<Chunk>& dst) {
    uint64_t nq = c.q1 - c.q0, prev = c.q0;
    for (double f : cuts) {
      uint64_t at = c.q0 + uint64_t(double(nq) * f);
      if (at > prev && at < c.q1) {
        dst.push_back(Chunk{prev, at, qoff[prev], qoff[at]});
        prev = at;
      }
    }
    dst.push_back(Chunk{prev, c.q1, qoff[prev], qoff[c.q1]});
  };
  std::vector<Chunk> out;
  if (!ramp && in.front().b1 - in.front().b0 >= MIN_SPLIT)
    split(in.front(), {0.25}, out);
  else
    out.push_back(in.front());
  for (size_t i = 1; i + 1 < in.size(); i++) out.push_back(in[i]);
  if (in.back().b1 - in.back().b0 >= MIN_SPLIT)
    split(in.back(), {0.5, 0.75}, out);
  else
    out.push_back(in.back());
  return out;
}

bool host_pack_enabled() {
  const int hp = g_host_pack.load(std::memory_order_relaxed);
  if (hp >= 0) return hp == 1 && host_pack_supported();
  static const bool on = [] {
    if (const char* e = getenv("AWRY_B200_HOST_PACK")) return e[0] != '0' && host_pack_supported();
    return host_pack_supported() && host_pool_threads() >= 4;
  }();
  return on;
}

// Where a batch's queries come from: ASCII bytes (the reference's `&str`s), or 2-bit codes the caller holds
// already (awry_*_batch_packed2: crumb of byte position p at bits 2*(p%4) of crumbs[p/4], exceptions sorted
// by position) -- then the host packer has nothing to do and a quarter of the bytes cross PCIe.
struct QuerySource {
  const uint8_t* qbytes = nullptr;
  const uint8_t* crumbs = nullptr;
  const uint64_t* exc = nullptr;  // ((position) << 8) | byte, ascending
  uint64_t n_exc = 0;
  const uint64_t* qoff = nullptr;
  bool pinned = false;  // bytes / crumbs and offsets are page-locked: the copy engine reads them in place
  bool strands = false;  // nucleotide, both strands: query q is searched as the virtual queries 2q and 2q + 1 (its
                         // reverse complement), whose results and CSR entries the outputs hold
  uint64_t per_query() const { return strands ? 2 : 1; }  // virtual queries (result slots) per query
};

// The chunker binary-searches the offsets and sizes every buffer from a chunk's byte range, so the ends of
// every chunk are checked here (a non-monotone array can make b1 < b0 or a chunk absurdly large); inside a
// chunk each query is checked against [b0, b1] on the device before it is touched (pack kernels).
void validate_chunks(const std::vector<Chunk>& chunks, uint64_t max_bytes) {
  for (const Chunk& c : chunks) {
    if (c.b1 < c.b0) fail(AWRY_ERR_INVALID_ARG, "query offsets are not monotone (queries %llu..%llu)",
                          (unsigned long long)c.q0, (unsigned long long)c.q1);
    // one query may exceed the chunk budget; several may not
    if (c.b1 - c.b0 > max_bytes && c.q1 - c.q0 > 1)
      fail(AWRY_ERR_INVALID_ARG, "query offsets are not monotone (queries %llu..%llu)", (unsigned long long)c.q0,
           (unsigned long long)c.q1);
    if (c.b1 - c.b0 >= (1ull << 32)) fail(AWRY_ERR_INVALID_ARG, "query %llu is longer than 4 GiB", (unsigned long long)c.q0);
  }
}

// Sequencer reads are all the same length: then a chunk's offsets are first + i * len and the device writes them
// itself (8 bytes per read that do not cross the link: 80 MB of the 455 MB a 10 M x 150-bp batch of packed reads
// uploads).  Checked exactly, on the pool, per chunk; AWRY_B200_UNIFORM_OFFSETS=0 always copies.
bool offsets_are_uniform(const uint64_t* off, uint64_t nq, uint64_t& len) {
  static const bool on = [] {
    const char* e = getenv("AWRY_B200_UNIFORM_OFFSETS");
    return !(e && e[0] == '0');
  }();
  if (!on || nq < 4096) return false;
  len = off[1] - off[0];
  if (off[1] < off[0] || len == 0 || len >= (1ull << 32) || off[nq] - off[0] != len * nq) return false;
  const uint64_t BLK = 1u << 16, nb = (nq + BLK - 1) / BLK, first = off[0], l = len;
  std::atomic<bool> ok{true};
  host_parallel_blocks(size_t(nb), [&](size_t b) {
    if (!ok.load(std::memory_order_relaxed)) return;
    const uint64_t lo = b * BLK, hi = std::min(nq, lo + BLK);
    uint64_t bad = 0;
    for (uint64_t i = lo; i <= hi; i++) bad |= off[i] ^ (first + i * l);
    if (bad) ok.store(false, std::memory_order_relaxed);
  });
  return ok.load();
}

// u64 words of a packed-query buffer for n queries whose offsets lie in [b_lo, b_hi]: query q starts at word
// 4 * (q + (qoff[q] >> sh)) - 4 * (b_lo >> sh) (kernels.hpp)
uint64_t query_words(int alphabet, uint64_t n, uint64_t b_lo, uint64_t b_hi) {
  const int sh = packed_unit_shift(alphabet);
  return 4 * (n + (b_hi >> sh) - (b_lo >> sh) + 2) + 32;
}

// What one search_reads call works in, all sized by the caller: `words` (query_words of the reads), for both strands
// also `voff` (2 nq + 1) and `vwords` (query_words of the virtual queries on [2 b_lo, 2 b_hi]); `out` and `defer`
// for the searched queries; `flag` latches what the prepass refuses.
struct SearchBuffers {
  uint64_t* words;
  uint64_t* voff;
  uint64_t* vwords;
  void* out;
  uint32_t* defer;
  unsigned long long* flag;
};

// ws's buffers for search_reads of nq reads on [b_lo, b_hi], `out_elem` bytes of result per searched query, grown as
// needed
SearchBuffers workspace_buffers(Workspace* ws, int alphabet, uint64_t nq, uint64_t b_lo, uint64_t b_hi, bool strands,
                                size_t out_elem, unsigned long long* flag) {
  const uint64_t nv = strands ? 2 * nq : nq;
  Workspace::grow_dev(ws->d_qwords, ws->d_qwords_cap, size_t(query_words(alphabet, nq, b_lo, b_hi)));
  Workspace::grow_dev(ws->d_out, ws->d_out_cap, size_t(nv) * out_elem);
  Workspace::grow_dev(ws->d_defer, ws->d_defer_cap, defer_words(nv));
  if (strands) {
    Workspace::grow_dev(ws->d_voff, ws->d_voff_cap, size_t(nv) + 1);
    Workspace::grow_dev(ws->d_vwords, ws->d_vwords_cap, size_t(query_words(AWRY_NUCLEOTIDE, nv, 2 * b_lo, 2 * b_hi)));
  }
  return SearchBuffers{ws->d_qwords, ws->d_voff, ws->d_vwords, ws->d_out, ws->d_defer, flag};
}

// Searches nq reads that are on the device, on one strand or both (the 2 nq virtual queries of kernels.hpp), into
// b.out, on stream `st`.  Their offsets are absolute and lie in [b_lo, b_hi].  d_qbytes: their ASCII bytes, biased
// accordingly -- the wave kernel packs them itself where it runs, launch_pack does otherwise; nullptr: b.words holds
// their words already (launch_pack2).  The pack runs under profile slot 2 and the search under slot 0, the strand
// kernels under neither; t0 / t1 (if set) are recorded around the search launch alone (PackBalance).  Returns
// whether one-hit queries were stored as text positions (SearchVariant::locate_positions).
bool search_reads(Replica& r, const uint8_t* d_qbytes, const uint64_t* d_qoff, uint64_t nq, uint64_t b_lo, uint64_t b_hi,
                  bool strands, SearchOut mode, const SearchBuffers& b, cudaStream_t st, cudaEvent_t t0 = nullptr,
                  cudaEvent_t t1 = nullptr, long long trace_i = -1) {
  const int alphabet = int(r.view.alphabet);
  uint64_t* const words = b.words - 4 * (b_lo >> packed_unit_shift(alphabet));
  SearchVariant v = current_variant();
  v.avg_len = uint32_t(std::min<uint64_t>((b_hi - b_lo) / std::max<uint64_t>(1, nq), 1u << 30));
  v.b_lo = b_lo;
  v.b_hi = b_hi;
  v.locate_positions = mode == OUT_SP_CNT_U32 && locate_positions_ok(r.view, v);
  const bool in_wave = d_qbytes && (strands ? search_strands_ascii(r.view, mode, v) : search_packs_ascii(r.view, mode, v));
  if (d_qbytes && !in_wave) {
    ProfScope p(2, r.device, st);
    CU(launch_pack(alphabet, d_qbytes, d_qoff, nq, words, b_lo, b_hi, b.flag, st));
  }
  const uint64_t* qoff = d_qoff;
  uint64_t* qwords = words;
  uint64_t n = nq;
  if (strands) {  // the strand wave kernel stages the virtual queries from the bytes itself
    qwords = b.vwords - 4 * ((2 * b_lo) >> 6);
    CU(launch_strand_offsets(d_qoff, nq, b_lo, b_hi, b.voff, st));
    if (!in_wave) CU(launch_strand_words(words, d_qoff, nq, b_lo, b_hi, b.voff, qwords, st));
    qoff = b.voff;
    n = 2 * nq;
    v.b_lo = 2 * b_lo;
    v.b_hi = 2 * b_hi;
  }
  gpu_mark(st, "packed on device", trace_i);
  ProfScope p(0, r.device, st);
  if (t0) CU(cudaEventRecord(t0, st));
  if (in_wave)
    CU(launch_search_ascii(r.view, d_qbytes, qoff, n, qwords, b.flag, mode, b.out, b.defer, v, r.sm_count, st, strands));
  else
    CU(launch_search(r.view, qwords, qoff, n, mode, b.out, b.defer, v, r.sm_count, st));
  if (t1) CU(cudaEventRecord(t1, st));
  return v.locate_positions;
}

// Uploads one chunk of queries and runs prepass + search on ws->st.  The search result lands
// in ws->d_out in the requested mode.
// `may_pack`: the caller's say on host packing for this chunk (PackBalance)
// `d_out_override`: where the search result goes instead of ws->d_out (a call-level array the chunks fill).
void enqueue_search(const awry_index* ix, Replica& r, PackBalance& bal, Workspace* ws, const QuerySource& qs,
                    const Chunk& c, SearchOut mode, bool may_pack = true, bool probe_link = false, bool copy_flag = true,
                    void* d_out_override = nullptr) {
  const uint64_t nq = c.q1 - c.q0, nbytes = c.b1 - c.b0;
  const size_t out_elem = mode == OUT_COUNT_U64 ? 8 : mode == OUT_RANGE_U64 ? 16 : sp_cnt_bytes(r.view);
  Workspace::grow_dev(ws->d_qbytes, ws->d_qbytes_cap, size_t(nbytes) + 16);
  Workspace::grow_dev(ws->d_qoff, ws->d_qoff_cap, size_t(nq) + 1);
  SearchBuffers b = workspace_buffers(ws, ix->alphabet, nq, c.b0, c.b1, qs.strands, out_elem, ws->d_flag);
  if (d_out_override) b.out = d_out_override;
  const uint64_t* src_o = qs.qoff + c.q0;
  const uint8_t* d_ascii = nullptr;  // the chunk's ASCII bytes on the device (nullptr: launch_pack2 wrote its words)
  ws->link_probe_bytes = 0;
  uint64_t uni_len = 0;
  const bool uniform = offsets_are_uniform(src_o, nq, uni_len);
  auto upload_offsets = [&] {
    if (uniform) {
      CU(launch_fill_offsets(ws->d_qoff, c.b0, uni_len, nq, ws->st));
    } else {
      CU(cudaMemcpyAsync(ws->d_qoff, src_o, (nq + 1) * 8, cudaMemcpyHostToDevice, ws->st));
      g_prof.h2d += (nq + 1) * 8;
    }
  };
  auto stage_offsets = [&] {  // pageable offsets: staged through pinned memory
    if (qs.pinned || uniform) return;
    Workspace::grow_host(ws->h_qoff, ws->h_qoff_cap, size_t(nq) + 1);
    parallel_memcpy(ws->h_qoff, src_o, (nq + 1) * 8);
    src_o = ws->h_qoff;
  };
  // 2-bit crumbs up, `base` the query byte the first one stands for, and launch_pack2 writes the words; the exceptions
  // carry their position relative to `exc_base`.  Pageable crumbs and exceptions are staged through pinned memory.
  auto upload_crumbs = [&](const uint8_t* src_c, bool pinned, size_t cbytes, uint64_t base, const uint64_t* src_e,
                           size_t n_exc, uint64_t exc_base) {
    stage_offsets();
    if (!pinned) {
      Workspace::grow_host(ws->h_qbytes, ws->h_qbytes_cap, cbytes + 64);
      parallel_memcpy(ws->h_qbytes, src_c, cbytes);
      src_c = ws->h_qbytes;
    }
    if (cbytes) CU(cudaMemcpyAsync(ws->d_qbytes, src_c, cbytes, cudaMemcpyHostToDevice, ws->st));
    upload_offsets();
    if (n_exc) {
      Workspace::grow_dev(ws->d_exc, ws->d_exc_cap, n_exc);
      if (!pinned) {
        Workspace::grow_host(ws->h_exc, ws->h_exc_cap, n_exc);
        memcpy(ws->h_exc, src_e, n_exc * 8);
        src_e = ws->h_exc;
      }
      CU(cudaMemcpyAsync(ws->d_exc, src_e, n_exc * 8, cudaMemcpyHostToDevice, ws->st));
    }
    g_prof.h2d += cbytes + n_exc * 8;
    gpu_mark(ws->st, "h2d done", (long long)c.q0);
    CU(cudaMemsetAsync(ws->d_flag, 0xff, 8, ws->st));
    ProfScope p(2, r.device, ws->st);
    CU(launch_pack2(reinterpret_cast<const uint32_t*>(ws->d_qbytes), base, ws->d_qoff, nq,
                    b.words - 4 * (c.b0 >> packed_unit_shift(ix->alphabet)), ws->d_exc, n_exc, exc_base, c.b0, c.b1, ws->d_flag,
                    ws->st));
  };
  if (qs.crumbs) {
    // pre-packed by the caller: bytes [b0/4, ceil(b1/4)) of the crumb array, exceptions of [b0, b1)
    const uint64_t cb0 = c.b0 >> 2, cb1 = (c.b1 + 3) >> 2;
    const uint64_t* e_lo = std::lower_bound(qs.exc, qs.exc + qs.n_exc, c.b0 << 8);
    const uint64_t* e_hi = std::lower_bound(e_lo, qs.exc + qs.n_exc, c.b1 << 8);
    upload_crumbs(qs.crumbs + cb0, qs.pinned, size_t(cb1 - cb0), cb0 << 2, e_lo, size_t(e_hi - e_lo), 0);
  } else {
    const uint8_t* src_b = qs.qbytes + c.b0;
    // Nucleotide chunks are packed to 2 bits per base by the host cores before the copy (a quarter of
    // the PCIe bytes; works the same for pageable and pinned caller memory).  Chunks with many bytes
    // outside ACGT go up as ASCII.
    bool packed = false;
    if (may_pack && ix->alphabet == AWRY_NUCLEOTIDE && host_pack_enabled() && nbytes >= 4096) {
      Workspace::grow_host(ws->h_qbytes, ws->h_qbytes_cap, size_t(nbytes) / 4 + 64);
      auto t0 = std::chrono::steady_clock::now();
      int sharers = 1;
      packed = host_pack_dna(src_b, size_t(nbytes), ws->h_qbytes, ws->exc_tmp, 64, 0, &sharers);
      if (packed)
        bal.note_host(double(nbytes), std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count(), sharers);
      trace_mark("  host pack done, bytes", (long long)nbytes);
    }
    if (packed) {  // the crumbs are in pinned memory already; the exceptions join them there
      const size_t n_exc = ws->exc_tmp.size();
      Workspace::grow_host(ws->h_exc, ws->h_exc_cap, n_exc);
      if (n_exc) memcpy(ws->h_exc, ws->exc_tmp.data(), n_exc * 8);
      upload_crumbs(ws->h_qbytes, true, (size_t(nbytes) + 3) / 4 + 8, c.b0, ws->h_exc, n_exc, c.b0);
    } else {
      if (!qs.pinned) {
        Workspace::grow_host(ws->h_qbytes, ws->h_qbytes_cap, size_t(nbytes) + 16);
        parallel_memcpy(ws->h_qbytes, src_b, nbytes);
        src_b = ws->h_qbytes;
      }
      stage_offsets();
      const bool probe = probe_link && qs.pinned && nbytes >= (8u << 20);
      if (probe) {
        if (!ws->ev_a) {
          CU(cudaEventCreate(&ws->ev_a));
          CU(cudaEventCreate(&ws->ev_b));
        }
        CU(cudaEventRecord(ws->ev_a, ws->st));
      }
      if (nbytes) CU(cudaMemcpyAsync(ws->d_qbytes, src_b, nbytes, cudaMemcpyHostToDevice, ws->st));
      if (probe) {
        CU(cudaEventRecord(ws->ev_b, ws->st));
        ws->link_probe_bytes = nbytes;
      }
      upload_offsets();
      g_prof.h2d += nbytes;
      CU(cudaMemsetAsync(ws->d_flag, 0xff, 8, ws->st));
      d_ascii = ws->d_qbytes - c.b0;  // offsets stay absolute: the kernels subtract the chunk's byte base
    }
  }
  ws->gpu_probe_bytes = 0;
  const bool time_kernel = qs.pinned && !qs.crumbs && nbytes >= (8u << 20);  // PackBalance: what the GPU consumes
  if (time_kernel && !ws->ev_s0) {
    CU(cudaEventCreate(&ws->ev_s0));
    CU(cudaEventCreate(&ws->ev_s1));
  }
  // (remembered for locate_chunk_walk: pass 2 must then be the gather from the unsampled array)
  ws->sp_cnt_positions = search_reads(r, d_ascii, ws->d_qoff, nq, c.b0, c.b1, qs.strands, mode, b, ws->st,
                                      time_kernel ? ws->ev_s0 : nullptr, time_kernel ? ws->ev_s1 : nullptr, (long long)c.q0);
  if (time_kernel) ws->gpu_probe_bytes = nbytes;
  gpu_mark(ws->st, "searched", (long long)c.q0);
  // (the locate pipeline copies the flag together with the hit total, after the scan: one hand-over between
  // the compute and copy engines per chunk instead of two)
  if (copy_flag) CU(cudaMemcpyAsync(ws->h_flag, ws->d_flag, 8, cudaMemcpyDeviceToHost, ws->st));
  trace_mark("  search enqueued, queries", (long long)nq);
}

[[noreturn]] void fail_bad_query(unsigned long long code, uint64_t q_base) {
  const unsigned long long q = q_base + (code >> 1);
  if ((code & 1) == BAD_OFFSETS)
    fail(AWRY_ERR_INVALID_ARG, "query offsets are not monotone at query %llu (its bytes lie outside the batch)", q);
  fail(AWRY_ERR_INVALID_QUERY,
       "query %llu is empty or contains a sentinel ('$'/'#'): the reference panics on it "
       "(fm_index.rs:406, bwt.rs:127)", q);
}

void check_flag(Workspace* ws, const Chunk& c) {
  if (*ws->h_flag != ~0ull) fail_bad_query(*ws->h_flag, c.q0);
}

// count / range search over [q_lo, q_hi) on one replica, 3-deep pipeline
void search_on_replica(const awry_index* ix, size_t ri, const QuerySource& qs, uint64_t q_lo, uint64_t q_hi,
                       SearchOut mode, void* out, size_t n_active_replicas = 1) {
  if (q_lo >= q_hi) return;
  Replica& r = *ix->reps[ri];
  PackBalance& bal = ix->balance_of(ri);
  DeviceGuard dg(r.device);
  const size_t out_elem = (mode == OUT_COUNT_U64 ? 8 : 16) * qs.per_query();  // per query
  const uint64_t* qoff = qs.qoff;
  const bool src_pinned = qs.pinned;
  const bool dst_pinned = is_pinned(out);
  // pre-packed queries are a quarter of the bytes: four times the reads per chunk keep the chunk count down
  const uint64_t max_bytes = chunk_max_bytes() * (qs.crumbs ? 2 : 1);
  if (qoff[q_hi] < qoff[q_lo]) fail(AWRY_ERR_INVALID_ARG, "query offsets are not monotone (queries %llu..%llu)",
                                     (unsigned long long)q_lo, (unsigned long long)q_hi);
  auto chunks = shaped_chunks(qoff, q_lo, q_hi, CHUNK_MAX_Q, max_bytes, qs.crumbs != nullptr);
  validate_chunks(chunks, max_bytes);
  constexpr int DEPTH = 3;
  Workspace* ws[DEPTH] = {nullptr, nullptr, nullptr};
  int pending[DEPTH] = {-1, -1, -1};
  auto finish = [&](int s) {
    if (pending[s] < 0) return;
    const Chunk& c = chunks[size_t(pending[s])];
    CU(cudaEventSynchronize(ws[s]->done));
    if (ws[s]->link_probe_bytes) {
      float ms = 0;
      if (cudaEventElapsedTime(&ms, ws[s]->ev_a, ws[s]->ev_b) == cudaSuccess)
        bal.note_link(double(ws[s]->link_probe_bytes), double(ms) * 1e-3);
      ws[s]->link_probe_bytes = 0;
    }
    if (ws[s]->gpu_probe_bytes) {
      float ms = 0;
      if (cudaEventElapsedTime(&ms, ws[s]->ev_s0, ws[s]->ev_s1) == cudaSuccess)
        bal.note_gpu(double(ws[s]->gpu_probe_bytes), double(ms) * 1e-3);
      ws[s]->gpu_probe_bytes = 0;
    }
    check_flag(ws[s], c);
    if (!dst_pinned)
      parallel_memcpy(static_cast<char*>(out) + c.q0 * out_elem, ws[s]->h_out, (c.q1 - c.q0) * out_elem);
    pending[s] = -1;
  };
  GpuTrace gpu_trace;  // AWRY_B200_TRACE=1: device-side timeline of the chunk pipeline on stderr
  g_gpu_trace = trace_on() ? &gpu_trace : nullptr;
  uint64_t bytes_total = 0, bytes_packed = 0;  // of the chunks enqueued so far (pinned sources only)
  const bool balanced = src_pinned && !qs.crumbs && ix->alphabet == AWRY_NUCLEOTIDE && host_pack_enabled();
  PackBalance::Plan plan{1.0, false, false};
  if (balanced) plan = bal.plan(n_active_replicas);
  try {
    for (size_t i = 0; i < chunks.size(); i++) {
      int s = int(i % DEPTH);
      if (!ws[s]) ws[s] = r.acquire();
      finish(s);
      const Chunk& c = chunks[i];
      bool may_pack = true, probe = false;
      if (balanced) {
        if (i == 0 && plan.probe_link && chunks.size() > 1) {
          may_pack = false;  // nothing else is in flight: the cleanest moment to time the link
          probe = true;
        } else if (i == 1 && plan.probe_host) {
          may_pack = true;
        } else {
          // a chunk goes up as it is as soon as the raw share is behind plan: raw chunks sit early in the batch,
          // where the host packs the following chunks while they cross the link, not at its end, where the host
          // would idle behind them (measured effect: none on a host whose memory system is the limit -- 15.4-15.9 ms
          // per 10 M reads for every share from 0.7 to 1.0, profiles/r02_s10_e2e_share_sweep.log)
          may_pack = !(double(bytes_total - bytes_packed) < (1.0 - plan.share) * double(bytes_total + (c.b1 - c.b0)));
        }
        bytes_total += c.b1 - c.b0;
        if (may_pack) bytes_packed += c.b1 - c.b0;
      }
      enqueue_search(ix, r, bal, ws[s], qs, c, mode, may_pack, probe);
      size_t bytes = (c.q1 - c.q0) * out_elem;
      void* dst = static_cast<char*>(out) + c.q0 * out_elem;
      if (!dst_pinned) {
        Workspace::grow_host(ws[s]->h_out, ws[s]->h_out_cap, bytes);
        dst = ws[s]->h_out;
      }
      CU(cudaMemcpyAsync(dst, ws[s]->d_out, bytes, cudaMemcpyDeviceToHost, ws[s]->st));
      gpu_mark(ws[s]->st, "results copied", (long long)c.q0);
      g_prof.d2h += bytes;
      CU(cudaEventRecord(ws[s]->done, ws[s]->st));
      pending[s] = int(i);
    }
    for (int s = 0; s < DEPTH; s++) finish(s);
    g_gpu_trace = nullptr;
    gpu_trace.dump();
  } catch (...) {
    g_gpu_trace = nullptr;
    for (int s = 0; s < DEPTH; s++)
      if (ws[s]) {
        cudaStreamSynchronize(ws[s]->st);
        r.release(ws[s]);
      }
    throw;
  }
  for (int s = 0; s < DEPTH; s++)
    if (ws[s]) r.release(ws[s]);
}

// splits [0,nq) across replicas by query bytes; one host thread per replica
template <class F>
void for_each_replica_range(const awry_index* ix, const uint64_t* qoff, uint64_t nq, F&& fn) {
  size_t nr = ix->reps.size();
  if (nr == 1 || nq < 2 * nr) {
    fn(0, 0, nq);
    return;
  }
  std::vector<uint64_t> cut(nr + 1, 0);
  cut[nr] = nq;
  uint64_t total = qoff[nq] - qoff[0];
  for (size_t i = 1; i < nr; i++) {
    uint64_t target = qoff[0] + total * i / nr;
    cut[i] = uint64_t(std::lower_bound(qoff, qoff + nq, target) - qoff);
    cut[i] = std::max(cut[i], cut[i - 1]);
  }
  std::vector<std::thread> th;
  std::vector<int> codes(nr, 0);
  std::vector<std::string> msgs(nr);
  for (size_t i = 0; i < nr; i++)
    th.emplace_back([&, i] {
      try {
        fn(i, cut[i], cut[i + 1]);
      } catch (const ApiError& e) {
        codes[i] = e.code;
        msgs[i] = e.what();
      } catch (const std::exception& e) {
        codes[i] = AWRY_ERR_INVALID_ARG;
        msgs[i] = e.what();
      }
    });
  for (auto& t : th) t.join();
  for (size_t i = 0; i < nr; i++)
    if (codes[i]) fail(codes[i], "%s", msgs[i].c_str());
}

struct LocatePart {
  std::vector<uint64_t> hit_off;  // local CSR over the replica's queries, size n+1
  awry_hit* hits = nullptr;       // malloc'd, or the caller's buffer when ext_cap != 0
  uint64_t n_hits = 0;
  uint64_t ext_cap = 0;           // caller-owned output: capacity in hits (0 = library allocates)
  uint64_t* ext_off = nullptr;    // caller-owned CSR offsets to fill directly (single replica)
};

// CSR offsets of a searched chunk (ws->d_out holds (sp, count) per query), no synchronisation
void locate_chunk_scan(Replica& r, Workspace* ws, uint64_t nq, uint64_t* d_hit_off, cudaStream_t st) {
  const void* d_sp_cnt = ws->d_out;
  size_t temp = 0;
  CU(scan_hit_offsets(r.view, d_sp_cnt, nq, d_hit_off, nullptr, temp, st));
  Workspace::grow_dev(reinterpret_cast<uint8_t*&>(ws->d_temp), ws->d_temp_cap, temp + 16);
  CU(scan_hit_offsets(r.view, d_sp_cnt, nq, d_hit_off, ws->d_temp, temp, st));
}

// device-side two-pass locate of a chunk whose queries were already searched (ws->d_out holds
// (sp, count) per query).  Step 1: CSR offsets + hit total (one synchronisation).
uint64_t locate_chunk_count(Replica& r, Workspace* ws, uint64_t nq, uint64_t* d_hit_off, cudaStream_t st) {
  locate_chunk_scan(r, ws, nq, d_hit_off, st);
  uint64_t n_hits = 0;
  CU(cudaMemcpyAsync(&n_hits, d_hit_off + nq, 8, cudaMemcpyDeviceToHost, st));
  CU(cudaStreamSynchronize(st));
  return n_hits;
}

// Step 2: LF-walk every hit; returns a stream-ordered device buffer with n_hits awry_hit entries.
uint64_t* locate_chunk_walk(Replica& r, Workspace* ws, uint64_t nq, uint64_t n_hits, uint32_t flags,
                            const uint64_t* d_hit_off, cudaStream_t st) {
  if (n_hits == 0) return nullptr;
  IndexView view = r.view;
  const int lv = g_locate_variant.load(std::memory_order_relaxed);
  if (lv != 0 && !ws->sp_cnt_positions) view.full_sa = nullptr;  // 1, 2: walk (unless pass 1 already wrote positions)
  if (lv == 1) view.walk_blocks = nullptr;                        // 1: to the file's row samples
  const void* d_sp_cnt = ws->d_out;
  uint64_t* d_hits = nullptr;
  CU(cudaMallocAsync(reinterpret_cast<void**>(&d_hits), n_hits * 16 + 16, st));  // pool: no driver round trip
  trace_mark("  hits buffer allocated, hits", (long long)n_hits);
  try {
    if (flags & AWRY_LOCATE_SORTED) {
      uint64_t *d_locs = nullptr, *d_sorted = nullptr;
      CU(cudaMallocAsync(reinterpret_cast<void**>(&d_locs), n_hits * 8 + 16, st));
      CU(cudaMallocAsync(reinterpret_cast<void**>(&d_sorted), n_hits * 8, st));
      {
        ProfScope p(1, r.device, st);
        CU(launch_walk(view, d_sp_cnt, d_hit_off, nq, n_hits, nullptr, d_locs, r.sm_count, st));
      }
      size_t t2 = 0;
      CU(sort_hit_segments(d_locs, d_sorted, n_hits, nq, d_hit_off, nullptr, t2, st));
      Workspace::grow_dev(reinterpret_cast<uint8_t*&>(ws->d_temp), ws->d_temp_cap, t2 + 16);
      CU(sort_hit_segments(d_locs, d_sorted, n_hits, nq, d_hit_off, ws->d_temp, t2, st));
      CU(launch_map_locations(view, d_sorted, n_hits, d_hits, st));
      cudaFreeAsync(d_locs, st);
      cudaFreeAsync(d_sorted, st);
    } else {
      ProfScope p(1, r.device, st);
      CU(launch_walk(view, d_sp_cnt, d_hit_off, nq, n_hits, d_hits, nullptr, r.sm_count, st));
    }
  } catch (...) {
    cudaFreeAsync(d_hits, st);
    throw;
  }
  return d_hits;
}

uint64_t* locate_chunk_device(const awry_index* ix, Replica& r, Workspace* ws, uint64_t nq,
                              uint32_t flags, uint64_t* d_hit_off, uint64_t* n_hits_out,
                              cudaStream_t st) {
  (void)ix;
  *n_hits_out = locate_chunk_count(r, ws, nq, d_hit_off, st);
  return locate_chunk_walk(r, ws, nq, *n_hits_out, flags, d_hit_off, st);
}

// parallel_locate over [q_lo, q_hi) on one replica.  The two passes of a chunk are separated by one small
// device->host read (the hit total sizes pass 2), and three chunks are in flight: while the host waits for
// chunk i's total, chunk i+1 is being packed, copied and searched, and chunk i-1's hits are on their way back.
// Chunk size: every chunk pays ~0.4 ms of fixed device-side latency (a persistent search kernel that fills
// the part and drains, a dozen small dependent operations, copies slowed 2-3x by the search kernel of the
// neighbouring chunk: profiles/r01_s50_locate_gpu_timeline.log), so 1 M x 50-bp queries take 3.31 / 2.55 /
// 2.51 / 2.71 ms end to end with chunks of 256 k / 384 k / 512 k / 1 M queries
// (profiles/r01_s51_locate_chunk_sweep.log): 512 k.
constexpr uint64_t LOCATE_CHUNK_BYTES = 64u << 20;
static uint64_t locate_chunk_q() {  // AWRY_B200_LOCATE_CHUNK_Q: queries per chunk (experiments; read per call)
  if (const char* e = getenv("AWRY_B200_LOCATE_CHUNK_Q")) return std::min<uint64_t>(1u << 24, std::max<uint64_t>(1024, strtoull(e, nullptr, 10)));
  return 1u << 19;
}
static uint64_t locate_chunk_bytes() {
  if (const char* e = getenv("AWRY_B200_LOCATE_CHUNK_MB")) return std::min<uint64_t>(1024, std::max<uint64_t>(1, strtoull(e, nullptr, 10))) << 20;
  return LOCATE_CHUNK_BYTES;
}

void locate_on_replica(const awry_index* ix, size_t ri, const QuerySource& qs, uint64_t q_lo, uint64_t q_hi,
                       uint32_t flags, LocatePart& part) {
  const bool ext = part.ext_cap != 0 || part.ext_off != nullptr;
  const uint64_t m = qs.per_query();  // CSR entries per query
  if (!part.ext_off) part.hit_off.assign(m * (q_hi - q_lo) + 1, 0);
  uint64_t* off_base = part.ext_off ? part.ext_off : part.hit_off.data();
  if (q_lo >= q_hi) return;
  Replica& r = *ix->reps[ri];
  PackBalance& bal = ix->balance_of(ri);
  DeviceGuard dg(r.device);
  const uint64_t* qoff = qs.qoff;
  const uint64_t max_bytes = std::min(chunk_max_bytes(), locate_chunk_bytes());
  auto chunks = make_chunks(qoff, q_lo, q_hi, locate_chunk_q(), max_bytes);
  validate_chunks(chunks, max_bytes);
  constexpr int DEPTH = 3;
  struct Slot {
    Workspace* ws = nullptr;
    int chunk = -1;
    int phase = 0;  // 1 = searched + scanned (total on its way), 2 = pass 2 enqueued (results on their way)
    uint64_t base = 0;
  } slot[DEPTH];
  size_t cap = 0;
  auto mark = [&](const char* what, int i) { trace_mark(what, i); };
  // offsets of a chunk are rebased onto the replica-local hit count before it; the slot shared with the
  // next chunk (index nq) is written by that chunk, the very last one after the loop
  auto stage_c = [&](Slot& s) {
    if (s.phase != 2) return;
    const Chunk& c = chunks[size_t(s.chunk)];
    CU(cudaEventSynchronize(s.ws->done));
    uint64_t* dst_off = off_base + m * (c.q0 - q_lo);
    const uint64_t nq = m * (c.q1 - c.q0), base = s.base;
    if (base)
      for (uint64_t i = 0; i < nq; i++) dst_off[i] += base;
    s.phase = 0;
    s.chunk = -1;
  };
  auto stage_a = [&](int i) {
    Slot& s = slot[i % DEPTH];
    if (!s.ws) s.ws = r.acquire();
    stage_c(s);
    Workspace* ws = s.ws;
    const Chunk& c = chunks[size_t(i)];
    const uint64_t nq = m * (c.q1 - c.q0);
    mark("A begin", i);
    gpu_mark(ws->st, "chunk begins", i);
    enqueue_search(ix, r, bal, ws, qs, c, OUT_SP_CNT_U32, true, false, false);
    mark("A searched", i);
    Workspace::grow_dev(ws->d_hit_off, ws->d_hit_off_cap, size_t(nq) + 1);
    locate_chunk_scan(r, ws, nq, ws->d_hit_off, ws->st);
    gpu_mark(ws->st, "scanned", i);
    CU(cudaMemcpyAsync(ws->h_flag, ws->d_flag, 8, cudaMemcpyDeviceToHost, ws->st));
    CU(cudaMemcpyAsync(ws->h_total, ws->d_hit_off + nq, 8, cudaMemcpyDeviceToHost, ws->st));
    CU(cudaEventRecord(ws->done, ws->st));
    gpu_mark(ws->st, "total copied", i);
    mark("A end", i);
    s.chunk = i;
    s.phase = 1;
  };
  auto stage_b = [&](int i) {
    Slot& s = slot[i % DEPTH];
    Workspace* ws = s.ws;
    const Chunk& c = chunks[size_t(i)];
    const uint64_t nq = m * (c.q1 - c.q0);
    mark("B wait", i);
    CU(cudaEventSynchronize(ws->done));
    mark("B total known", i);
    const uint64_t n_hits = *ws->h_total;
    check_flag(ws, c);
    s.base = part.n_hits;
    gpu_mark(ws->st, "pass 2 begins", i);
    CU(cudaMemcpyAsync(off_base + m * (c.q0 - q_lo), ws->d_hit_off, nq * 8, cudaMemcpyDeviceToHost, ws->st));
    gpu_mark(ws->st, "offsets copied", i);
    g_prof.d2h += nq * 8;
    const bool fits = !ext || part.n_hits + n_hits <= part.ext_cap;
    if (n_hits && fits) {
      if (!ext && part.n_hits + n_hits > cap) {
        for (auto& o : slot) stage_c(o);  // copies into the old buffer must land before it moves
        cap = std::max<size_t>(size_t(part.n_hits + n_hits), cap * 2);
        void* np = realloc(part.hits, cap * sizeof(awry_hit));
        if (!np) fail(AWRY_ERR_NOMEM, "out of host memory for %llu hits", (unsigned long long)cap);
        part.hits = static_cast<awry_hit*>(np);
      }
      uint64_t* d_hits = locate_chunk_walk(r, ws, nq, n_hits, flags, ws->d_hit_off, ws->st);
      gpu_mark(ws->st, "hits located", i);
      CU(cudaMemcpyAsync(part.hits + part.n_hits, d_hits, n_hits * 16, cudaMemcpyDeviceToHost, ws->st));
      gpu_mark(ws->st, "hits copied", i);
      cudaFreeAsync(d_hits, ws->st);
      g_prof.d2h += n_hits * 16;
    }
    CU(cudaEventRecord(ws->done, ws->st));
    mark("B end", i);
    s.phase = 2;
    part.n_hits += n_hits;  // keeps counting past the capacity so the caller learns the need
  };
  GpuTrace gpu_trace;
  g_gpu_trace = trace_on() ? &gpu_trace : nullptr;
  try {
    stage_a(0);
    for (int i = 0; i < int(chunks.size()); i++) {
      if (i + 1 < int(chunks.size())) stage_a(i + 1);
      stage_b(i);
    }
    for (auto& s : slot) stage_c(s);
    off_base[m * (q_hi - q_lo)] = part.n_hits;
    mark("done", int(chunks.size()));
    g_gpu_trace = nullptr;
    gpu_trace.dump();
  } catch (...) {
    g_gpu_trace = nullptr;
    for (auto& s : slot)
      if (s.ws) {
        cudaStreamSynchronize(s.ws->st);
        r.release(s.ws);
      }
    if (!ext) free(part.hits);
    part.hits = nullptr;
    throw;
  }
  for (auto& s : slot)
    if (s.ws) r.release(s.ws);
}

// parallel_locate into the caller's pinned buffers with no host round trip between the passes (the
// unsampled-SA gather, BWT order).  Per chunk: pack -> search -> scan -> the device hands the chunk its hit base
// (advance_hit_base_kernel, ordered behind the previous chunk's by an event) -> the gather writes the hits
// straight into `hits` (host memory, through its device view) and the rebased offsets into a device array
// that one copy returns.  The host enqueues chunk after chunk and waits once at the end; a workspace is
// reused when its chunk of three rounds ago has drained.  Returns the hit total (it may exceed capacity).
// cfg3 end to end: 2.2 ms -> see profiles/ (the two-sync pipeline above stays for library-owned results,
// sorted output and the LF-walk variants, which size their buffers from the total).
uint64_t locate_direct_on_replica(const awry_index* ix, size_t ri, const QuerySource& qs, uint64_t nq, uint64_t* hit_off,
                                  void* hits_dev, uint64_t capacity) {
  Replica& r = *ix->reps[ri];
  PackBalance& bal = ix->balance_of(ri);
  DeviceGuard dg(r.device);
  const uint64_t* qoff = qs.qoff;
  const uint64_t max_bytes = std::min(chunk_max_bytes(), locate_chunk_bytes());
  auto chunks = make_chunks(qoff, 0, nq, locate_chunk_q(), max_bytes);
  validate_chunks(chunks, max_bytes);
  // A call of this size is latency-bound and the device idles while the host packs the first chunk (0.4 ms for
  // 25 MB: profiles/r02_s2_locate_e2e_trace.log).  So the first chunk is cut to a quarter and goes up as it is --
  // the copy engine starts at once, the device packs it -- while the host packs what follows.
  bool first_raw = false;
  if (chunks.size() >= 1 && chunks[0].q1 - chunks[0].q0 >= (1u << 16) && qs.pinned && !qs.crumbs &&
      getenv("AWRY_B200_LOCATE_FIRST_RAW") == nullptr) {
    const Chunk c = chunks[0];
    const uint64_t cut = c.q0 + (c.q1 - c.q0) / 4;
    chunks[0] = Chunk{c.q0, cut, qoff[c.q0], qoff[cut]};
    chunks.insert(chunks.begin() + 1, Chunk{cut, c.q1, qoff[cut], qoff[c.q1]});
    first_raw = true;
  }
  const bool off_pinned = is_pinned(hit_off);
  const uint64_t m = qs.per_query();  // CSR entries per query
  constexpr int DEPTH = 3;
  Workspace* ws[DEPTH] = {nullptr, nullptr, nullptr};
  int pending[DEPTH] = {-1, -1, -1};
  auto finish = [&](int s) {
    if (pending[s] < 0) return;
    const Chunk& c = chunks[size_t(pending[s])];
    CU(cudaEventSynchronize(ws[s]->done));
    check_flag(ws[s], c);
    if (!off_pinned) memcpy(hit_off + m * c.q0, ws[s]->h_out, m * (c.q1 - c.q0) * 8);
    pending[s] = -1;
  };
  GpuTrace gpu_trace;
  g_gpu_trace = trace_on() ? &gpu_trace : nullptr;
  uint64_t total = 0;
  try {
    ws[0] = r.acquire();
    unsigned long long* const d_running = ws[0]->d_base + 1;
    CU(cudaMemsetAsync(d_running, 0, 8, ws[0]->st));
    CU(cudaEventRecord(ws[0]->ev_adv, ws[0]->st));  // chunk 0 waits for the counter's reset like for a predecessor
    cudaEvent_t prev_adv = ws[0]->ev_adv;
    for (size_t i = 0; i < chunks.size(); i++) {
      const int s = int(i % DEPTH);
      if (!ws[s]) ws[s] = r.acquire();
      finish(s);
      Workspace* w = ws[s];
      const Chunk& c = chunks[i];
      const uint64_t n = m * (c.q1 - c.q0);
      gpu_mark(w->st, "chunk begins", (long long)i);
      enqueue_search(ix, r, bal, w, qs, c, OUT_SP_CNT_U32, !(first_raw && i == 0), false, false);
      Workspace::grow_dev(w->d_hit_off, w->d_hit_off_cap, size_t(n) + 1);
      Workspace::grow_dev(w->d_off_out, w->d_off_out_cap, size_t(n) + 1);
      locate_chunk_scan(r, w, n, w->d_hit_off, w->st);
      gpu_mark(w->st, "scanned", (long long)i);
      // (chunk 0 waits for the counter's reset; a slot's event is re-recorded only after the wait on its
      // earlier state has been enqueued)
      CU(launch_gather_direct(r.view, reinterpret_cast<const uint2*>(w->d_out), w->d_hit_off, n, d_running, w->d_base,
                              hits_dev, capacity, w->d_off_out, r.sm_count, prev_adv, w->ev_adv, w->st));
      prev_adv = w->ev_adv;
      gpu_mark(w->st, "hits written", (long long)i);
      uint64_t* dst = hit_off + m * c.q0;
      if (!off_pinned) {
        Workspace::grow_host(w->h_out, w->h_out_cap, size_t(n) * 8);
        dst = reinterpret_cast<uint64_t*>(w->h_out);
      }
      CU(cudaMemcpyAsync(dst, w->d_off_out, n * 8, cudaMemcpyDeviceToHost, w->st));
      CU(cudaMemcpyAsync(w->h_flag, w->d_flag, 8, cudaMemcpyDeviceToHost, w->st));
      if (i + 1 == chunks.size()) CU(cudaMemcpyAsync(w->h_total, d_running, 8, cudaMemcpyDeviceToHost, w->st));
      g_prof.d2h += n * 8 + 16;
      CU(cudaEventRecord(w->done, w->st));
      pending[s] = int(i);
    }
    const int last = int((chunks.size() - 1) % DEPTH);
    for (int s = 0; s < DEPTH; s++) finish((last + 1 + s) % DEPTH);  // oldest first; the last chunk carries the total
    total = *ws[last]->h_total;
    g_prof.d2h += std::min(total, capacity) * sizeof(awry_hit);
    hit_off[m * nq] = total;
    g_gpu_trace = nullptr;
    gpu_trace.dump();
  } catch (...) {
    g_gpu_trace = nullptr;
    for (int s = 0; s < DEPTH; s++)
      if (ws[s]) {
        cudaStreamSynchronize(ws[s]->st);
        r.release(ws[s]);
      }
    throw;
  }
  for (int s = 0; s < DEPTH; s++)
    if (ws[s]) r.release(ws[s]);
  return total;
}

// the device's view of a page-locked host buffer (cudaHostAlloc / cudaHostRegister), or nullptr
void* device_view_of_pinned(const void* p) {
  if (!p || !is_pinned(p)) return nullptr;
  void* d = nullptr;
  if (cudaHostGetDevicePointer(&d, const_cast<void*>(p), 0) != cudaSuccess) {
    cudaGetLastError();
    return nullptr;
  }
  return d;
}

static bool direct_locate_enabled() {  // AWRY_B200_LOCATE_DIRECT=0: always the two-sync pipeline (A/B runs)
  const char* e = getenv("AWRY_B200_LOCATE_DIRECT");
  return !(e && e[0] == '0');
}

QuerySource ascii_source(const uint8_t* qbytes, const uint64_t* qoff) {
  QuerySource qs;
  qs.qbytes = qbytes;
  qs.qoff = qoff;
  qs.pinned = is_pinned(qbytes) && is_pinned(qoff);
  return qs;
}

// awry_*_batch_packed2 arguments -> QuerySource (nucleotide only; exceptions must ascend by position)
QuerySource packed2_source(const awry_index* ix, const uint8_t* crumbs, const uint64_t* qoff, uint64_t nq,
                           const uint64_t* exceptions, uint64_t n_exc) {
  if (ix->alphabet != AWRY_NUCLEOTIDE) fail(AWRY_ERR_UNSUPPORTED, "2-bit packed queries exist for the nucleotide alphabet only");
  if (!crumbs || !qoff || (n_exc && !exceptions)) fail(AWRY_ERR_INVALID_ARG, "null argument");
  for (uint64_t i = 1; i < n_exc; i++)
    if ((exceptions[i] >> 8) <= (exceptions[i - 1] >> 8))
      fail(AWRY_ERR_INVALID_ARG, "exception list is not strictly ascending by position (entry %llu)", (unsigned long long)i);
  if (n_exc && (exceptions[n_exc - 1] >> 8) >= qoff[nq] && qoff[nq] >= qoff[0])
    fail(AWRY_ERR_INVALID_ARG, "exception position %llu lies behind the last query byte",
         (unsigned long long)(exceptions[n_exc - 1] >> 8));
  QuerySource qs;
  qs.crumbs = crumbs;
  qs.exc = exceptions;
  qs.n_exc = n_exc;
  qs.qoff = qoff;
  qs.pinned = is_pinned(crumbs) && is_pinned(qoff) && (n_exc == 0 || is_pinned(exceptions));
  return qs;
}

void count_impl(const awry_index* ix, const QuerySource& qs, uint64_t nq, SearchOut mode, void* out) {
  const size_t nr = ix->reps.size();
  const size_t active = (nr == 1 || nq < 2 * nr) ? 1 : nr;  // (for_each_replica_range's own rule)
  for_each_replica_range(ix, qs.qoff, nq, [&](size_t ri, uint64_t lo, uint64_t hi) {
    search_on_replica(ix, ri, qs, lo, hi, mode, out, active);
  });
}

void locate_owned_impl(const awry_index* ix, const QuerySource& qs, uint64_t nq, uint32_t flags, uint64_t* hit_off,
                       awry_hit** hits, uint64_t* n_hits) {
  size_t nr = ix->reps.size();
  std::vector<LocatePart> parts(nr);
  std::vector<std::pair<uint64_t, uint64_t>> ranges(nr, {0, 0});
  try {
    for_each_replica_range(ix, qs.qoff, nq, [&](size_t ri, uint64_t lo, uint64_t hi) {
      ranges[ri] = {lo, hi};
      locate_on_replica(ix, ri, qs, lo, hi, flags, parts[ri]);
    });
  } catch (...) {
    for (auto& p : parts) free(p.hits);
    throw;
  }
  // concatenate in range order (results of the reference's order-preserving collect)
  uint64_t total = 0;
  for (auto& p : parts) total += p.n_hits;
  awry_hit* all = nullptr;
  if (nr == 1) {
    all = parts[0].hits;
    parts[0].hits = nullptr;
  } else if (total) {
    all = static_cast<awry_hit*>(malloc(total * sizeof(awry_hit)));
    if (!all) {
      for (auto& p : parts) free(p.hits);
      fail(AWRY_ERR_NOMEM, "out of host memory for %llu hits", (unsigned long long)total);
    }
  }
  uint64_t base = 0;
  const uint64_t m = qs.per_query();
  for (size_t ri = 0; ri < nr; ri++) {
    auto [lo, hi] = ranges[ri];
    if (hi > lo)
      for (uint64_t i = 0; i <= m * (hi - lo); i++) hit_off[m * lo + i] = base + parts[ri].hit_off[i];
    if (nr > 1 && parts[ri].n_hits) memcpy(all + base, parts[ri].hits, parts[ri].n_hits * sizeof(awry_hit));
    base += parts[ri].n_hits;
    if (nr > 1) free(parts[ri].hits);
  }
  hit_off[m * nq] = total;
  *hits = all;
  *n_hits = total;
}

// parallel_locate over SEVERAL replicas into the caller's pinned buffers (BWT order, unsampled array).  A
// replica's hits start behind those of the replicas before it, which nobody knows until they have searched; so
// the call has two phases with one meeting of the replica threads between them.  Phase 1, all replicas at once:
// the chunk pipeline packs, uploads and searches, the (sp, count) pairs land in one array per replica, one scan
// gives its local CSR offsets and its hit total.  The totals are prefix-summed on the host.  Phase 2, all
// replicas at once: one gather per replica writes the hits STRAIGHT into the caller's buffer at its base, the
// rebased offsets go back with one copy.  No staging buffer, no concatenation pass on the host.
struct ReplicaLocateState {
  uint64_t lo = 0, hi = 0, total = 0, base = 0;
  Workspace* ws = nullptr;  // holds the call-level arrays of this replica (d_out: pairs, d_hit_off: local offsets)
};

void locate_multi_phase1(const awry_index* ix, size_t ri, const QuerySource& qs, ReplicaLocateState& st, size_t n_active) {
  (void)n_active;
  if (st.lo >= st.hi) return;
  Replica& r = *ix->reps[ri];
  PackBalance& bal = ix->balance_of(ri);
  DeviceGuard dg(r.device);
  const uint64_t m = qs.per_query();
  const uint64_t n = m * (st.hi - st.lo);  // CSR entries
  const uint64_t max_bytes = std::min(chunk_max_bytes(), locate_chunk_bytes());
  auto chunks = make_chunks(qs.qoff, st.lo, st.hi, locate_chunk_q(), max_bytes);
  validate_chunks(chunks, max_bytes);
  st.ws = r.acquire();
  Workspace* top = st.ws;
  const size_t pair_bytes = sp_cnt_bytes(r.view);
  Workspace::grow_dev(top->d_out, top->d_out_cap, size_t(n) * pair_bytes);
  Workspace::grow_dev(top->d_hit_off, top->d_hit_off_cap, size_t(n) + 1);
  Workspace::grow_dev(top->d_off_out, top->d_off_out_cap, size_t(n) + 1);
  constexpr int DEPTH = 3;
  Workspace* ws[DEPTH] = {nullptr, nullptr, nullptr};
  int pending[DEPTH] = {-1, -1, -1};
  auto finish = [&](int s) {
    if (pending[s] < 0) return;
    CU(cudaEventSynchronize(ws[s]->done));
    check_flag(ws[s], chunks[size_t(pending[s])]);
    pending[s] = -1;
  };
  try {
    for (size_t i = 0; i < chunks.size(); i++) {
      const int s = int(i % DEPTH);
      if (!ws[s]) ws[s] = r.acquire();
      finish(s);
      const Chunk& c = chunks[i];
      enqueue_search(ix, r, bal, ws[s], qs, c, OUT_SP_CNT_U32, true, false, true,
                     top->d_out + size_t(m * (c.q0 - st.lo)) * pair_bytes);
      CU(cudaEventRecord(ws[s]->done, ws[s]->st));
      pending[s] = int(i);
    }
    for (int s = 0; s < DEPTH; s++) finish(s);  // every chunk has searched: the pairs are complete
    locate_chunk_scan(r, top, n, top->d_hit_off, top->st);
    CU(cudaMemcpyAsync(top->h_total, top->d_hit_off + n, 8, cudaMemcpyDeviceToHost, top->st));
    CU(cudaStreamSynchronize(top->st));
    st.total = *top->h_total;
  } catch (...) {
    for (int s = 0; s < DEPTH; s++)
      if (ws[s]) {
        cudaStreamSynchronize(ws[s]->st);
        r.release(ws[s]);
      }
    cudaStreamSynchronize(top->st);
    r.release(top);
    st.ws = nullptr;
    throw;
  }
  for (int s = 0; s < DEPTH; s++)
    if (ws[s]) r.release(ws[s]);
}

void locate_multi_phase2(const awry_index* ix, size_t ri, ReplicaLocateState& st, uint64_t* hit_off, void* hits_dev,
                         uint64_t capacity, uint64_t m) {
  if (st.lo >= st.hi || !st.ws) return;
  Replica& r = *ix->reps[ri];
  DeviceGuard dg(r.device);
  Workspace* top = st.ws;
  const uint64_t n = m * (st.hi - st.lo);  // CSR entries
  const bool off_pinned = is_pinned(hit_off);
  try {
    unsigned long long base = st.base;
    CU(cudaMemcpyAsync(top->d_base + 1, &base, 8, cudaMemcpyHostToDevice, top->st));  // (pageable source: copied at the call)
    CU(launch_gather_direct(r.view, reinterpret_cast<const uint2*>(top->d_out), top->d_hit_off, n, top->d_base + 1, top->d_base,
                            hits_dev, capacity, top->d_off_out, r.sm_count, nullptr, nullptr, top->st));
    uint64_t* dst = hit_off + m * st.lo;
    if (!off_pinned) {
      Workspace::grow_host(top->h_out, top->h_out_cap, size_t(n) * 8);
      dst = reinterpret_cast<uint64_t*>(top->h_out);
    }
    CU(cudaMemcpyAsync(dst, top->d_off_out, n * 8, cudaMemcpyDeviceToHost, top->st));
    g_prof.d2h += n * 8 + std::min(st.total, capacity > st.base ? capacity - st.base : 0) * sizeof(awry_hit);
    CU(cudaStreamSynchronize(top->st));
    if (!off_pinned) parallel_memcpy(hit_off + m * st.lo, top->h_out, n * 8);
  } catch (...) {
    cudaStreamSynchronize(top->st);
    r.release(top);
    st.ws = nullptr;
    throw;
  }
  r.release(top);
  st.ws = nullptr;
}

void locate_into_impl(const awry_index* ix, const QuerySource& qs, uint64_t nq, uint32_t flags, uint64_t* hit_off,
                      awry_hit* hits, uint64_t capacity, uint64_t* n_hits) {
  auto too_small = [&](uint64_t need) {
    fail(AWRY_ERR_CAPACITY, "hit buffer holds %llu entries, %llu needed", (unsigned long long)capacity,
         (unsigned long long)need);
  };
  if (ix->reps.size() == 1) {
    Replica& r0 = *ix->reps[0];
    void* hits_dev = capacity ? device_view_of_pinned(hits) : nullptr;
    if (hits_dev && !(flags & AWRY_LOCATE_SORTED) && r0.view.full_sa && g_locate_variant == 0 && direct_locate_enabled()) {
      *n_hits = locate_direct_on_replica(ix, 0, qs, nq, hit_off, hits_dev, capacity);
      if (*n_hits > capacity) too_small(*n_hits);
      return;
    }
    // hits and offsets land straight in the caller's (ideally pinned) buffers
    LocatePart part;
    part.hits = hits;
    part.ext_cap = capacity;
    part.ext_off = hit_off;  // marks the part as caller-owned even when capacity is 0
    locate_on_replica(ix, 0, qs, 0, nq, flags, part);
    *n_hits = part.n_hits;
    if (part.n_hits > capacity) too_small(part.n_hits);
    return;
  }
  {  // several replicas: two phases with the hits written straight into the caller's pinned buffer
    void* hits_dev = capacity ? device_view_of_pinned(hits) : nullptr;
    bool all_full_sa = true;
    for (auto& rp : ix->reps) all_full_sa = all_full_sa && rp->view.full_sa != nullptr;
    const size_t nr = ix->reps.size();
    if (hits_dev && !(flags & AWRY_LOCATE_SORTED) && all_full_sa && g_locate_variant == 0 && direct_locate_enabled() &&
        nq >= 2 * nr) {
      std::vector<ReplicaLocateState> st(nr);
      auto release_all = [&] {
        for (size_t ri = 0; ri < nr; ri++)
          if (st[ri].ws) {
            cudaSetDevice(ix->reps[ri]->device);
            cudaStreamSynchronize(st[ri].ws->st);
            ix->reps[ri]->release(st[ri].ws);
            st[ri].ws = nullptr;
          }
      };
      try {
        for_each_replica_range(ix, qs.qoff, nq, [&](size_t ri, uint64_t lo, uint64_t hi) {
          st[ri].lo = lo;
          st[ri].hi = hi;
          locate_multi_phase1(ix, ri, qs, st[ri], nr);
        });
        uint64_t total = 0;
        for (auto& x : st) {
          x.base = total;
          total += x.total;
        }
        for_each_replica_range(ix, qs.qoff, nq, [&](size_t ri, uint64_t, uint64_t) {
          locate_multi_phase2(ix, ri, st[ri], hit_off, hits_dev, capacity, qs.per_query());
        });
        hit_off[qs.per_query() * nq] = total;
        *n_hits = total;
      } catch (...) {
        release_all();
        throw;
      }
      if (*n_hits > capacity) too_small(*n_hits);
      return;
    }
  }
  awry_hit* tmp = nullptr;
  uint64_t n = 0;
  locate_owned_impl(ix, qs, nq, flags, hit_off, &tmp, &n);
  *n_hits = n;
  if (n > capacity) {
    free(tmp);
    too_small(n);
  }
  if (n) parallel_memcpy(hits, tmp, n * sizeof(awry_hit));
  free(tmp);
}

// ------------------------------------------------------------------ Hamming search (awry_*_hamming)

// stream-ordered device allocations of one call or slice, released in stream order when it goes out of scope
struct StreamScratch {
  cudaStream_t st;
  std::vector<void*> ptrs;
  explicit StreamScratch(cudaStream_t s) : st(s) {}
  ~StreamScratch() {
    for (void* p : ptrs) cudaFreeAsync(p, st);
  }
  template <class T>
  T* get(uint64_t n) {
    void* p = nullptr;
    const cudaError_t e = cudaMallocAsync(&p, size_t(n) * sizeof(T) + 16, st);
    if (e == cudaErrorMemoryAllocation) {
      cudaGetLastError();
      fail(AWRY_ERR_NOMEM, "out of device memory for %llu bytes of Hamming-search scratch",
           (unsigned long long)(n * sizeof(T)));
    }
    CU(e);
    ptrs.push_back(p);
    return static_cast<T*>(p);
  }
};

// candidates verified per slice (AWRY_B200_HAMMING_SLICE, read per call): bounds the scratch of the verification
static uint64_t hamming_slice() {
  if (const char* e = getenv("AWRY_B200_HAMMING_SLICE"))
    return std::min<uint64_t>(1ull << 30, std::max<uint64_t>(16, strtoull(e, nullptr, 10)));
  return 1ull << 26;
}

void hamming_check_index(const awry_index* ix, const char* what = "Hamming") {
  if (ix->alphabet != AWRY_NUCLEOTIDE) fail(AWRY_ERR_UNSUPPORTED, "%s search exists for the nucleotide alphabet only", what);
  for (auto& rp : ix->reps)
    if (rp->view.wide || !rp->view.rtext || !rp->view.full_sa)
      fail(AWRY_ERR_UNSUPPORTED,
           "%s search needs the unsampled suffix array and the text on every device (not built for this index: "
           "AWRY_B200_FULL_SA / AWRY_B200_TEXT, device memory, or 64-bit row pointers)", what);
}

// the hits of the locate call on one replica, in query order
struct HammingSink {
  std::vector<uint64_t> off;  // per (virtual) query: offset of its first hit in `hits`
  std::vector<awry_hit> hits;
  std::vector<uint8_t> dist;
};

// the outputs of the device-resident locate (awry_locate_device_{hamming,edit}[_strands])
struct DeviceHits {
  uint64_t* hit_off;  // device, nv + 1: the CSR over the (virtual) queries
  awry_hit** hits;    // a device allocation of *n_hits hits (not set when there are none)
  uint8_t** dist;     // likewise, each hit's distance; nullptr: not wanted
  uint64_t* n_hits;
};

// One batch of reads on one replica, all on stream `st`: pieces -> exact search of the pieces -> candidates ->
// verification against the text, in slices of at most hamming_slice() candidates.  Offsets are absolute and lie
// in [b_lo, b_hi] (d_qbytes is biased accordingly).  Count: d_counts (nq * (k + 1)) is zeroed and filled.  Locate:
// the hits are appended to `sink` (slices cut at read boundaries, the hits of a read sorted by text position).
// Device-resident locate (`dev`): a count pass and a place pass over the same slices, then one segmented sort; the
// hits stay on the device, and the call returns without waiting for the last kernels.
// `check_base` >= 0: a refused read fails the call (reported as read check_base + q) before anything is verified;
// < 0 (the device-resident call): it stays latched in *d_flag for awry_device_check.
// `strands`: the nq reads are searched as the 2 nq virtual queries of both strands (kernels.hpp), which take the
// place of the reads from the piece offsets on: counts, CSR offsets and the hits are per virtual query.
// `metric`: substitutions (Hamming, one window per candidate) or edits (awry_*_edit: 2k + 1 starts per candidate,
// kernels_edit.cu).  Stages 1 and 2 are the same for both; the metric picks the verification kernel and, for locate,
// the key slots per candidate.  A slice holds at most hamming_slice() key slots.
enum Metric { METRIC_HAMMING = 0, METRIC_EDIT = 1 };
const char* metric_name(Metric metric) { return metric == METRIC_EDIT ? "edit-distance" : "Hamming"; }
void hamming_run(Replica& r, const uint8_t* d_qbytes, const uint64_t* d_qoff, uint64_t nq, uint64_t b_lo, uint64_t b_hi,
                 uint32_t k, unsigned long long* d_flag, long long check_base, cudaStream_t st, uint64_t* d_counts,
                 HammingSink* sink, bool strands = false, Metric metric = METRIC_HAMMING, DeviceHits* dev = nullptr) {
  const bool edit = metric == METRIC_EDIT;
  const char* const what = metric_name(metric);
  const uint32_t shift = strands ? 1 : 0;  // virtual query -> read
  const uint64_t P = k + 1, nbytes = b_hi - b_lo, nv = nq << shift, np = nv * P;
  const uint64_t slots = edit ? 2 * k + 1 : 1;  // key slots per candidate
  if (np >= (1ull << 31)) fail(AWRY_ERR_INVALID_ARG, "batch too large for one %s search (%llu reads): split it", what, (unsigned long long)nq);
  StreamScratch sc(st);
  // 1. pieces, packed; the whole reads packed too (their prepass validates the offsets and latches what it refuses).
  // Single strand: the pieces are packed from the caller's bytes (DESIGN.md §1c: cutting them out of the read words
  // measured slower at k = 1 and 3).  Both strands: the virtual queries' offsets and words come from the reads', and
  // the pieces' words are cut out of the virtual words (a reverse-complement piece has no bytes to pack).
  const uint64_t rw_n = packed_words(0, nq, nbytes), w_lo = 4 * (b_lo >> 6);
  const uint64_t v_lo = b_lo << shift, v_hi = b_hi << shift, vw_n = packed_words(0, nv, nbytes << shift), vw_lo = 4 * (v_lo >> 6);
  const uint64_t* d_voff = d_qoff;
  uint64_t* d_poff = sc.get<uint64_t>(np + 1);
  uint64_t* const d_pw = sc.get<uint64_t>(packed_words(0, np, nbytes << shift)) - vw_lo;
  uint64_t* const d_rw = sc.get<uint64_t>(rw_n) - w_lo;
  uint64_t* d_vw = d_rw;
  {
    ProfScope p(2, r.device, st);
    if (!strands) {
      unsigned long long* d_pflag = sc.get<unsigned long long>(1);  // (piece indices: what it latches is reported per read)
      CU(cudaMemsetAsync(d_pflag, 0xff, 8, st));
      CU(launch_hamming_pieces(d_qoff, nq, k, b_lo, b_hi, 0, d_poff, d_flag, st));
      CU(launch_pack(AWRY_NUCLEOTIDE, d_qbytes, d_poff, np, d_pw, b_lo, b_hi, d_pflag, st));
      CU(launch_pack(AWRY_NUCLEOTIDE, d_qbytes, d_qoff, nq, d_rw, b_lo, b_hi, d_flag, st));
    } else {
      uint64_t* const voff = sc.get<uint64_t>(nv + 1);
      d_vw = sc.get<uint64_t>(vw_n) - vw_lo;
      CU(launch_pack(AWRY_NUCLEOTIDE, d_qbytes, d_qoff, nq, d_rw, b_lo, b_hi, d_flag, st));
      CU(launch_strand_offsets(d_qoff, nq, b_lo, b_hi, voff, st));
      CU(launch_strand_words(d_rw, d_qoff, nq, b_lo, b_hi, voff, d_vw, st));
      d_voff = voff;
      CU(launch_hamming_pieces(d_voff, nv, k, v_lo, v_hi, shift, d_poff, d_flag, st));
      CU(launch_hamming_piece_words(d_vw, d_voff, nv, v_lo, v_hi, k, d_pw, st));
    }
  }
  // 2. exact search of the pieces (the wave kernel stores a piece finished in the text as its position), CSR
  // offsets of their occurrences = the candidates
  uint2* d_sp = sc.get<uint2>(np);
  {
    ProfScope p(0, r.device, st);
    SearchVariant v = current_variant();
    v.avg_len = uint32_t(std::min<uint64_t>((nbytes << shift) / np, 1u << 30));
    v.b_lo = v_lo;
    v.b_hi = v_hi;
    v.locate_positions = locate_positions_ok(r.view, v);
    CU(launch_search(r.view, d_pw, d_poff, np, OUT_SP_CNT_U32, d_sp, sc.get<uint32_t>(defer_words(np)), v, r.sm_count, st));
  }
  uint64_t* d_hoff = sc.get<uint64_t>(np + 1);
  size_t temp = 0;
  CU(scan_hit_offsets(r.view, d_sp, np, d_hoff, nullptr, temp, st));
  CU(scan_hit_offsets(r.view, d_sp, np, d_hoff, sc.get<uint8_t>(temp), temp, st));
  // the candidate total (and, for locate, every read's candidate range) sizes the slices: one synchronisation
  uint64_t total = 0;
  unsigned long long flag = ~0ull;
  std::vector<uint64_t> qcand;
  uint64_t* d_qcand = nullptr;
  if (sink) {
    d_qcand = sc.get<uint64_t>(nv + 1);
    CU(launch_hamming_query_bounds(d_hoff, k, nv, d_qcand, st));
    qcand.resize(nv + 1);
    CU(cudaMemcpyAsync(qcand.data(), d_qcand, (nv + 1) * 8, cudaMemcpyDeviceToHost, st));
    g_prof.d2h += (nv + 1) * 8;
  }
  CU(cudaMemcpyAsync(&total, d_hoff + np, 8, cudaMemcpyDeviceToHost, st));
  if (check_base >= 0) CU(cudaMemcpyAsync(&flag, d_flag, 8, cudaMemcpyDeviceToHost, st));
  CU(cudaStreamSynchronize(st));
  if (flag != ~0ull && (flag & 1) == BAD_QUERY)
    fail(AWRY_ERR_INVALID_QUERY,
         "query %llu is empty, contains a sentinel ('$'/'#') or is not longer than %s = %u (every window "
         "would match)", (unsigned long long)(uint64_t(check_base) + (flag >> 1)), edit ? "max_edits" : "max_mismatches", k);
  if (flag != ~0ull) fail_bad_query(flag, uint64_t(check_base));

  HammingSlice a{};
  a.qwords = d_vw;
  a.qw_lo = strands ? vw_lo : w_lo;
  a.qw_n = strands ? vw_n : rw_n;
  a.qoff = d_voff;
  a.b_lo = v_lo;
  a.b_hi = v_hi;
  a.sp_cnt = d_sp;
  a.hoff = d_hoff;
  a.npieces = np;
  const uint64_t S = std::max<uint64_t>(1, hamming_slice() / slots);  // candidates per slice
  auto verify_all = [&](VerifyMode mode) {  // every candidate, in slices cut anywhere
    for (uint64_t c0 = 0; c0 < total; c0 += S) {
      StreamScratch ss(st);
      a.c0 = c0;
      a.n = std::min(S, total - c0);
      uint32_t* d_map = ss.get<uint32_t>(a.n);
      CU(launch_hamming_map(d_hoff, np, c0, a.n, d_map, nullptr, temp, st));
      CU(launch_hamming_map(d_hoff, np, c0, a.n, d_map, ss.get<uint8_t>(temp), temp, st));
      a.map = d_map;
      ProfScope p(1, r.device, st);
      CU(edit ? launch_edit_verify(r.view, a, k, mode, r.sm_count, st) : launch_hamming_verify(r.view, a, k, mode, r.sm_count, st));
    }
  };
  if (dev) {  // 3. device-resident locate (DESIGN.md §1e)
    // count pass: the CSR over the queries, and the hit total that sizes the outputs (the second synchronisation)
    a.counts = sc.get<uint64_t>(nv * P);
    CU(cudaMemsetAsync(a.counts, 0, nv * P * 8, st));
    verify_all(VERIFY_COUNT);
    uint64_t* d_sums = sc.get<uint64_t>(nv + 1);
    CU(launch_hamming_row_sums(a.counts, k, nv, d_sums, st));
    CU(scan_u64(d_sums, dev->hit_off, nv + 1, nullptr, temp, st));
    CU(scan_u64(d_sums, dev->hit_off, nv + 1, sc.get<uint8_t>(temp), temp, st));
    uint64_t n = 0;
    CU(cudaMemcpyAsync(&n, dev->hit_off + nv, 8, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    if (n == 0) return;
    // CUB's segmented sort reads its offsets as int: more than 2^31 - 1 keys are sorted in parts cut at query
    // boundaries, which needs the offsets on the host (the only case that reads them back)
    std::vector<std::pair<uint64_t, uint64_t>> parts{{0, nv}};  // query ranges
    std::vector<uint64_t> off;
    if (n >= (1ull << 31)) {
      off.resize(nv + 1);
      CU(cudaMemcpyAsync(off.data(), dev->hit_off, (nv + 1) * 8, cudaMemcpyDeviceToHost, st));
      CU(cudaStreamSynchronize(st));
      parts.clear();
      for (uint64_t q0 = 0; q0 < nv;) {
        if (off[q0 + 1] - off[q0] >= (1ull << 31))
          fail(AWRY_ERR_NOMEM, "query %llu has %llu hits, more than one sort can order (2^31)",
               (unsigned long long)(uint64_t(check_base < 0 ? 0 : check_base) + (q0 >> shift)),
               (unsigned long long)(off[q0 + 1] - off[q0]));
        uint64_t q1 = q0 + 1;
        while (q1 < nv && off[q1 + 1] - off[q0] < (1ull << 31)) q1++;
        parts.push_back({q0, q1});
        q0 = q1;
      }
    }
    // the outputs (released in stream order unless the call succeeds), then the scratch the hit total sizes
    StreamScratch out(st);
    awry_hit* d_hits = nullptr;
    uint8_t* d_dist = nullptr;
    uint64_t *d_keys = nullptr, *d_sorted = nullptr;
    try {
      d_hits = out.get<awry_hit>(n);  // (16 spare bytes behind the last hit, as every hit buffer)
      if (dev->dist) d_dist = out.get<uint8_t>(n);
      d_keys = sc.get<uint64_t>(n);
      d_sorted = sc.get<uint64_t>(n);
    } catch (const ApiError& x) {
      if (x.code != AWRY_ERR_NOMEM) throw;
      fail(AWRY_ERR_NOMEM, "out of device memory for the %llu hits of this %s locate", (unsigned long long)n, what);
    }
    // place pass: the same slices and the same acceptance as the count pass; each key takes a slot of its query's range
    a.keys = d_keys;
    a.acc = sc.get<uint64_t>(nv);
    a.q0 = 0;
    a.hit_off = dev->hit_off;
    CU(cudaMemsetAsync(a.acc, 0, nv * 8, st));
    verify_all(VERIFY_PLACE);
    // order: a query's positions are distinct, so the sorted keys do not depend on the order the atomics gave
    for (const auto& [q0, q1] : parts) {
      const uint64_t b = off.empty() ? 0 : off[q0], m = off.empty() ? n : off[q1] - off[q0];
      StreamScratch ss(st);
      size_t t2 = 0;
      CU(sort_hamming_keys(d_keys + b, d_sorted + b, m, q1 - q0, dev->hit_off + q0, b, nullptr, t2, st));
      CU(sort_hamming_keys(d_keys + b, d_sorted + b, m, q1 - q0, dev->hit_off + q0, b, ss.get<uint8_t>(t2), t2, st));
    }
    CU(launch_hamming_decode(d_sorted, n, d_dist, st));
    CU(launch_map_locations(r.view, d_sorted, n, reinterpret_cast<uint64_t*>(d_hits), st));
    out.ptrs.clear();  // the caller's now
    *dev->hits = d_hits;
    if (dev->dist) *dev->dist = d_dist;
    *dev->n_hits = n;
    return;
  }
  if (!sink) {  // 3. count
    CU(cudaMemsetAsync(d_counts, 0, nv * P * 8, st));
    a.counts = d_counts;
    verify_all(VERIFY_COUNT);
    return;
  }
  // 3. locate: slices cut at read boundaries (a read with more candidates than a slice gets one of its own size)
  sink->off.reserve(sink->off.size() + nv);
  for (uint64_t q0 = 0; q0 < nv;) {
    uint64_t q1 = q0 + 1;
    while (q1 < nv && qcand[q1 + 1] - qcand[q0] <= S) q1++;
    const uint64_t c0 = qcand[q0], n = qcand[q1] - c0, nr = q1 - q0;
    if (n * slots >= (1ull << 31))  // (a slice is sorted per read by one CUB call, whose offsets are int)
      fail(AWRY_ERR_NOMEM, "query %llu has %llu candidate windows, more than one slice can sort (2^31)",
           (unsigned long long)(uint64_t(check_base < 0 ? 0 : check_base) + (q0 >> shift)), (unsigned long long)(n * slots));
    const uint64_t base = sink->hits.size();
    if (n == 0) {
      sink->off.insert(sink->off.end(), nr, base);
      q0 = q1;
      continue;
    }
    StreamScratch ss(st);
    a.c0 = c0;
    a.n = n;
    a.q0 = q0;
    uint32_t* d_map = ss.get<uint32_t>(n);
    CU(launch_hamming_map(d_hoff, np, c0, n, d_map, nullptr, temp, st));
    CU(launch_hamming_map(d_hoff, np, c0, n, d_map, ss.get<uint8_t>(temp), temp, st));
    a.map = d_map;
    a.keys = ss.get<uint64_t>(n * slots);
    a.acc = ss.get<uint64_t>(nr + 1);
    CU(cudaMemsetAsync(a.acc, 0, (nr + 1) * 8, st));
    {
      ProfScope p(1, r.device, st);
      CU(edit ? launch_edit_verify(r.view, a, k, VERIFY_LOCATE, r.sm_count, st)
              : launch_hamming_verify(r.view, a, k, VERIFY_LOCATE, r.sm_count, st));
    }
    uint64_t* d_sorted = ss.get<uint64_t>(n * slots);
    size_t t2 = 0;
    if (edit) {
      CU(sort_edit_keys(a.keys, d_sorted, n * slots, nr, d_qcand + q0, c0, uint32_t(slots), nullptr, t2, st));
      CU(sort_edit_keys(a.keys, d_sorted, n * slots, nr, d_qcand + q0, c0, uint32_t(slots), ss.get<uint8_t>(t2), t2, st));
    } else {
      CU(sort_hamming_keys(a.keys, d_sorted, n, nr, d_qcand + q0, c0, nullptr, t2, st));
      CU(sort_hamming_keys(a.keys, d_sorted, n, nr, d_qcand + q0, c0, ss.get<uint8_t>(t2), t2, st));
    }
    uint64_t* d_qh = ss.get<uint64_t>(nr + 1);
    size_t t3 = 0;
    CU(scan_u64(a.acc, d_qh, nr + 1, nullptr, t3, st));
    CU(scan_u64(a.acc, d_qh, nr + 1, ss.get<uint8_t>(t3), t3, st));
    std::vector<uint64_t> qh(nr + 1);
    CU(cudaMemcpyAsync(qh.data(), d_qh, (nr + 1) * 8, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    const uint64_t n_acc = qh[nr];
    if (n_acc) {
      uint64_t* d_pos = ss.get<uint64_t>(n_acc);
      uint8_t* d_dist = ss.get<uint8_t>(n_acc);
      uint64_t* d_hits = ss.get<uint64_t>(2 * n_acc);
      if (edit)
        CU(launch_edit_compact(d_sorted, d_map, n * slots, k, d_qcand, c0, q0, d_qh, d_pos, d_dist, st));
      else
        CU(launch_hamming_compact(d_sorted, d_map, n, k, d_qcand, c0, q0, d_qh, d_pos, d_dist, st));
      CU(launch_map_locations(r.view, d_pos, n_acc, d_hits, st));
      sink->hits.resize(base + n_acc);
      sink->dist.resize(base + n_acc);
      CU(cudaMemcpyAsync(sink->hits.data() + base, d_hits, n_acc * 16, cudaMemcpyDeviceToHost, st));
      CU(cudaMemcpyAsync(sink->dist.data() + base, d_dist, n_acc, cudaMemcpyDeviceToHost, st));
      g_prof.d2h += n_acc * 17;
      CU(cudaStreamSynchronize(st));
    }
    for (uint64_t i = 0; i < nr; i++) sink->off.push_back(base + qh[i]);
    q0 = q1;
  }
}

// reads [lo, hi) of host buffers on replica ri: chunks of reads uploaded and searched one after the other (the
// host path does not overlap copies with compute yet).  `strands`: a chunk of n reads fills 2 n result slots.
void hamming_on_replica(const awry_index* ix, size_t ri, const uint8_t* qbytes, const uint64_t* qoff, uint64_t lo,
                        uint64_t hi, uint32_t k, uint64_t* counts, HammingSink* sink, bool strands = false,
                        Metric metric = METRIC_HAMMING) {
  if (lo >= hi) return;
  Replica& r = *ix->reps[ri];
  DeviceGuard dg(r.device);
  const uint64_t max_bytes = std::min(chunk_max_bytes(), locate_chunk_bytes());
  if (qoff[hi] < qoff[lo]) fail(AWRY_ERR_INVALID_ARG, "query offsets are not monotone (queries %llu..%llu)",
                                (unsigned long long)lo, (unsigned long long)hi);
  auto chunks = make_chunks(qoff, lo, hi, locate_chunk_q(), max_bytes);
  validate_chunks(chunks, max_bytes);
  Workspace* ws = r.acquire();
  try {
    for (const Chunk& c : chunks) {
      const uint64_t n = c.q1 - c.q0, nbytes = c.b1 - c.b0;
      Workspace::grow_dev(ws->d_qbytes, ws->d_qbytes_cap, size_t(nbytes) + 16);
      Workspace::grow_dev(ws->d_qoff, ws->d_qoff_cap, size_t(n) + 1);
      if (nbytes) CU(cudaMemcpyAsync(ws->d_qbytes, qbytes + c.b0, nbytes, cudaMemcpyHostToDevice, ws->st));
      CU(cudaMemcpyAsync(ws->d_qoff, qoff + c.q0, (n + 1) * 8, cudaMemcpyHostToDevice, ws->st));
      g_prof.h2d += nbytes + (n + 1) * 8;
      CU(cudaMemsetAsync(ws->d_flag, 0xff, 8, ws->st));
      if (sink) {
        hamming_run(r, ws->d_qbytes - c.b0, ws->d_qoff, n, c.b0, c.b1, k, ws->d_flag, (long long)c.q0, ws->st, nullptr, sink,
                    strands, metric);
      } else {
        StreamScratch sc(ws->st);
        const uint64_t slots = (strands ? 2 : 1) * (k + 1);  // counts per read
        uint64_t* d_counts = sc.get<uint64_t>(n * slots);
        hamming_run(r, ws->d_qbytes - c.b0, ws->d_qoff, n, c.b0, c.b1, k, ws->d_flag, (long long)c.q0, ws->st, d_counts, nullptr,
                    strands, metric);
        CU(cudaMemcpyAsync(counts + c.q0 * slots, d_counts, n * slots * 8, cudaMemcpyDeviceToHost, ws->st));
        g_prof.d2h += n * slots * 8;
      }
      CU(cudaStreamSynchronize(ws->st));
    }
  } catch (...) {
    cudaStreamSynchronize(ws->st);
    r.release(ws);
    throw;
  }
  r.release(ws);
}

// ------------------------------------------------------------------ both strands (awry_*_strands)

void strands_check_index(const awry_index* ix) {
  if (ix->alphabet != AWRY_NUCLEOTIDE) fail(AWRY_ERR_UNSUPPORTED, "both-strand search exists for the nucleotide alphabet only");
}

void strands_check_device_batch(uint64_t nq) {
  if (2 * nq >= (1ull << 32) - (1u << 24))  // (the search kernels' 32-bit ticket counter)
    fail(AWRY_ERR_INVALID_ARG, "batch too large for one both-strand search (%llu reads): split it", (unsigned long long)nq);
}

// the bound on k of each metric (the same number, named after its argument)
void check_max_k(uint32_t k, Metric metric) {
  if (metric == METRIC_EDIT) {
    if (k > AWRY_EDIT_MAX) fail(AWRY_ERR_INVALID_ARG, "max_edits must be 0 .. %d", AWRY_EDIT_MAX);
  } else if (k > AWRY_HAMMING_MAX) {
    fail(AWRY_ERR_INVALID_ARG, "max_mismatches must be 0 .. %d", AWRY_HAMMING_MAX);
  }
}

// awry_count_batch_{hamming,edit}[_strands]: counts (nq or 2 nq virtual queries) x (k+1)
void hamming_count_impl(const awry_index* ix, const uint8_t* qbytes, const uint64_t* qoff, uint64_t nq, uint32_t k,
                        uint64_t* counts, bool strands, Metric metric = METRIC_HAMMING) {
  need(ix);
  check_max_k(k, metric);
  if (nq == 0) return;
  if (!qbytes || !qoff || !counts) fail(AWRY_ERR_INVALID_ARG, "null argument");
  if (strands) strands_check_index(ix);
  hamming_check_index(ix, metric_name(metric));
  for_each_replica_range(ix, qoff, nq, [&](size_t ri, uint64_t lo, uint64_t hi) {
    hamming_on_replica(ix, ri, qbytes, qoff, lo, hi, k, counts, nullptr, strands, metric);
  });
}

// awry_locate_batch_{hamming,edit}[_strands]: hit_off is the CSR over the nq (or 2 nq virtual) queries
void hamming_locate_impl(const awry_index* ix, const uint8_t* qbytes, const uint64_t* qoff, uint64_t nq, uint32_t k,
                         uint64_t* hit_off, awry_hit* hits, uint8_t* hit_mismatches, uint64_t capacity, uint64_t* n_hits,
                         bool strands, Metric metric = METRIC_HAMMING) {
  need(ix);
  check_max_k(k, metric);
  if (!hit_off || !n_hits || (!hits && capacity)) fail(AWRY_ERR_INVALID_ARG, "null argument");
  *n_hits = 0;
  hit_off[0] = 0;
  if (nq == 0) return;
  if (!qbytes || !qoff) fail(AWRY_ERR_INVALID_ARG, "null argument");
  if (strands) strands_check_index(ix);
  hamming_check_index(ix, metric_name(metric));
  const uint64_t per = strands ? 2 : 1;  // result slots per read
  const size_t nr = ix->reps.size();
  std::vector<HammingSink> sinks(nr);
  std::vector<std::pair<uint64_t, uint64_t>> ranges(nr, {0, 0});
  for_each_replica_range(ix, qoff, nq, [&](size_t ri, uint64_t lo, uint64_t hi) {
    ranges[ri] = {lo, hi};
    hamming_on_replica(ix, ri, qbytes, qoff, lo, hi, k, nullptr, &sinks[ri], strands, metric);
  });
  // the replicas' CSRs, concatenated in range order; hits past `capacity` are dropped (the total still counts them)
  uint64_t total = 0;
  for (size_t ri = 0; ri < nr; ri++) {
    const auto [lo, hi] = ranges[ri];
    const HammingSink& s = sinks[ri];
    for (uint64_t i = 0; i < per * (hi - lo); i++) hit_off[per * lo + i] = total + s.off[i];
    const uint64_t n = s.hits.size(), fit = capacity > total ? std::min(n, capacity - total) : 0;
    if (fit) {
      memcpy(hits + total, s.hits.data(), fit * sizeof(awry_hit));
      if (hit_mismatches) memcpy(hit_mismatches + total, s.dist.data(), fit);
    }
    total += n;
  }
  hit_off[per * nq] = total;
  *n_hits = total;
  if (total > capacity)
    fail(AWRY_ERR_CAPACITY, "hit buffer holds %llu entries, %llu needed", (unsigned long long)capacity,
         (unsigned long long)total);
}

// ------------------------------------------------------------------ device-resident batches (awry_*_device*)
// What the prepass refuses stays latched in r.d_async_flag for awry_device_check.

// the first and last offset of a device-resident batch (one 16-byte read-back), checked; both strands also need the
// virtual offsets 2 e to fit
void device_batch_ends(const uint64_t* d_qoff, uint64_t nq, cudaStream_t st, uint64_t ends[2], bool strands) {
  CU(cudaMemcpyAsync(&ends[0], d_qoff, 8, cudaMemcpyDeviceToHost, st));
  CU(cudaMemcpyAsync(&ends[1], d_qoff + nq, 8, cudaMemcpyDeviceToHost, st));
  CU(cudaStreamSynchronize(st));
  if (ends[1] < ends[0]) fail(AWRY_ERR_INVALID_ARG, "query offsets are not monotone");
  if (strands && ends[1] >= (1ull << 62)) fail(AWRY_ERR_INVALID_ARG, "query offsets beyond 2^62");
}

// awry_count_device[_strands]: counts of the nq (or 2 nq virtual) queries
void count_device_impl(const awry_index* ix, int replica, const uint8_t* d_qbytes, const uint64_t* d_qoff, uint64_t nq,
                       uint64_t* d_counts, void* cuda_stream, bool strands) {
  need(ix);
  if (replica < 0 || size_t(replica) >= ix->reps.size()) fail(AWRY_ERR_INVALID_ARG, "replica out of range");
  if (strands) strands_check_index(ix);
  if (nq == 0) return;
  if (!d_qbytes || !d_qoff || !d_counts) fail(AWRY_ERR_INVALID_ARG, "null argument");
  if (strands) strands_check_device_batch(nq);
  Replica& r = *ix->reps[size_t(replica)];
  DeviceGuard dg(r.device);
  cudaStream_t st = static_cast<cudaStream_t>(cuda_stream);
  uint64_t e[2] = {0, 0};
  device_batch_ends(d_qoff, nq, st, e, strands);
  const uint64_t nv = strands ? 2 * nq : nq;
  const uint64_t w = query_words(ix->alphabet, nq, e[0], e[1]);
  const uint64_t vw = strands ? query_words(AWRY_NUCLEOTIDE, nv, 2 * e[0], 2 * e[1]) : 0, vo = strands ? nv + 1 : 0;
  uint64_t* buf = nullptr;  // one stream-ordered allocation: read words, [virtual words, virtual offsets,] defer list
  CU(cudaMallocAsync(reinterpret_cast<void**>(&buf), (w + vw + vo) * 8 + defer_words(nv) * 4, st));
  try {
    search_reads(r, d_qbytes, d_qoff, nq, e[0], e[1], strands, OUT_COUNT_U64,
                 SearchBuffers{buf, buf + w + vw, buf + w, d_counts, reinterpret_cast<uint32_t*>(buf + w + vw + vo),
                               r.d_async_flag},
                 st);
  } catch (...) {
    cudaFreeAsync(buf, st);
    throw;
  }
  CU(cudaFreeAsync(buf, st));
}

// awry_locate_device[_strands]: the hits of the nq (or 2 nq virtual) queries, in a stream-ordered device buffer
void locate_device_impl(const awry_index* ix, int replica, const uint8_t* d_qbytes, const uint64_t* d_qoff, uint64_t nq,
                        uint32_t flags, uint64_t* d_hit_off, awry_hit** d_hits, uint64_t* n_hits, void* cuda_stream,
                        bool strands) {
  need(ix);
  if (replica < 0 || size_t(replica) >= ix->reps.size()) fail(AWRY_ERR_INVALID_ARG, "replica out of range");
  if (!d_hit_off || !d_hits || !n_hits) fail(AWRY_ERR_INVALID_ARG, "null argument");
  *d_hits = nullptr;
  *n_hits = 0;
  if (strands) strands_check_index(ix);
  if (nq == 0) return;
  if (!d_qbytes || !d_qoff) fail(AWRY_ERR_INVALID_ARG, "null argument");
  if (strands) strands_check_device_batch(nq);
  Replica& r = *ix->reps[size_t(replica)];
  DeviceGuard dg(r.device);
  cudaStream_t st = static_cast<cudaStream_t>(cuda_stream);
  uint64_t e[2] = {0, 0};
  device_batch_ends(d_qoff, nq, st, e, strands);
  const uint64_t nv = strands ? 2 * nq : nq;
  Workspace* ws = r.acquire();
  try {
    const SearchBuffers b = workspace_buffers(ws, ix->alphabet, nq, e[0], e[1], strands, sp_cnt_bytes(r.view), r.d_async_flag);
    ws->sp_cnt_positions = search_reads(r, d_qbytes, d_qoff, nq, e[0], e[1], strands, OUT_SP_CNT_U32, b, st);
    uint64_t n = 0;
    uint64_t* h = locate_chunk_device(ix, r, ws, nv, flags, d_hit_off, &n, st);
    CU(cudaStreamSynchronize(st));
    *d_hits = reinterpret_cast<awry_hit*>(h);
    *n_hits = n;
  } catch (...) {
    cudaStreamSynchronize(st);
    r.release(ws);
    throw;
  }
  r.release(ws);
}

// awry_count_device_{hamming,edit}[_strands]: counts (nq or 2 nq virtual queries) x (k+1)
void hamming_count_device_impl(const awry_index* ix, int replica, const uint8_t* d_qbytes, const uint64_t* d_qoff,
                               uint64_t nq, uint32_t k, uint64_t* d_counts, void* cuda_stream, bool strands,
                               Metric metric = METRIC_HAMMING) {
  need(ix);
  check_max_k(k, metric);
  if (replica < 0 || size_t(replica) >= ix->reps.size()) fail(AWRY_ERR_INVALID_ARG, "replica out of range");
  if (nq == 0) return;
  if (!d_qbytes || !d_qoff || !d_counts) fail(AWRY_ERR_INVALID_ARG, "null argument");
  if (strands) strands_check_index(ix);
  hamming_check_index(ix, metric_name(metric));
  Replica& r = *ix->reps[size_t(replica)];
  DeviceGuard dg(r.device);
  cudaStream_t st = static_cast<cudaStream_t>(cuda_stream);
  uint64_t e[2] = {0, 0};
  device_batch_ends(d_qoff, nq, st, e, strands);
  hamming_run(r, d_qbytes, d_qoff, nq, e[0], e[1], k, r.d_async_flag, -1, st, d_counts, nullptr, strands, metric);
}

// awry_locate_device_{hamming,edit}[_strands]: the hits of the nq (or 2 nq virtual) queries, in stream-ordered device
// buffers; argument checks and errors as hamming_count_device_impl, outputs as locate_device_impl
void hamming_locate_device_impl(const awry_index* ix, int replica, const uint8_t* d_qbytes, const uint64_t* d_qoff,
                                uint64_t nq, uint32_t k, uint64_t* d_hit_off, awry_hit** d_hits, uint8_t** d_dist,
                                uint64_t* n_hits, void* cuda_stream, bool strands, Metric metric) {
  need(ix);
  check_max_k(k, metric);
  if (replica < 0 || size_t(replica) >= ix->reps.size()) fail(AWRY_ERR_INVALID_ARG, "replica out of range");
  if (!d_hit_off || !d_hits || !n_hits) fail(AWRY_ERR_INVALID_ARG, "null argument");
  *d_hits = nullptr;
  if (d_dist) *d_dist = nullptr;
  *n_hits = 0;
  if (nq == 0) return;
  if (!d_qbytes || !d_qoff) fail(AWRY_ERR_INVALID_ARG, "null argument");
  if (strands) strands_check_index(ix);
  hamming_check_index(ix, metric_name(metric));
  Replica& r = *ix->reps[size_t(replica)];
  DeviceGuard dg(r.device);
  cudaStream_t st = static_cast<cudaStream_t>(cuda_stream);
  uint64_t e[2] = {0, 0};
  device_batch_ends(d_qoff, nq, st, e, strands);
  DeviceHits out{d_hit_off, d_hits, d_dist, n_hits};
  hamming_run(r, d_qbytes, d_qoff, nq, e[0], e[1], k, r.d_async_flag, -1, st, nullptr, nullptr, strands, metric, &out);
}

// ------------------------------------------------------------------ alignment of located hits (awry_align_*)

// One batch of reads on one replica, on stream `st`: the prepass of hamming_run (the reads packed; both strands: the
// virtual offsets and words), each search query's length (0: refused), then the hits in slices of at most
// hamming_slice(): the query of every hit from the hit offsets (hamming_map's scatter and max-scan), and one
// alignment per hit.  d_hit_off (nv + 1) holds absolute hit indices; hit hit0 + i is d_hits[i] and gets d_out[i].
// `check_base` >= 0: a refused read fails the call, reported as read check_base + q; < 0: it stays latched in *d_flag.
void align_run(Replica& r, const uint8_t* d_qbytes, const uint64_t* d_qoff, uint64_t nq, uint64_t b_lo, uint64_t b_hi,
               Metric metric, bool strands, uint32_t k, unsigned long long* d_flag, long long check_base,
               const uint64_t* d_hit_off, uint64_t hit0, const awry_hit* d_hits, uint64_t n_hits, awry_alignment* d_out,
               cudaStream_t st) {
  const uint32_t shift = strands ? 1 : 0;
  const uint64_t nv = nq << shift, nbytes = b_hi - b_lo;
  StreamScratch sc(st);
  const uint64_t rw_n = packed_words(0, nq, nbytes), w_lo = 4 * (b_lo >> 6);
  const uint64_t v_lo = b_lo << shift, v_hi = b_hi << shift, vw_n = packed_words(0, nv, nbytes << shift), vw_lo = 4 * (v_lo >> 6);
  uint64_t* const d_rw = sc.get<uint64_t>(rw_n) - w_lo;
  const uint64_t *d_vw = d_rw, *d_voff = d_qoff;
  CU(launch_pack(AWRY_NUCLEOTIDE, d_qbytes, d_qoff, nq, d_rw, b_lo, b_hi, d_flag, st));
  if (strands) {
    uint64_t* const voff = sc.get<uint64_t>(nv + 1);
    uint64_t* const vw = sc.get<uint64_t>(vw_n) - vw_lo;
    CU(launch_strand_offsets(d_qoff, nq, b_lo, b_hi, voff, st));
    CU(launch_strand_words(d_rw, d_qoff, nq, b_lo, b_hi, voff, vw, st));
    d_voff = voff;
    d_vw = vw;
  }
  uint32_t* const d_qlen = sc.get<uint32_t>(nv);
  AlignSlice a{};
  a.qwords = d_vw;
  a.qw_lo = strands ? vw_lo : w_lo;
  a.qw_n = strands ? vw_n : rw_n;
  a.qoff = d_voff;
  a.qlen = d_qlen;
  a.nq = nv;
  a.hit_end = d_hit_off + nv;
  a.hit_total = hit0 + n_hits;
  CU(launch_align_reads(d_vw, d_voff, nv, v_lo, v_hi, a.qw_lo, a.qw_n, k, shift, d_qlen, d_flag, st));
  if (check_base >= 0) {
    unsigned long long flag = ~0ull;
    CU(cudaMemcpyAsync(&flag, d_flag, 8, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    if (flag != ~0ull && (flag & 1) == BAD_QUERY)
      fail(AWRY_ERR_INVALID_QUERY, "query %llu is empty, contains a sentinel ('$'/'#') or is not longer than k = %u",
           (unsigned long long)(uint64_t(check_base) + (flag >> 1)), k);
    if (flag != ~0ull) fail_bad_query(flag, uint64_t(check_base));
  }
  const uint64_t S = hamming_slice();
  for (uint64_t c0 = 0; c0 < n_hits; c0 += S) {
    StreamScratch ss(st);
    a.n = std::min(S, n_hits - c0);
    uint32_t* const d_map = ss.get<uint32_t>(a.n);
    size_t temp = 0;
    CU(launch_hamming_map(d_hit_off, nv, hit0 + c0, a.n, d_map, nullptr, temp, st));
    CU(launch_hamming_map(d_hit_off, nv, hit0 + c0, a.n, d_map, ss.get<uint8_t>(temp), temp, st));
    a.map = d_map;
    a.hits = reinterpret_cast<const uint64_t*>(d_hits + c0);
    a.out = reinterpret_cast<uint32_t*>(d_out + c0);
    ProfScope p(1, r.device, st);
    CU(launch_align_hits(r.view, a, k, metric == METRIC_EDIT, r.sm_count, st));
  }
}

// the checks both align calls make before touching the index
void align_check_args(uint32_t metric, uint32_t strands, uint32_t k) {
  if (metric > AWRY_METRIC_EDIT) fail(AWRY_ERR_INVALID_ARG, "metric must be AWRY_METRIC_HAMMING (0) or AWRY_METRIC_EDIT (1)");
  if (strands > 1) fail(AWRY_ERR_INVALID_ARG, "strands must be 0 or 1");
  check_max_k(k, Metric(metric));
}

void align_check_index(const awry_index* ix, uint64_t nv) {
  need(ix);
  hamming_check_index(ix, "alignment");
  if (nv >= (1ull << 32) - 1) fail(AWRY_ERR_INVALID_ARG, "batch too large for one alignment call: split it");
}

// awry_align_batch: reads [lo, hi) of host buffers on replica ri, in chunks of reads; each chunk uploads its reads, its
// part of hit_off and its hits, and copies its alignments back
void align_on_replica(const awry_index* ix, size_t ri, const uint8_t* qbytes, const uint64_t* qoff, uint64_t lo, uint64_t hi,
                      Metric metric, bool strands, uint32_t k, const uint64_t* hit_off, const awry_hit* hits,
                      awry_alignment* out) {
  if (lo >= hi) return;
  Replica& r = *ix->reps[ri];
  DeviceGuard dg(r.device);
  const uint64_t max_bytes = std::min(chunk_max_bytes(), locate_chunk_bytes()), per = strands ? 2 : 1;
  auto chunks = make_chunks(qoff, lo, hi, locate_chunk_q(), max_bytes);
  validate_chunks(chunks, max_bytes);
  Workspace* ws = r.acquire();
  try {
    for (const Chunk& c : chunks) {
      const uint64_t n = c.q1 - c.q0, nbytes = c.b1 - c.b0, v0 = per * c.q0, nv = per * n;
      const uint64_t h0 = hit_off[v0], nh = hit_off[v0 + nv] - h0;
      StreamScratch sc(ws->st);
      Workspace::grow_dev(ws->d_qbytes, ws->d_qbytes_cap, size_t(nbytes) + 16);
      Workspace::grow_dev(ws->d_qoff, ws->d_qoff_cap, size_t(n) + 1);
      uint64_t* const d_hoff = sc.get<uint64_t>(nv + 1);
      awry_hit* const d_hits = sc.get<awry_hit>(nh);
      awry_alignment* const d_out = sc.get<awry_alignment>(nh);
      if (nbytes) CU(cudaMemcpyAsync(ws->d_qbytes, qbytes + c.b0, nbytes, cudaMemcpyHostToDevice, ws->st));
      CU(cudaMemcpyAsync(ws->d_qoff, qoff + c.q0, (n + 1) * 8, cudaMemcpyHostToDevice, ws->st));
      CU(cudaMemcpyAsync(d_hoff, hit_off + v0, (nv + 1) * 8, cudaMemcpyHostToDevice, ws->st));
      if (nh) CU(cudaMemcpyAsync(d_hits, hits + h0, nh * sizeof(awry_hit), cudaMemcpyHostToDevice, ws->st));
      g_prof.h2d += nbytes + (n + 1) * 8 + (nv + 1) * 8 + nh * sizeof(awry_hit);
      CU(cudaMemsetAsync(ws->d_flag, 0xff, 8, ws->st));
      align_run(r, ws->d_qbytes - c.b0, ws->d_qoff, n, c.b0, c.b1, metric, strands, k, ws->d_flag, (long long)c.q0,
                d_hoff, h0, d_hits, nh, d_out, ws->st);
      if (nh) CU(cudaMemcpyAsync(out + h0, d_out, nh * sizeof(awry_alignment), cudaMemcpyDeviceToHost, ws->st));
      g_prof.d2h += nh * sizeof(awry_alignment);
      CU(cudaStreamSynchronize(ws->st));
    }
  } catch (...) {
    cudaStreamSynchronize(ws->st);
    r.release(ws);
    throw;
  }
  r.release(ws);
}

void align_batch_impl(const awry_index* ix, const uint8_t* qbytes, const uint64_t* qoff, uint64_t nq, uint32_t metric,
                      uint32_t strands, uint32_t k, const uint64_t* hit_off, const awry_hit* hits, awry_alignment* out) {
  align_check_args(metric, strands, k);
  if (!hit_off) fail(AWRY_ERR_INVALID_ARG, "null argument");
  const uint64_t nv = nq << strands;
  if (hit_off[0] != 0) fail(AWRY_ERR_INVALID_ARG, "hit_off[0] must be 0");
  for (uint64_t v = 0; v < nv; v++)
    if (hit_off[v + 1] < hit_off[v]) fail(AWRY_ERR_INVALID_ARG, "hit offsets are not monotone at query %llu", (unsigned long long)(v >> strands));
  if (nq && (!qbytes || !qoff)) fail(AWRY_ERR_INVALID_ARG, "null argument");
  if (hit_off[nv] && (!hits || !out)) fail(AWRY_ERR_INVALID_ARG, "null argument");
  align_check_index(ix, nv);
  if (nq == 0) return;
  if (qoff[nq] < qoff[0]) fail(AWRY_ERR_INVALID_ARG, "query offsets are not monotone");
  for_each_replica_range(ix, qoff, nq, [&](size_t ri, uint64_t lo, uint64_t hi) {
    align_on_replica(ix, ri, qbytes, qoff, lo, hi, Metric(metric), strands != 0, k, hit_off, hits, out);
  });
}

void align_device_impl(const awry_index* ix, int replica, const uint8_t* d_qbytes, const uint64_t* d_qoff, uint64_t nq,
                       uint32_t metric, uint32_t strands, uint32_t k, const uint64_t* d_hit_off, const awry_hit* d_hits,
                       uint64_t n_hits, awry_alignment* d_out, void* cuda_stream) {
  align_check_args(metric, strands, k);
  if (!d_hit_off || (nq && (!d_qbytes || !d_qoff)) || (n_hits && (!d_hits || !d_out)))
    fail(AWRY_ERR_INVALID_ARG, "null argument");
  align_check_index(ix, nq << strands);
  if (replica < 0 || size_t(replica) >= ix->reps.size()) fail(AWRY_ERR_INVALID_ARG, "replica out of range");
  if (nq == 0) return;
  if (strands) strands_check_device_batch(nq);
  Replica& r = *ix->reps[size_t(replica)];
  DeviceGuard dg(r.device);
  cudaStream_t st = static_cast<cudaStream_t>(cuda_stream);
  uint64_t e[2] = {0, 0};
  device_batch_ends(d_qoff, nq, st, e, strands != 0);
  align_run(r, d_qbytes, d_qoff, nq, e[0], e[1], Metric(metric), strands != 0, k, r.d_async_flag, -1, d_hit_off, 0, d_hits,
            n_hits, d_out, st);
}

// awry_alignment_cigar: run-length encoded op letters; '=' runs fill the query between the ops
void alignment_cigar_impl(const awry_alignment* a, uint32_t query_len, char* buf, size_t cap, size_t* needed) {
  if (!a || (!buf && cap)) fail(AWRY_ERR_INVALID_ARG, "null argument");
  if (a->n_ops != a->distance || a->n_ops > AWRY_EDIT_MAX)
    fail(AWRY_ERR_INVALID_ARG, "not an alignment (distance %u, %u ops)", unsigned(a->distance), unsigned(a->n_ops));
  std::string s;
  char last = 0;
  uint64_t run = 0, at = 0;  // query symbols used
  auto put = [&](char c, uint64_t n) {  // (adjacent ops of one kind merge: "2X")
    if (n == 0) return;
    if (c != last) {
      if (run) s += std::to_string(run) + last;
      last = c;
      run = 0;
    }
    run += n;
  };
  for (unsigned t = 0; t < a->n_ops; t++) {
    const awry_edit_op& o = a->ops[t];
    const bool uses_q = o.op == 'X' || o.op == 'I';
    if ((!uses_q && o.op != 'D') || o.qpos < at || o.qpos + (uses_q ? 1u : 0u) > query_len)
      fail(AWRY_ERR_INVALID_ARG, "op %u ('%c' at query position %u) is out of order or outside the query", t,
           o.op >= 32 && o.op < 127 ? char(o.op) : '?', o.qpos);
    put('=', o.qpos - at);
    put(char(o.op), 1);
    at = o.qpos + (uses_q ? 1 : 0);
  }
  put('=', query_len - at);
  if (run) s += std::to_string(run) + last;
  if (needed) *needed = s.size() + 1;
  if (s.size() + 1 > cap) fail(AWRY_ERR_CAPACITY, "the CIGAR needs %zu bytes, the buffer holds %zu", s.size() + 1, cap);
  memcpy(buf, s.c_str(), s.size() + 1);
}

}  // namespace host
}  // namespace awry

extern "C" {

int awry_count_batch(const awry_index* ix, const uint8_t* qbytes, const uint64_t* qoff, uint64_t nq, uint64_t* counts) {
  return guarded([&] {
    need(ix);
    if (nq == 0) return;
    if (!qbytes || !qoff || !counts) fail(AWRY_ERR_INVALID_ARG, "null argument");
    count_impl(ix, ascii_source(qbytes, qoff), nq, OUT_COUNT_U64, counts);
  });
}

int awry_search_batch(const awry_index* ix, const uint8_t* qbytes, const uint64_t* qoff, uint64_t nq, awry_range* ranges) {
  return guarded([&] {
    need(ix);
    if (nq == 0) return;
    if (!qbytes || !qoff || !ranges) fail(AWRY_ERR_INVALID_ARG, "null argument");
    count_impl(ix, ascii_source(qbytes, qoff), nq, OUT_RANGE_U64, ranges);
  });
}

int awry_count_batch_packed2(const awry_index* ix, const uint8_t* crumbs, const uint64_t* qoff, uint64_t nq,
                             const uint64_t* exceptions, uint64_t n_exc, uint64_t* counts) {
  return guarded([&] {
    need(ix);
    if (nq == 0) return;
    if (!counts) fail(AWRY_ERR_INVALID_ARG, "null argument");
    count_impl(ix, packed2_source(ix, crumbs, qoff, nq, exceptions, n_exc), nq, OUT_COUNT_U64, counts);
  });
}

int awry_locate_batch(const awry_index* ix, const uint8_t* qbytes, const uint64_t* qoff, uint64_t nq, uint32_t flags,
                      uint64_t* hit_off, awry_hit** hits, uint64_t* n_hits) {
  return guarded([&] {
    need(ix);
    if (!hit_off || !hits || !n_hits) fail(AWRY_ERR_INVALID_ARG, "null argument");
    *hits = nullptr;
    *n_hits = 0;
    hit_off[0] = 0;
    if (nq == 0) return;
    if (!qbytes || !qoff) fail(AWRY_ERR_INVALID_ARG, "null argument");
    locate_owned_impl(ix, ascii_source(qbytes, qoff), nq, flags, hit_off, hits, n_hits);
  });
}

void awry_hits_free(awry_hit* hits) { free(hits); }

int awry_locate_batch_into(const awry_index* ix, const uint8_t* qbytes, const uint64_t* qoff, uint64_t nq,
                           uint32_t flags, uint64_t* hit_off, awry_hit* hits, uint64_t capacity, uint64_t* n_hits) {
  return guarded([&] {
    need(ix);
    if (!hit_off || !n_hits || (!hits && capacity)) fail(AWRY_ERR_INVALID_ARG, "null argument");
    *n_hits = 0;
    hit_off[0] = 0;
    if (nq == 0) return;
    if (!qbytes || !qoff) fail(AWRY_ERR_INVALID_ARG, "null argument");
    locate_into_impl(ix, ascii_source(qbytes, qoff), nq, flags, hit_off, hits, capacity, n_hits);
  });
}

int awry_locate_batch_packed2(const awry_index* ix, const uint8_t* crumbs, const uint64_t* qoff, uint64_t nq,
                              const uint64_t* exceptions, uint64_t n_exc, uint32_t flags, uint64_t* hit_off,
                              awry_hit* hits, uint64_t capacity, uint64_t* n_hits) {
  return guarded([&] {
    need(ix);
    if (!hit_off || !n_hits || (!hits && capacity)) fail(AWRY_ERR_INVALID_ARG, "null argument");
    *n_hits = 0;
    hit_off[0] = 0;
    if (nq == 0) return;
    locate_into_impl(ix, packed2_source(ix, crumbs, qoff, nq, exceptions, n_exc), nq, flags, hit_off, hits, capacity, n_hits);
  });
}

int awry_count_device(const awry_index* ix, int replica, const uint8_t* d_qbytes, const uint64_t* d_qoff, uint64_t nq,
                      uint64_t* d_counts, void* cuda_stream) {
  return guarded([&] { count_device_impl(ix, replica, d_qbytes, d_qoff, nq, d_counts, cuda_stream, false); });
}

int awry_locate_device(const awry_index* ix, int replica, const uint8_t* d_qbytes, const uint64_t* d_qoff, uint64_t nq,
                       uint32_t flags, uint64_t* d_hit_off, awry_hit** d_hits, uint64_t* n_hits, void* cuda_stream) {
  return guarded([&] {
    locate_device_impl(ix, replica, d_qbytes, d_qoff, nq, flags, d_hit_off, d_hits, n_hits, cuda_stream, false);
  });
}

int awry_count_batch_hamming(const awry_index* ix, const uint8_t* qbytes, const uint64_t* qoff, uint64_t nq,
                             uint32_t max_mismatches, uint64_t* counts) {
  return guarded([&] { hamming_count_impl(ix, qbytes, qoff, nq, max_mismatches, counts, false); });
}

int awry_locate_batch_hamming(const awry_index* ix, const uint8_t* qbytes, const uint64_t* qoff, uint64_t nq,
                              uint32_t max_mismatches, uint64_t* hit_off, awry_hit* hits, uint8_t* hit_mismatches,
                              uint64_t capacity, uint64_t* n_hits) {
  return guarded([&] {
    hamming_locate_impl(ix, qbytes, qoff, nq, max_mismatches, hit_off, hits, hit_mismatches, capacity, n_hits, false);
  });
}

int awry_count_device_hamming(const awry_index* ix, int replica, const uint8_t* d_qbytes, const uint64_t* d_qoff,
                              uint64_t nq, uint32_t max_mismatches, uint64_t* d_counts, void* cuda_stream) {
  return guarded([&] {
    hamming_count_device_impl(ix, replica, d_qbytes, d_qoff, nq, max_mismatches, d_counts, cuda_stream, false);
  });
}

int awry_count_batch_hamming_strands(const awry_index* ix, const uint8_t* qbytes, const uint64_t* qoff, uint64_t nq,
                                     uint32_t max_mismatches, uint64_t* counts) {
  return guarded([&] { hamming_count_impl(ix, qbytes, qoff, nq, max_mismatches, counts, true); });
}

int awry_locate_batch_hamming_strands(const awry_index* ix, const uint8_t* qbytes, const uint64_t* qoff, uint64_t nq,
                                      uint32_t max_mismatches, uint64_t* hit_off, awry_hit* hits, uint8_t* hit_mismatches,
                                      uint64_t capacity, uint64_t* n_hits) {
  return guarded([&] {
    hamming_locate_impl(ix, qbytes, qoff, nq, max_mismatches, hit_off, hits, hit_mismatches, capacity, n_hits, true);
  });
}

int awry_count_device_hamming_strands(const awry_index* ix, int replica, const uint8_t* d_qbytes, const uint64_t* d_qoff,
                                      uint64_t nq, uint32_t max_mismatches, uint64_t* d_counts, void* cuda_stream) {
  return guarded([&] {
    hamming_count_device_impl(ix, replica, d_qbytes, d_qoff, nq, max_mismatches, d_counts, cuda_stream, true);
  });
}

int awry_count_batch_edit(const awry_index* ix, const uint8_t* qbytes, const uint64_t* qoff, uint64_t nq,
                          uint32_t max_edits, uint64_t* counts) {
  return guarded([&] { hamming_count_impl(ix, qbytes, qoff, nq, max_edits, counts, false, METRIC_EDIT); });
}

int awry_locate_batch_edit(const awry_index* ix, const uint8_t* qbytes, const uint64_t* qoff, uint64_t nq,
                           uint32_t max_edits, uint64_t* hit_off, awry_hit* hits, uint8_t* hit_edits, uint64_t capacity,
                           uint64_t* n_hits) {
  return guarded([&] {
    hamming_locate_impl(ix, qbytes, qoff, nq, max_edits, hit_off, hits, hit_edits, capacity, n_hits, false, METRIC_EDIT);
  });
}

int awry_count_device_edit(const awry_index* ix, int replica, const uint8_t* d_qbytes, const uint64_t* d_qoff,
                           uint64_t nq, uint32_t max_edits, uint64_t* d_counts, void* cuda_stream) {
  return guarded([&] {
    hamming_count_device_impl(ix, replica, d_qbytes, d_qoff, nq, max_edits, d_counts, cuda_stream, false, METRIC_EDIT);
  });
}

int awry_count_batch_edit_strands(const awry_index* ix, const uint8_t* qbytes, const uint64_t* qoff, uint64_t nq,
                                  uint32_t max_edits, uint64_t* counts) {
  return guarded([&] { hamming_count_impl(ix, qbytes, qoff, nq, max_edits, counts, true, METRIC_EDIT); });
}

int awry_locate_batch_edit_strands(const awry_index* ix, const uint8_t* qbytes, const uint64_t* qoff, uint64_t nq,
                                   uint32_t max_edits, uint64_t* hit_off, awry_hit* hits, uint8_t* hit_edits,
                                   uint64_t capacity, uint64_t* n_hits) {
  return guarded([&] {
    hamming_locate_impl(ix, qbytes, qoff, nq, max_edits, hit_off, hits, hit_edits, capacity, n_hits, true, METRIC_EDIT);
  });
}

int awry_count_device_edit_strands(const awry_index* ix, int replica, const uint8_t* d_qbytes, const uint64_t* d_qoff,
                                   uint64_t nq, uint32_t max_edits, uint64_t* d_counts, void* cuda_stream) {
  return guarded([&] {
    hamming_count_device_impl(ix, replica, d_qbytes, d_qoff, nq, max_edits, d_counts, cuda_stream, true, METRIC_EDIT);
  });
}

int awry_locate_device_hamming(const awry_index* ix, int replica, const uint8_t* d_qbytes, const uint64_t* d_qoff,
                               uint64_t nq, uint32_t max_mismatches, uint64_t* d_hit_off, awry_hit** d_hits,
                               uint8_t** d_hit_mismatches, uint64_t* n_hits, void* cuda_stream) {
  return guarded([&] {
    hamming_locate_device_impl(ix, replica, d_qbytes, d_qoff, nq, max_mismatches, d_hit_off, d_hits, d_hit_mismatches,
                               n_hits, cuda_stream, false, METRIC_HAMMING);
  });
}

int awry_locate_device_hamming_strands(const awry_index* ix, int replica, const uint8_t* d_qbytes, const uint64_t* d_qoff,
                                       uint64_t nq, uint32_t max_mismatches, uint64_t* d_hit_off, awry_hit** d_hits,
                                       uint8_t** d_hit_mismatches, uint64_t* n_hits, void* cuda_stream) {
  return guarded([&] {
    hamming_locate_device_impl(ix, replica, d_qbytes, d_qoff, nq, max_mismatches, d_hit_off, d_hits, d_hit_mismatches,
                               n_hits, cuda_stream, true, METRIC_HAMMING);
  });
}

int awry_locate_device_edit(const awry_index* ix, int replica, const uint8_t* d_qbytes, const uint64_t* d_qoff,
                            uint64_t nq, uint32_t max_edits, uint64_t* d_hit_off, awry_hit** d_hits,
                            uint8_t** d_hit_edits, uint64_t* n_hits, void* cuda_stream) {
  return guarded([&] {
    hamming_locate_device_impl(ix, replica, d_qbytes, d_qoff, nq, max_edits, d_hit_off, d_hits, d_hit_edits, n_hits,
                               cuda_stream, false, METRIC_EDIT);
  });
}

int awry_locate_device_edit_strands(const awry_index* ix, int replica, const uint8_t* d_qbytes, const uint64_t* d_qoff,
                                    uint64_t nq, uint32_t max_edits, uint64_t* d_hit_off, awry_hit** d_hits,
                                    uint8_t** d_hit_edits, uint64_t* n_hits, void* cuda_stream) {
  return guarded([&] {
    hamming_locate_device_impl(ix, replica, d_qbytes, d_qoff, nq, max_edits, d_hit_off, d_hits, d_hit_edits, n_hits,
                               cuda_stream, true, METRIC_EDIT);
  });
}

int awry_align_batch(const awry_index* ix, const uint8_t* qbytes, const uint64_t* qoff, uint64_t nq, uint32_t metric,
                     uint32_t strands, uint32_t k, const uint64_t* hit_off, const awry_hit* hits, awry_alignment* out) {
  return guarded([&] { align_batch_impl(ix, qbytes, qoff, nq, metric, strands, k, hit_off, hits, out); });
}

int awry_align_device(const awry_index* ix, int replica, const uint8_t* d_qbytes, const uint64_t* d_qoff, uint64_t nq,
                      uint32_t metric, uint32_t strands, uint32_t k, const uint64_t* d_hit_off, const awry_hit* d_hits,
                      uint64_t n_hits, awry_alignment* d_out, void* cuda_stream) {
  return guarded([&] {
    align_device_impl(ix, replica, d_qbytes, d_qoff, nq, metric, strands, k, d_hit_off, d_hits, n_hits, d_out, cuda_stream);
  });
}

int awry_alignment_cigar(const awry_alignment* a, uint32_t query_len, char* buf, size_t cap, size_t* needed) {
  return guarded([&] { alignment_cigar_impl(a, query_len, buf, cap, needed); });
}

int awry_count_batch_strands(const awry_index* ix, const uint8_t* qbytes, const uint64_t* qoff, uint64_t nq,
                             uint64_t* counts) {
  return guarded([&] {
    need(ix);
    strands_check_index(ix);
    if (nq == 0) return;
    if (!qbytes || !qoff || !counts) fail(AWRY_ERR_INVALID_ARG, "null argument");
    QuerySource qs = ascii_source(qbytes, qoff);
    qs.strands = true;
    count_impl(ix, qs, nq, OUT_COUNT_U64, counts);
  });
}

int awry_locate_batch_strands(const awry_index* ix, const uint8_t* qbytes, const uint64_t* qoff, uint64_t nq,
                              uint32_t flags, uint64_t* hit_off, awry_hit* hits, uint64_t capacity, uint64_t* n_hits) {
  return guarded([&] {
    need(ix);
    if (!hit_off || !n_hits || (!hits && capacity)) fail(AWRY_ERR_INVALID_ARG, "null argument");
    *n_hits = 0;
    hit_off[0] = 0;
    strands_check_index(ix);
    if (nq == 0) return;
    if (!qbytes || !qoff) fail(AWRY_ERR_INVALID_ARG, "null argument");
    QuerySource qs = ascii_source(qbytes, qoff);
    qs.strands = true;
    locate_into_impl(ix, qs, nq, flags, hit_off, hits, capacity, n_hits);
  });
}

int awry_count_device_strands(const awry_index* ix, int replica, const uint8_t* d_qbytes, const uint64_t* d_qoff,
                              uint64_t nq, uint64_t* d_counts, void* cuda_stream) {
  return guarded([&] { count_device_impl(ix, replica, d_qbytes, d_qoff, nq, d_counts, cuda_stream, true); });
}

int awry_locate_device_strands(const awry_index* ix, int replica, const uint8_t* d_qbytes, const uint64_t* d_qoff,
                               uint64_t nq, uint32_t flags, uint64_t* d_hit_off, awry_hit** d_hits, uint64_t* n_hits,
                               void* cuda_stream) {
  return guarded([&] {
    locate_device_impl(ix, replica, d_qbytes, d_qoff, nq, flags, d_hit_off, d_hits, n_hits, cuda_stream, true);
  });
}

int awry_device_free(const awry_index* ix, int replica, void* d_ptr) {
  return guarded([&] {
    need(ix);
    if (replica < 0 || size_t(replica) >= ix->reps.size()) fail(AWRY_ERR_INVALID_ARG, "replica out of range");
    if (!d_ptr) return;
    DeviceGuard dg(ix->reps[size_t(replica)]->device);
    CU(cudaFreeAsync(d_ptr, nullptr));  // came from the stream-ordered pool
  });
}

int awry_device_check(const awry_index* ix, int replica, void* cuda_stream) {
  return guarded([&] {
    need(ix);
    if (replica < 0 || size_t(replica) >= ix->reps.size()) fail(AWRY_ERR_INVALID_ARG, "replica out of range");
    Replica& r = *ix->reps[size_t(replica)];
    DeviceGuard dg(r.device);
    cudaStream_t st = static_cast<cudaStream_t>(cuda_stream);
    unsigned long long flag = ~0ull;
    CU(cudaMemcpyAsync(&flag, r.d_async_flag, 8, cudaMemcpyDeviceToHost, st));
    CU(cudaMemsetAsync(r.d_async_flag, 0xff, 8, st));
    CU(cudaStreamSynchronize(st));
    if (flag != ~0ull) fail_bad_query(flag, 0);
  });
}

// ---- instrumentation ----

int awry_set_host_pack(int mode) {
  return guarded([&] {
    if (mode < -1 || mode > 1) fail(AWRY_ERR_INVALID_ARG, "host pack mode must be -1 (auto), 0 (off) or 1 (on)");
    g_host_pack = mode;
  });
}

int awry_host_pack_dna(const uint8_t* src, uint64_t n, uint8_t* dst, uint64_t* exceptions, uint64_t exc_cap, uint64_t* n_exc) {
  return guarded([&] {
    if (!src || !dst || !n_exc) fail(AWRY_ERR_INVALID_ARG, "null argument");
    std::vector<uint64_t> exc;
    host_pack_dna(src, size_t(n), dst, exc, 0);
    *n_exc = exc.size();
    if (exceptions)
      for (size_t i = 0; i < exc.size() && i < exc_cap; i++) exceptions[i] = exc[i];
  });
}

int awry_set_host_threads(int n) {
  return guarded([&] {
    if (n < 0 || n > 256) fail(AWRY_ERR_INVALID_ARG, "host thread count must be 0 (default) .. 256");
    host_set_threads(n);
  });
}

int awry_host_threads(void) { return host_pool_threads(); }

int awry_set_count_variant(int variant) {
  return guarded([&] {
    if (variant < 0 || variant > 1)
      fail(AWRY_ERR_INVALID_ARG, "count variant must be 0 (default: finish one-row intervals in the text) or 1 (backward search only)");
    g_count_variant = variant;
  });
}

int awry_set_locate_variant(int variant) {
  return guarded([&] {
    if (variant < 0 || variant > 2)
      fail(AWRY_ERR_INVALID_ARG, "locate variant must be 0 (default), 1 (LF-walk to row samples) or 2 (bounded walk)");
    g_locate_variant = variant;
  });
}

int awry_set_search_variant(int lanes_per_query, int threads_per_block, int blocks_per_sm) {
  if (lanes_per_query != 0 && lanes_per_query != -1 && lanes_per_query != 1 && lanes_per_query != 2 &&
      lanes_per_query != 4 && lanes_per_query != 8 && (lanes_per_query < 80 || lanes_per_query > 84))
    return AWRY_ERR_INVALID_ARG;
  int slots = -1;  // default choice of the pair kernel's flavour
  if (lanes_per_query >= 80) {  // 80 / 81 / 82: the pair kernel with 0 (branching refill) / 1 / 2 state-machine slots; 83 / 84: 1 / 2 slots at a lower residency
    slots = lanes_per_query - 80;
    lanes_per_query = 8;
  }
  store_variant(lanes_per_query, threads_per_block, blocks_per_sm, slots);
  return AWRY_OK;
}

}  // extern "C"
