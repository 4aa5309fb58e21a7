// host.hpp -- shared host-side internals of libawry_b200 (not part of the ABI): error handling, profiling
// accounting, per-call workspaces, device replicas and the helpers the translation units share.
//   api.cu        index lifetime: `.awry` loader, replicas, getters, single steps, instrumentation
//   batch.cu      batched count / locate pipelines (host buffers and device-resident entry points)
//   reads_api.cu  streaming FASTQ / FASTA front-end (host side of reads.cu)
//   build_api.cu  GPU index construction entry points (host side of build.cu)
#pragma once
#include <algorithm>
#include <atomic>
#include <cerrno>
#include <chrono>
#include <condition_variable>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <memory>
#include <mutex>
#include <stdexcept>
#include <string>
#include <thread>
#include <vector>

#include <fcntl.h>
#include <sys/stat.h>
#include <unistd.h>

#include "../../include/awry_b200.h"
#include "build.hpp"
#include "hostpack.hpp"
#include "kernels.hpp"
#include "reads.hpp"

namespace awry {
namespace host {


extern thread_local char g_err[1024];  // awry_last_error(): per thread

struct ApiError : std::runtime_error {
  int code;
  ApiError(int c, const std::string& m) : std::runtime_error(m), code(c) {}
};

[[noreturn]] void fail(int code, const char* fmt, ...);

#define CU(expr)                                                                          \
  do {                                                                                    \
    cudaError_t e__ = (expr);                                                             \
    if (e__ != cudaSuccess)                                                               \
      fail(AWRY_ERR_CUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e__), __FILE__, __LINE__); \
  } while (0)

template <class F>
int guarded(F&& f) {
  try {
    f();
    return AWRY_OK;
  } catch (const ApiError& e) {
    snprintf(g_err, sizeof g_err, "%s", e.what());
    return e.code;
  } catch (const std::bad_alloc&) {
    snprintf(g_err, sizeof g_err, "out of host memory");
    return AWRY_ERR_NOMEM;
  } catch (const std::exception& e) {
    snprintf(g_err, sizeof g_err, "%s", e.what());
    return AWRY_ERR_INVALID_ARG;
  } catch (...) {
    snprintf(g_err, sizeof g_err, "unknown error");
    return AWRY_ERR_INVALID_ARG;
  }
}

struct DeviceGuard {
  int prev = -1;
  explicit DeviceGuard(int dev) {
    cudaGetDevice(&prev);
    CU(cudaSetDevice(dev));
  }
  ~DeviceGuard() {
    if (prev >= 0) cudaSetDevice(prev);
  }
};

// ------------------------------------------------------------------ profiling

struct ProfState {
  std::mutex mu;
  bool enabled = false;
  struct Span {
    cudaEvent_t a, b;
    int kind;  // 0 search, 1 walk, 2 pack
    int device;
  };
  std::vector<Span> spans;
  uint64_t n[3] = {0, 0, 0};
  double ms[3] = {0, 0, 0};
  std::atomic<uint64_t> h2d{0}, d2h{0};
};
extern ProfState g_prof;

void prof_collect_locked();

struct ProfScope {
  bool on;
  cudaStream_t st;
  ProfState::Span sp{};
  ProfScope(int kind, int device, cudaStream_t s) : st(s) {
    on = g_prof.enabled;
    if (!on) return;
    sp.kind = kind;
    sp.device = device;
    cudaEventCreate(&sp.a);
    cudaEventCreate(&sp.b);
    cudaEventRecord(sp.a, st);
  }
  ~ProfScope() {
    if (!on) return;
    cudaEventRecord(sp.b, st);
    std::lock_guard<std::mutex> lk(g_prof.mu);
    g_prof.spans.push_back(sp);
    if (g_prof.spans.size() >= 8192) prof_collect_locked();  // nobody asked for a while: fold the events in
  }
};

// Process-wide EXPERIMENT knobs (awry_set_search_variant / _locate_variant / _host_pack): A/B switches for the
// benchmarks and tests, not per-call configuration -- results never depend on them, only speed.  Atomics, so
// that a thread flipping one while others search is a benign race: a call reads each knob once.
extern std::atomic<uint64_t> g_variant_bits;  // lanes (16 bits, biased by 1) | tpb (16) | blocks_per_sm (16) | slots (8, biased by 1)
extern std::atomic<int> g_host_pack;      // -1 = auto (AWRY_B200_HOST_PACK, CPU support, >= 4 pool threads), 0 = off, 1 = on
extern std::atomic<int> g_count_variant;   // 0 = finish one-row intervals in the text when it is on the device, 1 = backward search only
extern std::atomic<int> g_locate_variant;  // 0 = best pass 2 present, 1 = LF-walk to row samples, 2 = bounded walk
inline SearchVariant current_variant() {
  const uint64_t b = g_variant_bits.load(std::memory_order_relaxed);
  SearchVariant v;
  v.lanes = int(b & 0xffff) - 1;
  v.tpb = int((b >> 16) & 0xffff);
  v.blocks_per_sm = int((b >> 32) & 0xffff);
  v.slots = int((b >> 48) & 0xff) - 1;
  v.finish_in_text = g_count_variant.load(std::memory_order_relaxed) == 0;
  return v;
}
// locate pass 1 may store text positions (CNT_AT_TEXT_POS) when pass 2 will be the gather from the unsampled array
inline bool locate_positions_ok(const IndexView& view, const SearchVariant& v) {
  return view.rtext && view.full_sa && v.finish_in_text && g_locate_variant.load(std::memory_order_relaxed) == 0;
}
inline void store_variant(int lanes, int tpb, int blocks_per_sm, int slots) {
  g_variant_bits.store(uint64_t(uint16_t(lanes + 1)) | (uint64_t(uint16_t(tpb)) << 16) | (uint64_t(uint16_t(blocks_per_sm)) << 32) |
                           (uint64_t(uint8_t(slots + 1)) << 48),
                       std::memory_order_relaxed);
}


// ------------------------------------------------------------------ index

struct Workspace {
  int device = 0;
  cudaStream_t st = nullptr;
  cudaEvent_t done = nullptr;
  // pinned staging
  bool sp_cnt_positions = false;  // the (sp, count) pairs in d_out may hold text positions (CNT_AT_TEXT_POS): pass 2
                                  // must be the gather from the unsampled array
  uint8_t* h_qbytes = nullptr;
  size_t h_qbytes_cap = 0;
  uint64_t* h_qoff = nullptr;
  size_t h_qoff_cap = 0;  // entries
  uint8_t* h_out = nullptr;
  size_t h_out_cap = 0;  // bytes
  unsigned long long* h_flag = nullptr;
  unsigned long long* h_total = nullptr;  // hit total of a locate chunk (second word of the h_flag allocation)
  uint64_t* h_exc = nullptr;  // host-packed chunks: exception list (bytes outside ACGT)
  size_t h_exc_cap = 0;
  std::vector<uint64_t> exc_tmp;
  cudaEvent_t ev_a = nullptr, ev_b = nullptr;  // timing of a raw chunk's H2D copy (PackBalance)
  uint64_t link_probe_bytes = 0;
  cudaEvent_t ev_s0 = nullptr, ev_s1 = nullptr;  // timing of a chunk's search kernel (PackBalance: what the GPU consumes)
  uint64_t gpu_probe_bytes = 0;
  // device
  uint8_t* d_qbytes = nullptr;
  size_t d_qbytes_cap = 0;
  uint64_t* d_qoff = nullptr;
  size_t d_qoff_cap = 0;
  uint64_t* d_qwords = nullptr;
  size_t d_qwords_cap = 0;
  uint32_t* d_defer = nullptr;
  size_t d_defer_cap = 0;
  uint8_t* d_out = nullptr;
  size_t d_out_cap = 0;
  uint64_t* d_hit_off = nullptr;
  size_t d_hit_off_cap = 0;
  void* d_temp = nullptr;
  size_t d_temp_cap = 0;
  unsigned long long* d_flag = nullptr;
  uint64_t* d_exc = nullptr;
  size_t d_exc_cap = 0;
  // sync-free locate pass 2: [0] = this chunk's hit base, [1] = the call's running hit total (first slot's)
  unsigned long long* d_base = nullptr;
  cudaEvent_t ev_adv = nullptr;  // recorded after the chunk's advance_hit_base_kernel
  uint64_t* d_off_out = nullptr;  // rebased CSR offsets of the chunk, on their way to the caller
  size_t d_off_out_cap = 0;
  uint64_t* d_voff = nullptr;  // both strands: the chunk's virtual offsets and words (kernels.hpp)
  size_t d_voff_cap = 0;
  uint64_t* d_vwords = nullptr;
  size_t d_vwords_cap = 0;
  // reads-file front-end scratch, kept across calls (pinned allocations cost ~0.4 ms per MiB)
  struct ReadsScratch {
    uint64_t chunk = 0, carry = 0;
    uint8_t* h_buf[3] = {nullptr, nullptr, nullptr};
    uint8_t *d_raw = nullptr, *d_raw_b = nullptr, *d_qbytes = nullptr;  // raw chunks: double-buffered
    cudaStream_t st_in = nullptr;                                        // upload stream of the raw chunks
    cudaEvent_t ev_in[2] = {nullptr, nullptr};
    uint32_t *d_nl = nullptr, *d_small = nullptr, *d_seq_len = nullptr, *d_is_hdr = nullptr, *d_hdr_rank = nullptr;
    uint64_t *d_seq_off = nullptr, *d_qoff = nullptr;
    size_t cap_lines = 0, cap_qoff = 0, temp_bytes = 0;
    void* d_temp = nullptr;
    void* h_plan = nullptr;
    void release() {
      for (auto& b : h_buf) {
        cudaFreeHost(b);
        b = nullptr;
      }
      cudaFree(d_raw);
      cudaFree(d_raw_b);
      if (st_in) cudaStreamDestroy(st_in);
      for (auto& e : ev_in)
        if (e) cudaEventDestroy(e);
      cudaFree(d_qbytes);
      cudaFree(d_nl);
      cudaFree(d_small);
      cudaFree(d_seq_len);
      cudaFree(d_is_hdr);
      cudaFree(d_hdr_rank);
      cudaFree(d_seq_off);
      cudaFree(d_qoff);
      cudaFree(d_temp);
      cudaFreeHost(h_plan);
      *this = ReadsScratch();
    }
  } rs;

  template <class T>
  static void grow_dev(T*& p, size_t& cap, size_t need) {
    if (need <= cap) return;
    if (p) cudaFree(p);
    p = nullptr;
    cap = 0;
    size_t want = need + need / 8 + 256;
    CU(cudaMalloc(reinterpret_cast<void**>(&p), want * sizeof(T)));
    cap = want;
  }
  template <class T>
  static void grow_host(T*& p, size_t& cap, size_t need) {
    if (need <= cap) return;
    if (p) cudaFreeHost(p);
    p = nullptr;
    cap = 0;
    size_t want = need + need / 8 + 256;
    CU(cudaHostAlloc(reinterpret_cast<void**>(&p), want * sizeof(T), cudaHostAllocDefault));
    cap = want;
  }
  void init(int dev) {
    device = dev;
    CU(cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking));
    CU(cudaEventCreateWithFlags(&done, cudaEventDisableTiming));
    CU(cudaHostAlloc(reinterpret_cast<void**>(&h_flag), 2 * sizeof(unsigned long long), cudaHostAllocDefault));
    h_total = h_flag + 1;
    CU(cudaMalloc(reinterpret_cast<void**>(&d_flag), sizeof(unsigned long long)));
    CU(cudaMalloc(reinterpret_cast<void**>(&d_base), 2 * sizeof(unsigned long long)));
    CU(cudaEventCreateWithFlags(&ev_adv, cudaEventDisableTiming));
  }
  void destroy() {
    cudaSetDevice(device);
    if (st) cudaStreamSynchronize(st);
    cudaFreeHost(h_qbytes);
    cudaFreeHost(h_qoff);
    cudaFreeHost(h_out);
    cudaFreeHost(h_flag);
    cudaFreeHost(h_exc);
    cudaFree(d_exc);
    cudaFree(d_qbytes);
    cudaFree(d_qoff);
    cudaFree(d_qwords);
    cudaFree(d_defer);
    cudaFree(d_out);
    cudaFree(d_hit_off);
    cudaFree(d_temp);
    cudaFree(d_flag);
    cudaFree(d_base);
    cudaFree(d_off_out);
    cudaFree(d_voff);
    cudaFree(d_vwords);
    if (ev_adv) cudaEventDestroy(ev_adv);
    rs.release();
    if (ev_a) cudaEventDestroy(ev_a);
    if (ev_b) cudaEventDestroy(ev_b);
    if (ev_s0) cudaEventDestroy(ev_s0);
    if (ev_s1) cudaEventDestroy(ev_s1);
    if (done) cudaEventDestroy(done);
    if (st) cudaStreamDestroy(st);
  }
};

struct Replica {
  int device = 0;
  int sm_count = 148;
  uint4* d_blocks = nullptr;
  uint64_t* d_sa = nullptr;
  uint2* d_table = nullptr;
  uint4* d_pair = nullptr;
  uint32_t* d_full_sa = nullptr;  // unsampled suffix array (locate accelerator)
  uint8_t* d_rtext = nullptr;     // reversed 4-bit text (count accelerator, needs d_full_sa)
  size_t bytes_rtext = 0;
  uint4* d_walk = nullptr;        // memory-lean locate: walk blocks, mark ranks, position-sampled SA (layout.cuh)
  uint32_t* d_walk_rank = nullptr;
  uint32_t* d_pos_samples = nullptr;
  size_t bytes_lean = 0;
  uint64_t* d_seq_starts = nullptr;
  unsigned long long* d_async_flag = nullptr;  // first bad query seen by *_device calls
  size_t bytes_blocks = 0, bytes_sa = 0, bytes_table = 0, bytes_pair = 0, bytes_full_sa = 0;
  uint32_t c2[16] = {0};
  IndexView view{};
  // wide index (bwt_len >= 2^32 - 256): 64-bit row pointers, kernels_wide.cu; view.wide points at wview
  WideView wview{};
  ulonglong2* d_table_w = nullptr;  // k-mer seeds with 64-bit row pointers
  uint64_t* d_sb = nullptr;         // superblock counts the block counts are relative to
  uint64_t dollar_row = 0;
  std::mutex ws_mu;
  std::vector<Workspace*> free_ws;
  std::vector<Workspace*> all_ws;

  Workspace* acquire() {
    {
      std::lock_guard<std::mutex> lk(ws_mu);
      if (!free_ws.empty()) {
        Workspace* w = free_ws.back();
        free_ws.pop_back();
        return w;
      }
    }
    auto* w = new Workspace();
    w->init(device);
    std::lock_guard<std::mutex> lk(ws_mu);
    all_ws.push_back(w);
    return w;
  }
  void release(Workspace* w) {
    std::lock_guard<std::mutex> lk(ws_mu);
    free_ws.push_back(w);
  }
};

// Pack on the host or send ASCII?  Three rates decide, all MEASURED per replica of a handle and smoothed
// across its calls, in query bytes per second: H, what the host packs for this replica -- the POOL's rate (the
// host clock around the packer, times the parallel regions that shared the pool meanwhile) divided by the
// replicas of the call: a replica that timed only its own pack calls would see the pool whenever the others
// happen to be copying, overrate it, and all replicas together would pack 40 % of the bytes where 25 % is right
// (8 GPUs behind 32 cores: 0.95 G reads/s that way, profiles/r02_m8_bench_line_n8_before_global_balance.json);
// P, what its PCIe link
// moves raw (CUDA events around the copy of a raw first chunk); G, what its search kernel consumes (CUDA
// events around the kernel).  H >= 1.15 G: the host keeps the GPU fed on its own -- pack everything, a quarter
// of the bytes cross the link (one GPU behind 16 host threads: H = 121, G = 82 GB/s; mixing raw chunks in was
// measured and is worse there, a 128-MiB raw copy holds the copy engine for 2.6 ms,
// profiles/r01_s19_e2e_pack_share.log).  Otherwise host and link work side by side: a share f = H / (H + P)
// of the bytes is packed and the rest goes up as ASCII (the device packs it), so the GPU sees H + P -- several
// GPUs behind few cores (2 GPUs / 24 threads: H = 60-90 per replica against G = 82) are fed by both.
// AWRY_B200_PACK_SHARE=<0..1> pins the packed share of the bytes instead (experiments).
struct PackBalance {
  std::mutex mu;
  double host_rate = 0, link_rate = 0, gpu_rate = 0;  // bytes/s, 0 = not measured yet
  double fixed_share = -1;
  uint64_t calls = 0;
  bool mixed = true;  // AWRY_B200_PACK_MIXED=0: all-or-nothing
  PackBalance() {
    if (const char* e = getenv("AWRY_B200_PACK_SHARE")) fixed_share = std::min(1.0, std::max(0.0, atof(e)));
    if (const char* e = getenv("AWRY_B200_PACK_MIXED")) mixed = e[0] != '0';
  }
  void note_host(double bytes, double seconds, int sharers = 1) {  // host_rate: of the whole pool
    if (seconds <= 0 || bytes < (8 << 20)) return;
    std::lock_guard<std::mutex> lk(mu);
    double r = bytes / seconds * double(sharers < 1 ? 1 : sharers);
    host_rate = host_rate > 0 ? 0.7 * host_rate + 0.3 * r : r;
  }
  void note_link(double bytes, double seconds) {
    if (seconds <= 0 || bytes < (8 << 20)) return;
    std::lock_guard<std::mutex> lk(mu);
    double r = bytes / seconds;
    link_rate = link_rate > 0 ? 0.7 * link_rate + 0.3 * r : r;
  }
  void note_gpu(double bytes, double seconds) {
    if (seconds <= 0 || bytes < (8 << 20)) return;
    std::lock_guard<std::mutex> lk(mu);
    double r = bytes / seconds;
    gpu_rate = gpu_rate > 0 ? 0.7 * gpu_rate + 0.3 * r : r;
  }
  // per call: the packed share of the bytes and whether chunk 0 / chunk 1 serve as probes
  struct Plan {
    double share;
    bool probe_link, probe_host;
  };
  Plan plan(size_t n_replicas = 1) {
    std::lock_guard<std::mutex> lk(mu);
    if (fixed_share >= 0) return Plan{fixed_share, false, false};
    const bool refresh = calls++ % 32 == 0;
    if (this->host_rate <= 0 || link_rate <= 0) return Plan{1.0, true, true};
    const double host_rate = this->host_rate / double(n_replicas ? n_replicas : 1);  // this replica's share of the pool
    // (until the kernel's rate is known, "clearly faster than the link" stands in for "feeds the GPU")
    const bool host_suffices = gpu_rate > 0 ? host_rate >= 1.15 * gpu_rate : host_rate > 2.0 * link_rate;
    if (host_suffices) return Plan{1.0, refresh, false};
    if (!mixed) return host_rate > link_rate ? Plan{1.0, refresh, false} : Plan{0.0, true, refresh};
    // host and link side by side: a share f of the bytes is packed at host_rate and crosses the link as f / 4,
    // the rest crosses as it is -- f / host_rate = (1 - 0.75 f) / link_rate
    double f = host_rate / (link_rate + 0.75 * host_rate);
    if (f < 0.15) f = 0.0;
    if (f > 0.9) f = 1.0;
    return Plan{f, true, f == 0.0 && refresh};
  }
};

}  // namespace host
}  // namespace awry

struct awry_index {
  uint64_t version = 1, sa_ratio = 0, bwt_len = 0;
  int alphabet = 0;
  int card = 6;
  uint32_t kmer_len_file = 0, kmer_len_dev = 0;
  uint64_t prefix_sums[23] = {0};
  uint64_t n_sa_words = 0;
  uint32_t sa_bits = 0;
  uint32_t lean_ratio = 0;  // sampling distance of the derived position-sampled suffix array (0 = not built)
  bool wide = false;        // 64-bit row pointers (bwt_len >= 2^32 - 256, or AWRY_B200_WIDE=1)
  uint32_t sb_shift = 31;   // log2(rows per superblock) of a wide index
  uint64_t n_superblocks() const { return (bwt_len >> sb_shift) + 1; }
  std::vector<uint64_t> seq_starts;
  std::vector<std::string> headers;
  std::vector<std::unique_ptr<awry::host::Replica>> reps;
  // per replica: host-pack vs raw-copy balance (measured rates; the only mutable state of a handle)
  mutable std::vector<std::unique_ptr<awry::host::PackBalance>> balance;
  awry::host::PackBalance& balance_of(size_t replica) const { return *balance[replica]; }
};

namespace awry {
namespace host {

// ---- api.cu
uint32_t bits_per_element(uint64_t bwt_len);                  // compressed_suffix_array.rs:124-130
uint64_t sa_word_len(uint64_t bwt_len, uint64_t ratio);        // compressed_suffix_array.rs:113-123
uint64_t ipow(uint64_t b, uint32_t e);
unsigned io_threads();  // threads of a parallel positional read (AWRY_B200_IO_THREADS, default min(8, cores))
// sequential byte source: a file (FmIndex::load) or caller memory sections (FmIndex::new hand-over)
struct Source {
  FILE* f = nullptr;
  // arrays already on replica 0's device in the reference layout (awry_index_build): no staging
  const uint64_t* dev_blocks = nullptr;
  const uint64_t* dev_sa = nullptr;
  std::vector<std::pair<const uint8_t*, size_t>> segs;
  size_t cur = 0, off = 0;
  void read(void* dst, size_t n, const char* what) {
    if (n == 0) return;
    if (f) {
      if (n >= (32u << 20)) {
        // large sections (blocks, SA words): positional reads from several threads -- one thread
        // copying out of the page cache tops out at a few GB/s, far below the PCIe rate behind it
        off_t pos = ftello(f);
        int fd = fileno(f);
        unsigned nt = io_threads();
        size_t per = ((n + nt - 1) / nt + 4095) & ~size_t(4095);
        std::vector<std::thread> th;
        std::vector<int> ok(nt, 1);
        for (unsigned t = 0; t < nt; t++) {
          size_t lo = std::min(n, size_t(t) * per), hi = std::min(n, lo + per);
          if (lo >= hi) break;
          th.emplace_back([=, &ok] {
            size_t done = lo;
            while (done < hi) {
              ssize_t r = pread(fd, static_cast<char*>(dst) + done, hi - done, pos + off_t(done));
              if (r <= 0) {
                ok[t] = 0;
                return;
              }
              done += size_t(r);
            }
          });
        }
        for (auto& t : th) t.join();
        for (unsigned t = 0; t < nt; t++)
          if (!ok[t]) fail(AWRY_ERR_IO, "unexpected end of file while reading %s", what);
        if (fseeko(f, pos + off_t(n), SEEK_SET) != 0) fail(AWRY_ERR_IO, "seek failed while reading %s", what);
        return;
      }
      if (fread(dst, 1, n, f) != n) fail(AWRY_ERR_IO, "unexpected end of file while reading %s", what);
      return;
    }
    uint8_t* d = static_cast<uint8_t*>(dst);
    while (n) {
      if (cur >= segs.size()) fail(AWRY_ERR_INVALID_ARG, "index parts too short while reading %s", what);
      size_t take = std::min(segs[cur].second - off, n);
      memcpy(d, segs[cur].first + off, take);
      off += take;
      d += take;
      n -= take;
      if (off == segs[cur].second) {
        cur++;
        off = 0;
      }
    }
  }
};

extern thread_local bool g_skip_accelerators;  // replicas that exist only to fill a file's k-mer table section
std::vector<int> pick_devices(const int* devices, int n_dev);
void check_header(awry_index* ix);
void make_replicas(awry_index* ix, const std::vector<int>& devs, Source& src, bool from_file);
inline const awry_index* need(const awry_index* ix) {
  if (!ix || ix->reps.empty()) fail(AWRY_ERR_INVALID_ARG, "null or empty index handle");
  return ix;
}

// ---- batch.cu
bool is_pinned(const void* p);
void parallel_memcpy(void* dst, const void* src, size_t n);
uint64_t locate_chunk_count(Replica& r, Workspace* ws, uint64_t nq, uint64_t* d_hit_off, cudaStream_t st);
uint64_t* locate_chunk_walk(Replica& r, Workspace* ws, uint64_t nq, uint64_t n_hits, uint32_t flags,
                            const uint64_t* d_hit_off, cudaStream_t st);

}  // namespace host
}  // namespace awry
