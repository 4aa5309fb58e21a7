// kernels_align.cu -- the alignment of located Hamming and edit-distance hits (awry_align_*, include/awry_b200.h,
// DESIGN.md §1f).  One thread per hit: the packed search-order query against IndexView::rtext, with at most k <= 3
// operations, written as one awry_alignment.  Search order runs backwards through the query and rtext backwards
// through the text, so "forward from s" is a descending walk in both streams (desc8 / rtext8, kernels_common.cuh).
#include "../../include/awry_b200.h"
#include "kernels_common.cuh"

namespace awry {

static_assert(sizeof(awry_alignment) == 44 && sizeof(awry_edit_op) == 12, "11 u32 per alignment");

// search query lengths (kernels.hpp).  A '$' / '#' packs to code 5 (DNA_SENTINEL): a nibble >= 5 has bit 3, or bit 2
// with bit 0 or 1.
__global__ void __launch_bounds__(256)
    align_reads_kernel(const uint64_t* __restrict__ qwords, const uint64_t* __restrict__ qoff, uint64_t nq, ByteRange br,
                       uint64_t qw_lo, uint64_t qw_n, uint32_t k, uint32_t shift, uint32_t* __restrict__ qlen,
                       unsigned long long* first_bad) {
  const uint64_t stride = gridDim.x * uint64_t(blockDim.x);
  for (uint64_t q = blockIdx.x * uint64_t(blockDim.x) + threadIdx.x; q < nq; q += stride) {
    const uint64_t o0 = qoff[q];
    uint32_t len = checked_len(o0, qoff[q + 1], br);  // 0: refused by the prepass, or empty
    if (len != 0 && len <= k) {
      atomicMin(first_bad, bad_query_code(q >> shift, BAD_QUERY));
      len = 0;
    }
    if (len) {
      const uint64_t w0 = 4 * (q + (o0 >> 6));
      AWRY_CHK(w0 >= qw_lo && w0 - qw_lo + (len + 15) / 16 <= qw_n);
      uint64_t bad = 0;
      for (uint32_t i = 0; 16 * i < len; i++) {
        uint64_t x = __ldg(qwords + w0 + i);
        if (len - 16 * i < 16) x &= (1ull << (4 * (len - 16 * i))) - 1;
        bad |= ((x >> 2) & (x | (x >> 1))) | (x >> 3);
      }
      if (bad & 0x1111111111111111ull) len = 0;  // (latched by the prepass)
    }
    qlen[q] = len;
  }
}

cudaError_t launch_align_reads(const uint64_t* d_qwords, const uint64_t* d_qoff, uint64_t nq, uint64_t b_lo, uint64_t b_hi,
                               uint64_t qw_lo, uint64_t qw_n, uint32_t k, uint32_t shift, uint32_t* d_qlen,
                               unsigned long long* d_first_bad, cudaStream_t s) {
  if (nq == 0) return cudaSuccess;
  const unsigned grid = unsigned(std::min<uint64_t>((nq + 255) / 256, 148 * 16));
  align_reads_kernel<<<grid, 256, 0, s>>>(d_qwords, d_qoff, nq, ByteRange{b_lo, b_hi}, qw_lo, qw_n, k, shift, d_qlen,
                                          d_first_bad);
  COUNT_LAUNCH();
  return cudaGetLastError();
}

// symbol y of a packed search-order query, and reversed-text symbol x (0 <= x < bwt_len)
__device__ __forceinline__ uint32_t read_sym(const uint32_t* rq, uint32_t y) { return (__ldg(rq + (y >> 3)) >> (4 * (y & 7))) & 15u; }
__device__ __forceinline__ uint32_t rtext_sym(const IndexView& ix, int64_t x) {
  AWRY_CHK(x >= 0 && uint64_t(x >> 1) < ix.n_rtext);
  return (__ldg(ix.rtext + (x >> 1)) >> (4 * (x & 1))) & 15u;
}
// device symbol (A0 C1 G2 T3 N4) -> ASCII
__device__ __forceinline__ uint32_t sym_ascii(uint32_t c) { return c < 4 ? (0x54474341u >> (8 * c)) & 0xffu : uint32_t('N'); }

// ---- edit distance: iterative deepening.  State (i, j): Q[0 .. i) aligned against T[s .. s + j).  Q[i] is search-order
// symbol L - 1 - i, T[s + j] is rtext[r0 - j] with r0 = bwt_len - 1 - s; j < tleft = n - s while T[s + j] exists.
struct EditWalk {
  const uint32_t* rq;
  int64_t r0;
  uint32_t len, tleft;
};
// the path found: op o (in search depth order, 0 = first) sits in slot b - 1 - o of a search with budget b.  Scalar
// fields, not arrays: through the 40 inlined levels of edit_search an array stayed in local memory.
struct EditPath {
  uint64_t at0, at1, at2;  // slot u: qpos | tpos << 32
  uint32_t op0, op1, op2, end;
  template <int U>
  __device__ __forceinline__ void set(uint32_t qpos, uint32_t tpos, uint32_t op) {
    const uint64_t at = qpos | (uint64_t(tpos) << 32);
    if constexpr (U == 0) {
      at0 = at;
      op0 = op;
    } else if constexpr (U == 1) {
      at1 = at;
      op1 = op;
    } else {
      at2 = at;
      op2 = op;
    }
  }
  __device__ __forceinline__ uint64_t at(uint32_t u) const { return u == 0 ? at0 : u == 1 ? at1 : at2; }
  __device__ __forceinline__ uint32_t op(uint32_t u) const { return u == 0 ? op0 : u == 1 ? op1 : op2; }
};

// longest common extension: advance (i, j) over equal symbols, 8 per step, up to the first difference or the query's
// end.  The text beyond its end reads as '$' / 0xF, which no query symbol equals.
__device__ __forceinline__ void extend(const IndexView& ix, const EditWalk& w, uint32_t& i, uint32_t& j) {
  while (i < w.len) {
    const uint32_t rem = w.len - i;
    uint32_t x = desc8(w.rq, w.len - 1 - i) ^ rtext8(ix, w.r0 - int64_t(j) - 7);  // Q[i + t], T[s + j + t] in nibble 7 - t
    if (rem < 8) x &= ~0u << (4 * (8 - rem));
    const uint32_t m = x ? __clz(x) >> 2 : min(rem, 8u);
    i += m;
    j += m;
    if (x) return;
  }
}

// whether the rest of Q aligns from (i, j) within B more operations; a match is always taken (it never costs an
// optimal alignment anything), then X, I, D in that order, so the first success is the lexicographically smallest
template <int B>
__device__ __forceinline__ bool edit_search(const IndexView& ix, const EditWalk& w, uint32_t i, uint32_t j, EditPath& p) {
  extend(ix, w, i, j);
  if (i == w.len) {
    p.end = j;
    return true;
  }
  if constexpr (B == 0) {
    return false;
  } else {
    const bool text = j < w.tleft;  // X and D consume T[s + j]: not past the text's end
    uint32_t op = 0;
    if (text && edit_search<B - 1>(ix, w, i + 1, j + 1, p))
      op = 'X';
    else if (edit_search<B - 1>(ix, w, i + 1, j, p))
      op = 'I';
    else if (text && edit_search<B - 1>(ix, w, i, j + 1, p))
      op = 'D';
    if (op) p.set<B - 1>(i, j, op);
    return op != 0;
  }
}

// d(s): the smallest budget b <= K that succeeds (K + 1: none)
template <int B, int K>
__device__ __forceinline__ uint32_t edit_deepen(const IndexView& ix, const EditWalk& w, EditPath& p) {
  if (edit_search<B>(ix, w, 0, 0, p)) return B;
  if constexpr (B < K) {
    return edit_deepen<B + 1, K>(ix, w, p);
  } else {
    return K + 1;
  }
}

// One thread per hit.  out: text_len, distance | n_ops << 8, then per op qpos, tpos, op | query_sym << 8 | text_sym << 16.
template <int K, bool EDIT>
__global__ void __launch_bounds__(256, 4) align_hits_kernel(IndexView ix, AlignSlice a) {
  const uint64_t stride = gridDim.x * uint64_t(blockDim.x);
  const uint64_t n_text = uint64_t(ix.bwt_len) - 1;
  if (blockIdx.x == 0 && threadIdx.x == 0) AWRY_CHK(*a.hit_end == a.hit_total);
  for (uint64_t h = blockIdx.x * uint64_t(blockDim.x) + threadIdx.x; h < a.n; h += stride) {
    const uint32_t v = a.map[h];
    AWRY_CHK(v < a.nq);
    const uint64_t seq = a.hits[2 * h], local = a.hits[2 * h + 1];
    const uint32_t len = a.qlen[v];
    uint32_t o[11] = {0, K + 1, 0, 0, 0, 0, 0, 0, 0, 0, 0};
    uint64_t s = n_text;
    if (len && seq < ix.n_seqs) {
      const uint64_t st = __ldg(ix.seq_starts + seq);
      s = st + local < st ? n_text : st + local;
    }
    if (s < n_text) {
      const uint64_t w0 = 4 * (v + (a.qoff[v] >> 6));
      AWRY_CHK(w0 >= a.qw_lo && w0 - a.qw_lo + (len + 7) / 8 / 2 + 8 < a.qw_n);
      const uint32_t* const rq = reinterpret_cast<const uint32_t*>(a.qwords + w0);
      const int64_t r0 = int64_t(ix.bwt_len) - 1 - int64_t(s);  // rtext index of T[s]
      uint32_t d = K + 1, qpos[AWRY_EDIT_MAX] = {}, tpos[AWRY_EDIT_MAX] = {}, op[AWRY_EDIT_MAX] = {}, tlen = 0;
      if (!EDIT) {
        if (s + len <= n_text) {
          // search-order symbol y of Q against rtext[r0 - len + 1 + y]; mismatch c (ascending y) is op d - 1 - c
          const int64_t rb = r0 - int64_t(len) + 1;
          uint32_t c = 0, at[AWRY_EDIT_MAX] = {};
          for (uint32_t y = 0; y < len && c <= uint32_t(K); y += 8) {
            uint32_t x = read8(rq, y) ^ rtext8(ix, rb + y);
            if (len - y < 8) x &= (1u << (4 * (len - y))) - 1u;
            uint32_t m = (x | (x >> 1) | (x >> 2) | (x >> 3)) & 0x11111111u;
            for (; m && c <= uint32_t(K); m &= m - 1, c++) {
#pragma unroll
              for (int t = 0; t < K; t++)
                if (c == uint32_t(t)) at[t] = y + ((__ffs(m) - 1) >> 2);
            }
          }
          if (c <= uint32_t(K)) {
            d = c;
            tlen = len;
#pragma unroll
            for (int t = 0; t < K; t++) {
#pragma unroll
              for (int u = 0; u < K; u++)
                if (uint32_t(t) < c && uint32_t(u) == c - 1 - t) {
                  qpos[t] = len - 1 - at[u];
                  tpos[t] = qpos[t];
                  op[t] = 'X';
                }
            }
          }
        }
      } else {
        const EditWalk w{rq, r0, len, uint32_t(n_text - s)};
        EditPath p{};
        d = edit_deepen<0, K>(ix, w, p);
        if (d <= uint32_t(K)) {
          tlen = p.end;
#pragma unroll
          for (int t = 0; t < K; t++) {
            if (uint32_t(t) < d) {
              const uint64_t at = p.at(d - 1 - t);
              qpos[t] = uint32_t(at);
              tpos[t] = uint32_t(at >> 32);
              op[t] = p.op(d - 1 - t);
            }
          }
        }
      }
      if (d <= uint32_t(K)) {
        o[0] = tlen;
        o[1] = d | (d << 8);
#pragma unroll
        for (int t = 0; t < K; t++) {
          if (uint32_t(t) < d) {
            const uint32_t qs = op[t] == 'D' ? 0u : sym_ascii(read_sym(rq, len - 1 - qpos[t]));
            const uint32_t ts = op[t] == 'I' ? 0u : sym_ascii(rtext_sym(ix, r0 - int64_t(tpos[t])));
            o[2 + 3 * t] = qpos[t];
            o[3 + 3 * t] = tpos[t];
            o[4 + 3 * t] = op[t] | (qs << 8) | (ts << 16);
          }
        }
      }
    }
    uint32_t* const dst = a.out + 11 * h;
#pragma unroll
    for (int t = 0; t < 11; t++) dst[t] = o[t];
  }
}

template <int K>
static void launch_align_k(const IndexView& ix, const AlignSlice& a, bool edit, unsigned grid, cudaStream_t s) {
  if (edit)
    align_hits_kernel<K, true><<<grid, 256, 0, s>>>(ix, a);
  else
    align_hits_kernel<K, false><<<grid, 256, 0, s>>>(ix, a);
}

cudaError_t launch_align_hits(const IndexView& ix, const AlignSlice& a, uint32_t k, bool edit, int sm_count, cudaStream_t s) {
  if (a.n == 0) return cudaSuccess;
  if (k > 3 || ix.rtext == nullptr) return cudaErrorInvalidValue;
  const unsigned grid = unsigned(std::max<uint64_t>(1, std::min<uint64_t>(uint64_t(sm_count) * 8, (a.n + 255) / 256)));
  switch (k) {
    case 0: launch_align_k<0>(ix, a, edit, grid, s); break;
    case 1: launch_align_k<1>(ix, a, edit, grid, s); break;
    case 2: launch_align_k<2>(ix, a, edit, grid, s); break;
    default: launch_align_k<3>(ix, a, edit, grid, s); break;
  }
  COUNT_LAUNCH();
  return cudaGetLastError();
}

}  // namespace awry
