// kernels.cu -- hand-written sm_100a kernels of the batched FM-index search path.
//
// Reference functions replaced (paths under /root/reference/src):
//   pack_kernel           Symbol::new_ascii / index()            alphabet.rs:109-114, :169-248
//   build_table_kernel    KmerLookupTable (a CORRECT seed table)  kmer_lookup_table.rs:17-20, :121-167
//   search kernels        get_search_range_for_string + update_range_with_symbol + count_string
//                                                                 fm_index.rs:402-438, :499-501, :559-582
//   walk_kernel           locate_string + backstep + reconstruct_value + get_seq_location
//                                                                 fm_index.rs:516-544, :585-593,
//                                                                 compressed_suffix_array.rs:76-111,
//                                                                 sequence_index.rs:108-141
//   transpose kernels     load-time re-layout of bwt.rs:12-25 blocks (fm_index_file.rs:215-262)
#include <atomic>
#include <cstdio>
#include <cub/device/device_scan.cuh>
#include <cub/device/device_segmented_sort.cuh>
#include <thrust/iterator/counting_iterator.h>
#include <thrust/iterator/transform_iterator.h>

#include "kernels_common.cuh"

namespace awry {

std::atomic<uint64_t> g_launches{0};
uint64_t kernel_launch_count() { return g_launches.load(); }
void kernel_launch_count_reset() { g_launches.store(0); }

// ------------------------------------------------------------------ symbol tables

__constant__ uint8_t c_ascii_to_dsym[2][256];  // ASCII -> device symbol (alphabet.rs:169-248)
__constant__ uint8_t c_amino_code_to_idx[32];  // reference 5-bit code -> index (alphabet.rs:197-222)

static uint8_t host_ascii_to_ref_index(int alphabet, uint8_t ch) {
  if (ch >= 'a' && ch <= 'z') ch = uint8_t(ch - 'a' + 'A');
  if (ch == '$' || ch == '#') return 0;
  if (alphabet == 0) {
    switch (ch) {
      case 'A': return 1;
      case 'C': return 2;
      case 'G': return 3;
      case 'T':
      case 'U': return 5;
      default: return 4;
    }
  }
  static const char L[23] = "$ACDEFGHIKLMNPQRSTVWXY";
  for (int i = 1; i < 22; i++)
    if (i != 20 && L[i] == char(ch)) return uint8_t(i);
  return 20;
}

cudaError_t init_device_tables() {
  uint8_t lut[2][256];
  static const uint8_t dna_ref_to_dsym[6] = {DNA_SENTINEL, 0, 1, 2, DNA_N, 3};
  for (int c = 0; c < 256; c++) {
    lut[0][c] = dna_ref_to_dsym[host_ascii_to_ref_index(0, uint8_t(c))];
    lut[1][c] = host_ascii_to_ref_index(1, uint8_t(c));
  }
  cudaError_t e = cudaMemcpyToSymbol(c_ascii_to_dsym, lut, sizeof lut);
  if (e != cudaSuccess) return e;
  static const uint8_t codes[22] = {0x00, 0x0c, 0x17, 0x03, 0x06, 0x1e, 0x1a, 0x1b, 0x19, 0x15, 0x1c,
                                    0x1d, 0x08, 0x09, 0x04, 0x13, 0x0a, 0x05, 0x16, 0x01, 0x1f, 0x02};
  uint8_t c2i[32];
  for (int c = 0; c < 32; c++) c2i[c] = 20;  // unknown codes decode to X
  for (int i = 0; i < 22; i++) c2i[codes[i]] = uint8_t(i);
  return cudaMemcpyToSymbol(c_amino_code_to_idx, c2i, sizeof c2i);
}

// ------------------------------------------------------------------ load-time re-layout

// one thread per 16-B output chunk; 8 chunks per 256-row reference block (bwt.rs:12-17)
__global__ void transpose_dna_kernel(const uint64_t* __restrict__ ref, uint64_t first_rb,
                                     uint64_t n_rb, uint64_t bwt_len, uint4* __restrict__ out,
                                     unsigned long long* dollar_row, const uint64_t* __restrict__ sb, uint32_t sb_shift) {
  uint64_t t = blockIdx.x * uint64_t(blockDim.x) + threadIdx.x;
  if (t >= n_rb * 8) return;
  uint64_t lrb = t >> 3;
  uint32_t h = uint32_t(t >> 2) & 1, j = uint32_t(t) & 3;
  const uint64_t* rb = ref + lrb * 20;
  uint32_t w = 2 * h + (j >> 1), sh = 32 * (j & 1);
  uint32_t r0 = uint32_t(rb[w] >> sh), r1 = uint32_t(rb[4 + w] >> sh), r2 = uint32_t(rb[8 + w] >> sh);
  uint64_t row0 = (first_rb + lrb) * 256 + 128 * h + 32 * j;
  uint32_t valid = row0 >= bwt_len ? 0u : (bwt_len - row0 >= 32 ? ~0u : ((1u << (bwt_len - row0)) - 1u));
  // reference codes (alphabet.rs:237-244): $100 A110 C101 G011 T001, everything else decodes to N
  uint32_t isS = ~r0 & ~r1 & r2, isA = ~r0 & r1 & r2, isC = r0 & ~r1 & r2, isG = r0 & r1 & ~r2,
           isT = r0 & ~r1 & ~r2;
  uint32_t isN = ~(isS | isA | isC | isG | isT);
  uint32_t d0 = ((isC | isT | isS) & valid) | ~valid;  // device codes A0 C1 G2 T3 N4 $5, pad 7
  uint32_t d1 = ((isG | isT) & valid) | ~valid;
  uint32_t d2 = ((isN | isS) & valid) | ~valid;
  if (isS & valid) *dollar_row = row0 + uint64_t(__ffs(isS & valid) - 1);
  // milestone of symbol j (A,C,G,T = reference index 1,2,3,5) at the start of this 128-row block
  const int ref_idx = j == 3 ? 5 : int(j) + 1;
  uint64_t cnt = rb[12 + ref_idx];
  if (h == 1) {
#pragma unroll
    for (int ww = 0; ww < 2; ww++) {
      uint64_t a = rb[ww], b = rb[4 + ww], c = rb[8 + ww];
      uint64_t m = j == 0 ? (~a & b & c) : j == 1 ? (a & ~b & c) : j == 2 ? (a & b & ~c) : (a & ~b & ~c);
      cnt += uint64_t(__popcll(m));
    }
  }
  if (sb != nullptr) cnt -= sb[(row0 >> sb_shift) * SB_STRIDE + j];  // wide index: relative to the superblock
  out[(first_rb + lrb) * 8 + h * 4 + j] = make_uint4(d0, d1, d2, uint32_t(cnt));
}

// Amino re-layout, step 1: one thread per 32-row slice (8 per 256-row reference block, bwt.rs:19-25)
// re-encodes the 5 reference planes into planes of the symbol INDEX and writes them into slice 0/1
// of the 64-row device block that owns the rows.
__global__ void transpose_amino_kernel(const uint64_t* __restrict__ ref, uint64_t first_rb,
                                       uint64_t n_rb, uint64_t bwt_len, uint4* __restrict__ out,
                                       unsigned long long* dollar_row) {
  uint64_t t = blockIdx.x * uint64_t(blockDim.x) + threadIdx.x;
  if (t >= n_rb * 8) return;
  uint64_t lrb = t >> 3;
  uint32_t j = uint32_t(t) & 7;  // 32-row slice of the reference block
  const uint64_t* rb = ref + lrb * 44;
  uint32_t w = j >> 1, sh = 32 * (j & 1);
  uint32_t r[5], d[5] = {0, 0, 0, 0, 0};
#pragma unroll
  for (int p = 0; p < 5; p++) r[p] = uint32_t(rb[4 * p + w] >> sh);
  uint64_t row0 = (first_rb + lrb) * 256 + 32 * j;
  uint32_t valid = row0 >= bwt_len ? 0u : (bwt_len - row0 >= 32 ? ~0u : ((1u << (bwt_len - row0)) - 1u));
  for (int bit = 0; bit < 32; bit++) {
    uint32_t code = 0;
#pragma unroll
    for (int p = 0; p < 5; p++) code |= ((r[p] >> bit) & 1u) << p;
    uint32_t idx = ((valid >> bit) & 1u) ? c_amino_code_to_idx[code] : 0u;
    if (((valid >> bit) & 1u) && code == 0) *dollar_row = row0 + uint64_t(bit);
#pragma unroll
    for (int p = 0; p < 5; p++) d[p] |= ((idx >> p) & 1u) << bit;
  }
  // device block = 64 rows: reference block x 4 + j/2; slice j%2; plane words 0..4 of the slice
  uint32_t* o = reinterpret_cast<uint32_t*>(out + ((first_rb + lrb) * 4 + (j >> 1)) * AMINO_BLOCK_UINT4) + 8 * (j & 1);
#pragma unroll
  for (int p = 0; p < 5; p++) o[p] = d[p];
}

// Amino re-layout, step 2: one thread per (reference block, symbol): block-start counts of the four
// 64-row device blocks = the reference milestone + symbols seen in the earlier device blocks,
// counted on the re-encoded planes so counts and planes agree for every input.
__global__ void amino_counts_kernel(const uint64_t* __restrict__ ref, uint64_t first_rb, uint64_t n_rb,
                                    uint4* __restrict__ out, const uint64_t* __restrict__ sb, uint32_t sb_shift) {
  uint64_t t = blockIdx.x * uint64_t(blockDim.x) + threadIdx.x;
  if (t >= n_rb * 32) return;
  uint64_t lrb = t >> 5;
  uint32_t s = uint32_t(t) & 31;
  if (s == 0 || s > 21) return;
  uint64_t ms = ref[lrb * 44 + 20 + s];
  if (sb != nullptr) ms -= sb[(((first_rb + lrb) * 256) >> sb_shift) * SB_STRIDE + s];  // wide index: relative
  uint32_t cnt = uint32_t(ms);
  for (uint32_t d = 0; d < 4; d++) {
    uint32_t* blk = reinterpret_cast<uint32_t*>(out + ((first_rb + lrb) * 4 + d) * AMINO_BLOCK_UINT4);
    blk[amino_count_word(s)] = cnt;
#pragma unroll
    for (int sl = 0; sl < 2; sl++) {
      uint32_t m = ~0u;
#pragma unroll
      for (int p = 0; p < 5; p++) m &= ((s >> p) & 1u) ? blk[8 * sl + p] : ~blk[8 * sl + p];
      cnt += __popc(m);
    }
  }
}

cudaError_t launch_transpose(int alphabet, const uint64_t* d_ref_blocks, uint64_t first_ref_block,
                             uint64_t n_ref_blocks, uint64_t bwt_len, uint4* d_blocks,
                             unsigned long long* d_dollar_row, const uint64_t* d_sb, uint32_t sb_shift, cudaStream_t s) {
  if (n_ref_blocks == 0) return cudaSuccess;
  uint64_t threads = n_ref_blocks * 8;
  unsigned grid = unsigned((threads + 255) / 256);
  if (alphabet == 0)
    transpose_dna_kernel<<<grid, 256, 0, s>>>(d_ref_blocks, first_ref_block, n_ref_blocks, bwt_len,
                                              d_blocks, d_dollar_row, d_sb, sb_shift);
  else {
    transpose_amino_kernel<<<grid, 256, 0, s>>>(d_ref_blocks, first_ref_block, n_ref_blocks,
                                                bwt_len, d_blocks, d_dollar_row);
    COUNT_LAUNCH();
    uint64_t t2 = n_ref_blocks * 32;
    amino_counts_kernel<<<unsigned((t2 + 255) / 256), 256, 0, s>>>(d_ref_blocks, first_ref_block,
                                                                    n_ref_blocks, d_blocks, d_sb, sb_shift);
  }
  COUNT_LAUNCH();
  return cudaGetLastError();
}

// one thread per superblock that starts inside [first_rb, first_rb + n_rb): its absolute counts are the
// milestones of its first reference block (fm_index.rs:212-217), reordered to SB_STRIDE slots
__global__ void gather_superblocks_kernel(int alphabet, const uint64_t* __restrict__ ref, uint64_t first_rb, uint64_t n_rb,
                                          uint32_t sb_shift, uint64_t* __restrict__ sb) {
  const uint64_t rb_per_sb = 1ull << (sb_shift - 8);
  const uint64_t s0 = (first_rb + rb_per_sb - 1) / rb_per_sb;
  const uint64_t sidx = s0 + blockIdx.x * uint64_t(blockDim.x) + threadIdx.x;
  const uint64_t rb = sidx * rb_per_sb;
  if (rb >= first_rb + n_rb) return;
  const uint64_t* ms = ref + (rb - first_rb) * (alphabet == 0 ? 20 : 44) + (alphabet == 0 ? 12 : 20);
  uint64_t* o = sb + sidx * SB_STRIDE;
  if (alphabet == 0) {
    o[0] = ms[1];
    o[1] = ms[2];
    o[2] = ms[3];
    o[3] = ms[5];
  } else {
    for (int i = 0; i < 22; i++) o[i] = ms[i];
  }
}
cudaError_t launch_gather_superblocks(int alphabet, const uint64_t* d_ref_blocks, uint64_t first_ref_block,
                                      uint64_t n_ref_blocks, uint32_t sb_shift, uint64_t* d_sb, cudaStream_t s) {
  if (n_ref_blocks == 0) return cudaSuccess;
  const uint64_t rb_per_sb = 1ull << (sb_shift - 8);
  const uint64_t n = n_ref_blocks / rb_per_sb + 2;
  gather_superblocks_kernel<<<unsigned((n + 127) / 128), 128, 0, s>>>(alphabet, d_ref_blocks, first_ref_block, n_ref_blocks,
                                                                      sb_shift, d_sb);
  COUNT_LAUNCH();
  return cudaGetLastError();
}

// ------------------------------------------------------------------ FmIndex::save: device layout -> bwt.rs blocks

// Inverse of transpose_dna_kernel: one thread per 64-bit plane word (4 per 256-row reference block,
// bwt.rs:12-17).  Rows 64w..64w+63 of reference block rb are chunks 2(w&1), 2(w&1)+1 of device block
// 2rb + (w>>1).  Device codes A0 C1 G2 T3 N4 $5 (padding 7) -> reference codes $100 A110 C101 G011 N010
// T001 (alphabet.rs:309-327); padding rows come out as all-zero planes, as set_symbol_at never touched them.
// The thread of word 0 also writes the 8 milestones (bwt.rs:29; fm_index.rs:212-217), N derived as in layout.cuh.
__global__ void untranspose_dna_kernel(const uint4* __restrict__ blocks, uint64_t first_rb, uint64_t n_rb,
                                       uint64_t dollar_row, uint64_t* __restrict__ ref, const uint64_t* __restrict__ sb,
                                       uint32_t sb_shift) {
  uint64_t t = blockIdx.x * uint64_t(blockDim.x) + threadIdx.x;
  if (t >= n_rb * 4) return;
  const uint64_t lrb = t >> 2, rb = first_rb + lrb;
  const uint32_t w = uint32_t(t) & 3;
  const uint4* db = blocks + (rb * 2 + (w >> 1)) * DNA_BLOCK_UINT4;
  uint64_t r0 = 0, r1 = 0, r2 = 0;
#pragma unroll
  for (int half = 0; half < 2; half++) {
    const uint4 ch = db[2 * (w & 1) + half];
    const uint32_t d0 = ch.x, d1 = ch.y, d2 = ch.z;
    const uint32_t isA = ~d0 & ~d1 & ~d2, isC = d0 & ~d1 & ~d2, isG = ~d0 & d1 & ~d2, isT = d0 & d1 & ~d2,
                   isN = ~d0 & ~d1 & d2, isS = d0 & ~d1 & d2;
    r0 |= uint64_t(isC | isG | isT) << (32 * half);
    r1 |= uint64_t(isA | isG | isN) << (32 * half);
    r2 |= uint64_t(isS | isA | isC) << (32 * half);
  }
  uint64_t* out = ref + lrb * 20;
  out[w] = r0;
  out[4 + w] = r1;
  out[8 + w] = r2;
  if (w == 0) {
    const uint4* b0 = blocks + rb * 2 * DNA_BLOCK_UINT4;
    const uint64_t start = rb * 256;
    uint64_t a = b0[0].w, c = b0[1].w, g = b0[2].w, tt = b0[3].w;
    if (sb != nullptr) {  // wide index: block counts are relative to the superblock
      const uint64_t* o = sb + (start >> sb_shift) * SB_STRIDE;
      a += o[0];
      c += o[1];
      g += o[2];
      tt += o[3];
    }
    const uint64_t s = dollar_row < start ? 1 : 0;
    out[12] = s;
    out[13] = a;
    out[14] = c;
    out[15] = g;
    out[16] = start - (a + c + g + tt) - s;
    out[17] = tt;
    out[18] = 0;
    out[19] = 0;
  }
}

// Inverse of transpose_amino_kernel + amino_counts_kernel: one thread per 32-row slice (8 per reference
// block, bwt.rs:19-25) turns the planes of the symbol INDEX back into planes of the reference's 5-bit codes
// (alphabet.rs:255-303; '$' and padding rows are code 00000); slice 0 also writes the 24 milestones.
__constant__ uint8_t c_amino_idx_to_code[32];
__global__ void untranspose_amino_kernel(const uint4* __restrict__ blocks, uint64_t first_rb, uint64_t n_rb,
                                         uint64_t dollar_row, uint64_t* __restrict__ ref, const uint64_t* __restrict__ sb,
                                         uint32_t sb_shift) {
  uint64_t t = blockIdx.x * uint64_t(blockDim.x) + threadIdx.x;
  if (t >= n_rb * 8) return;
  const uint64_t lrb = t >> 3, rb = first_rb + lrb;
  const uint32_t j = uint32_t(t) & 7;
  const uint32_t* d =
      reinterpret_cast<const uint32_t*>(blocks + (rb * 4 + (j >> 1)) * AMINO_BLOCK_UINT4) + 8 * (j & 1);
  uint32_t dp[5], r[5] = {0, 0, 0, 0, 0};
#pragma unroll
  for (int p = 0; p < 5; p++) dp[p] = d[p];
  for (int bit = 0; bit < 32; bit++) {
    uint32_t idx = 0;
#pragma unroll
    for (int p = 0; p < 5; p++) idx |= ((dp[p] >> bit) & 1u) << p;
    const uint32_t code = c_amino_idx_to_code[idx];
#pragma unroll
    for (int p = 0; p < 5; p++) r[p] |= ((code >> p) & 1u) << bit;
  }
  uint32_t* out32 = reinterpret_cast<uint32_t*>(ref + lrb * 44);
#pragma unroll
  for (int p = 0; p < 5; p++) out32[(4 * p + (j >> 1)) * 2 + (j & 1)] = r[p];  // little-endian halves of the u64 words
  if (j == 0) {
    uint64_t* ms = ref + lrb * 44 + 20;
    const uint32_t* b0 = reinterpret_cast<const uint32_t*>(blocks + rb * 4 * AMINO_BLOCK_UINT4);
    ms[0] = dollar_row < rb * 256 ? 1 : 0;
    const uint64_t* o = sb != nullptr ? sb + ((rb * 256) >> sb_shift) * SB_STRIDE : nullptr;
    for (uint32_t s = 1; s <= 21; s++) ms[s] = uint64_t(b0[amino_count_word(s)]) + (o ? o[s] : 0ull);
    ms[22] = 0;
    ms[23] = 0;
  }
}

cudaError_t launch_untranspose(int alphabet, const uint4* d_blocks, uint64_t dollar_row, uint64_t first_ref_block,
                               uint64_t n_ref_blocks, uint64_t* d_ref_blocks, const uint64_t* d_sb, uint32_t sb_shift,
                               cudaStream_t s) {
  if (n_ref_blocks == 0) return cudaSuccess;
  if (alphabet == 0) {
    uint64_t threads = n_ref_blocks * 4;
    untranspose_dna_kernel<<<unsigned((threads + 255) / 256), 256, 0, s>>>(d_blocks, first_ref_block, n_ref_blocks,
                                                                            dollar_row, d_ref_blocks, d_sb, sb_shift);
  } else {
    // same table as init_device_tables (index -> 5-bit code); indices 22..31 never occur in device blocks
    static const uint8_t i2c[32] = {0x00, 0x0c, 0x17, 0x03, 0x06, 0x1e, 0x1a, 0x1b, 0x19, 0x15, 0x1c,
                                    0x1d, 0x08, 0x09, 0x04, 0x13, 0x0a, 0x05, 0x16, 0x01, 0x1f, 0x02};
    cudaError_t e = cudaMemcpyToSymbolAsync(c_amino_idx_to_code, i2c, sizeof i2c, 0, cudaMemcpyHostToDevice, s);
    if (e != cudaSuccess) return e;
    uint64_t threads = n_ref_blocks * 8;
    untranspose_amino_kernel<<<unsigned((threads + 255) / 256), 256, 0, s>>>(d_blocks, first_ref_block, n_ref_blocks,
                                                                              dollar_row, d_ref_blocks, d_sb, sb_shift);
  }
  COUNT_LAUNCH();
  return cudaGetLastError();
}

// ------------------------------------------------------------------ k-mer seed table

uint64_t table_entries(int alphabet, uint32_t k) {
  uint64_t b = alphabet == 0 ? 4 : 20, r = 1;
  for (uint32_t i = 0; i < k; i++) r *= b;
  return r;
}

__device__ __forceinline__ uint32_t amino_digit_to_sym(uint32_t d) { return d < 19 ? d + 1 : 21; }

// entry idx = sum_j digit_j * B^j, digit_0 = LAST query character (search order).
// One thread per k-mer: k-1 LF steps with early exit; absent k-mers get SearchRange::zero().
template <int ALPHA>
__global__ void build_table_kernel(IndexView ix, uint2* __restrict__ table, uint64_t n, uint32_t k) {
  constexpr uint32_t B = ALPHA == 0 ? 4 : 20;
  uint64_t idx = blockIdx.x * uint64_t(blockDim.x) + threadIdx.x;
  if (idx >= n) return;
  uint64_t rest = idx;
  uint32_t d = uint32_t(rest % B);
  rest /= B;
  uint32_t c = ALPHA == 0 ? d : amino_digit_to_sym(d);
  uint32_t sp = ix.c_lo[c], ep = ix.c_hi[c];
  for (uint32_t j = 1; j < k && sp <= ep; j++) {
    d = uint32_t(rest % B);
    rest /= B;
    lf_update<ALPHA>(ix, sp, ep, ALPHA == 0 ? d : amino_digit_to_sym(d));
  }
  table[idx] = sp <= ep ? make_uint2(sp, ep) : make_uint2(1u, 0u);
}

// Nucleotide tables deeper than 4^10 entries are built level by level: the entry of a j-mer is ONE LF step on the
// entry of its first j - 1 symbols (the low digits of its index), so level j costs 4^j steps instead of j * 4^j
// (k = 15: 1.4 G steps instead of 16 G; the two scratch levels take 4^(k-1) + 4^(k-2) entries).
__global__ void __launch_bounds__(256)
    extend_table_kernel(IndexView ix, const uint2* __restrict__ prev, uint2* __restrict__ next, uint64_t n_next, uint32_t j) {
  const uint64_t idx = blockIdx.x * uint64_t(blockDim.x) + threadIdx.x;
  if (idx >= n_next) return;
  const uint64_t n_prev = n_next >> 2;
  const uint2 r = prev[idx & (n_prev - 1)];
  uint32_t sp = r.x, ep = r.y;
  if (sp <= ep) lf_update<0>(ix, sp, ep, uint32_t(idx >> (2 * (j - 1))));
  next[idx] = sp <= ep ? make_uint2(sp, ep) : make_uint2(1u, 0u);
}

cudaError_t launch_build_table(const IndexView& ix, uint2* d_table, uint32_t k, cudaStream_t s) {
  uint64_t n = table_entries(int(ix.alphabet), k);
  constexpr uint32_t K0 = 10;  // levels up to here: one thread per k-mer walks all of its steps
  if (ix.alphabet == 0 && k > K0) {
    uint2* scratch[2] = {nullptr, nullptr};
    cudaError_t e = cudaMalloc(reinterpret_cast<void**>(&scratch[0]), (n >> 2) * sizeof(uint2));
    if (e == cudaSuccess && k > K0 + 1) e = cudaMalloc(reinterpret_cast<void**>(&scratch[1]), (n >> 4) * sizeof(uint2));
    if (e == cudaSuccess) {
      // level j lands in scratch[(k - 1 - j) & 1], so level k - 1 is in scratch[0] (the large one) and k - 2 in scratch[1]
      uint2* cur = scratch[(k - 1 - K0) & 1];
      const uint64_t n0 = table_entries(0, K0);
      build_table_kernel<0><<<unsigned((n0 + 255) / 256), 256, 0, s>>>(ix, cur, n0, K0);
      COUNT_LAUNCH();
      for (uint32_t j = K0 + 1; j <= k && e == cudaSuccess; j++) {
        uint2* const dst = j == k ? d_table : scratch[(k - 1 - j) & 1];
        const uint64_t nj = table_entries(0, j);
        extend_table_kernel<<<unsigned((nj + 255) / 256), 256, 0, s>>>(ix, cur, dst, nj, j);
        COUNT_LAUNCH();
        e = cudaGetLastError();
        cur = dst;
      }
      if (e == cudaSuccess) e = cudaStreamSynchronize(s);
    }
    cudaFree(scratch[0]);
    cudaFree(scratch[1]);
    if (e == cudaSuccess) return e;
    cudaGetLastError();  // scratch did not fit (or a launch failed): the one-pass kernel below needs none
  }
  unsigned grid = unsigned((n + 255) / 256);
  if (ix.alphabet == 0)
    build_table_kernel<0><<<grid, 256, 0, s>>>(ix, d_table, n, k);
  else
    build_table_kernel<1><<<grid, 256, 0, s>>>(ix, d_table, n, k);
  COUNT_LAUNCH();
  return cudaGetLastError();
}

// The k-mer table exactly as the REFERENCE populates and saves it (kmer_lookup_table.rs:121-167):
// (card-2)^k entries of (start,end) u64; entry index = sum_j d_j * (card-2)^j with d_j the symbol
// INDEX of the j-th character from the end, only indices 1 .. card-3 are ever visited (so T / Y and
// every k-mer with a zero digit stay SearchRange::zero() = (1,0)), no early exit on empty ranges.
// Written into `.awry` files by awry_build_index_file so the reference can load them; the search
// path never reads it (kmer_lookup_table.rs:90-110).
template <int ALPHA>
__global__ void ref_table_kernel(IndexView ix, uint64_t first, uint64_t count, uint32_t k, ulonglong2* __restrict__ out) {
  constexpr uint32_t ENC = ALPHA == 0 ? 4 : 20;  // num_encoding_symbols() = cardinality - 2
  uint64_t t = blockIdx.x * uint64_t(blockDim.x) + threadIdx.x;
  if (t >= count) return;
  uint64_t rest = first + t;
  uint32_t d = uint32_t(rest % ENC);
  rest /= ENC;
  bool visited = d != 0;
  // device symbol of reference index d (nucleotide: 1,2,3 -> A,C,G = 0,1,2; amino: unchanged)
  uint32_t c = ALPHA == 0 ? d - 1 : d;
  uint32_t sp = 1, ep = 0;
  if (visited) {
    sp = ix.c_lo[c];
    ep = ix.c_hi[c];
  }
  for (uint32_t j = 1; j < k && visited; j++) {
    d = uint32_t(rest % ENC);
    rest /= ENC;
    if (d == 0) {
      visited = false;
      break;
    }
    lf_update<ALPHA>(ix, sp, ep, ALPHA == 0 ? d - 1 : d);
  }
  out[t] = visited ? make_ulonglong2(sp, ep) : make_ulonglong2(1, 0);
}

cudaError_t launch_ref_table(const IndexView& ix, uint64_t first, uint64_t count, uint32_t k, void* d_out,
                             cudaStream_t s) {
  if (count == 0) return cudaSuccess;
  if (ix.wide) return launch_ref_table_wide(*ix.wide, first, count, k, d_out, s);
  unsigned grid = unsigned((count + 255) / 256);
  if (ix.alphabet == 0)
    ref_table_kernel<0><<<grid, 256, 0, s>>>(ix, first, count, k, static_cast<ulonglong2*>(d_out));
  else
    ref_table_kernel<1><<<grid, 256, 0, s>>>(ix, first, count, k, static_cast<ulonglong2*>(d_out));
  COUNT_LAUNCH();
  return cudaGetLastError();
}

// ------------------------------------------------------------------ nucleotide pair index

uint64_t pair_block_count(uint64_t bwt_len) { return (bwt_len + PAIR_ROWS_PER_BLOCK - 1) / PAIR_ROWS_PER_BLOCK; }

// One CTA (3 warps) per 96-row pair block.  Row code = 4*BWT[row] + BWT[LF(row)], or "special".
__global__ void __launch_bounds__(96)
    pair_planes_kernel(IndexView ix, uint4* __restrict__ pair_blocks, uint32_t* __restrict__ hist /* [16][n] */,
                       uint64_t n_pblocks) {
  __shared__ uint32_t cnt[16];
  const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x < 16) cnt[threadIdx.x] = 0;
  __syncthreads();
  const uint64_t blk = blockIdx.x;
  const uint64_t row64 = blk * PAIR_ROWS_PER_BLOCK + threadIdx.x;
  uint32_t code = 16;  // special (also the padding rows past bwt_len)
  if (row64 < ix.bwt_len) {
    uint32_t row = uint32_t(row64);
    uint32_t b1 = row >> 7, l1 = row & 127;
    DnaBlockRegs blk1 = dna_load_block(ix, b1);
    uint32_t a = dna_code_at(blk1, l1);
    if (a < 4) {
      uint32_t j = ix.c_lo[a] + dna_occ_in_block(ix, blk1, b1, l1, a) - 1;  // LF(row)
      uint32_t lj = j & 127;
      AWRY_CHK(uint64_t(j >> 7) * DNA_BLOCK_UINT4 + 3 < ix.n_blocks_u4);
      uint4 ch = ldg128(ix.blocks + size_t(j >> 7) * DNA_BLOCK_UINT4 + (lj >> 5));
      uint32_t t = lj & 31;
      uint32_t b = ((ch.x >> t) & 1u) | (((ch.y >> t) & 1u) << 1) | (((ch.z >> t) & 1u) << 2);
      if (b < 4) code = 4 * a + b;
    }
  }
  uint32_t* words = reinterpret_cast<uint32_t*>(pair_blocks + blk * PAIR_BLOCK_UINT4);
#pragma unroll
  for (int p = 0; p < 5; p++) {
    uint32_t w = __ballot_sync(0xffffffffu, (code >> p) & 1u);
    if (lane == 0) words[8 * warp + p] = w;
  }
  for (uint32_t p = 0; p < 16; p++) {
    uint32_t m = __ballot_sync(0xffffffffu, code == p);
    if (lane == 0 && m) atomicAdd(&cnt[p], uint32_t(__popc(m)));
  }
  __syncthreads();
  if (threadIdx.x < 16) hist[uint64_t(threadIdx.x) * n_pblocks + blk] = cnt[threadIdx.x];
}

// slot of pair count p inside a pair block, as a 32-bit word index
__host__ __device__ __forceinline__ uint32_t pair_count_word(uint32_t p) {
  return p < 9 ? 8 * (p / 3) + 5 + (p % 3) : 24 + (p - 9);
}

__global__ void pair_counts_kernel(const uint32_t* __restrict__ ms /* [16][n] exclusive sums */,
                                   uint64_t n_pblocks, uint4* __restrict__ pair_blocks) {
  uint64_t t = blockIdx.x * uint64_t(blockDim.x) + threadIdx.x;
  if (t >= n_pblocks * 16) return;
  uint64_t blk = t >> 4;
  uint32_t p = uint32_t(t) & 15;
  uint32_t* words = reinterpret_cast<uint32_t*>(pair_blocks + blk * PAIR_BLOCK_UINT4);
  words[pair_count_word(p)] = ms[uint64_t(p) * n_pblocks + blk];
  if (p == 15) words[31] = 0;
}

// C2[4a+b] = C[b] + Occ(b, C[a]-1)
__global__ void pair_c2_kernel(IndexView ix, uint32_t* __restrict__ out) {
  uint32_t p = threadIdx.x;
  if (p >= 16) return;
  uint32_t a = p >> 2, b = p & 3;
  uint32_t pos = ix.c_lo[a] - 1;  // C[a] >= 1: row 0 is the '$'-suffix
  DnaBlockRegs blk = dna_load_block(ix, pos >> 7);
  out[p] = ix.c_lo[b] + dna_occ_in_block(ix, blk, pos >> 7, pos & 127, b);
}

cudaError_t build_pair_index(const IndexView& ix, uint4* d_pair_blocks, uint32_t* c2_host, cudaStream_t s) {
  const uint64_t n = pair_block_count(ix.bwt_len);
  uint32_t* d_hist = nullptr;
  cudaError_t e = cudaMalloc(&d_hist, n * 16 * sizeof(uint32_t) + 64);
  if (e != cudaSuccess) return e;
  void* d_temp = nullptr;
  auto cleanup = [&](cudaError_t r) {
    cudaFree(d_hist);
    cudaFree(d_temp);
    return r;
  };
  pair_planes_kernel<<<unsigned(n), 96, 0, s>>>(ix, d_pair_blocks, d_hist, n);
  COUNT_LAUNCH();
  if ((e = cudaGetLastError()) != cudaSuccess) return cleanup(e);
  size_t tb = 0;
  if ((e = cub::DeviceScan::ExclusiveSum(nullptr, tb, d_hist, d_hist, (long long)n, s)) != cudaSuccess) return cleanup(e);
  if ((e = cudaMalloc(&d_temp, tb + 16)) != cudaSuccess) return cleanup(e);
  for (int p = 0; p < 16; p++) {
    e = cub::DeviceScan::ExclusiveSum(d_temp, tb, d_hist + uint64_t(p) * n, d_hist + uint64_t(p) * n, (long long)n, s);
    COUNT_LAUNCH();
    if (e != cudaSuccess) return cleanup(e);
  }
  uint64_t threads = n * 16;
  pair_counts_kernel<<<unsigned((threads + 255) / 256), 256, 0, s>>>(d_hist, n, d_pair_blocks);
  COUNT_LAUNCH();
  if ((e = cudaGetLastError()) != cudaSuccess) return cleanup(e);
  uint32_t* d_c2 = reinterpret_cast<uint32_t*>(d_hist);  // reuse after the counts are written
  if ((e = cudaStreamSynchronize(s)) != cudaSuccess) return cleanup(e);
  pair_c2_kernel<<<1, 32, 0, s>>>(ix, d_c2);
  COUNT_LAUNCH();
  if ((e = cudaMemcpyAsync(c2_host, d_c2, 64, cudaMemcpyDeviceToHost, s)) != cudaSuccess) return cleanup(e);
  e = cudaStreamSynchronize(s);
  return cleanup(e);
}

// ------------------------------------------------------------------ query packing prepass

// PL lanes per query; lane t packs words t, t+PL, ...  Flags the first empty / sentinel query.
// The ASCII table is copied to shared memory first: per-lane indices differ, and divergent
// constant-bank reads would serialise.
// RC (nucleotide): the words of the query's reverse complement instead -- search-order symbol si is the complement
// of text byte si (codes below 4 XOR 3; N and the sentinel stay).
template <int ALPHA, bool RC = false>
__device__ __forceinline__ uint64_t pack_word_bytes(const uint8_t* __restrict__ src, uint32_t len, uint32_t first,
                                                    const uint8_t* lut, bool& bad) {
  constexpr int BITS = ALPHA == 0 ? 4 : 8;
  constexpr int SPW = 64 / BITS;
  constexpr uint32_t SENT = ALPHA == 0 ? DNA_SENTINEL : AMINO_SENTINEL;
  uint64_t word = 0;
#pragma unroll 4
  for (int t = 0; t < SPW; t++) {
    uint32_t si = first + t;
    if (si < len) {
      uint32_t d = lut[src[RC ? si : len - 1 - si]];
      bad |= d == SENT;
      if (RC && d < 4) d ^= 3u;
      word |= uint64_t(d) << (BITS * t);
    }
  }
  return word;
}

// 4 ASCII bases (the first in the low byte) -> their 4 codes as nibbles in the same order (the first base in the low
// nibble), SIMD-in-register: ((c & 0xDF) >> 1) & 3 maps A,C,T,G to 0,1,2,3 and x ^ (x >> 1) swaps the last two.
// `diff` gets a non-zero byte for every byte that is not one of ACGT/acgt (whose nibble is then meaningless).
__device__ __forceinline__ uint32_t ascii4_codes(uint32_t w4, uint32_t& diff) {
  const uint32_t up = w4 & 0xDFDFDFDFu;
  const uint32_t x4 = (up >> 1) & 0x03030303u;
  const uint32_t c4 = x4 ^ ((x4 >> 1) & 0x01010101u);
  const uint32_t sel = c4 | (c4 >> 4);
  const uint32_t nib = (sel & 0xffu) | ((sel >> 8) & 0xff00u);  // 4 nibbles = 4 codes
  diff = up ^ __byte_perm(0x54474341u, 0, nib);                 // "ACGT"[code] per byte
  return nib;
}
// ... in search order (the last base in the low nibble)
__device__ __forceinline__ uint32_t ascii4_to_nibbles(uint32_t w4, uint32_t& diff) {
  return ascii4_codes(__byte_perm(w4, 0, 0x0123), diff);
}

template <int ALPHA, int PL = 8>
__global__ void __launch_bounds__(256)
    pack_kernel(const uint8_t* __restrict__ qbytes, const uint64_t* __restrict__ qoff, uint64_t nq,
                uint64_t* __restrict__ qwords, uint64_t b_lo, uint64_t b_hi, unsigned long long* first_bad) {
  constexpr int SPW = ALPHA == 0 ? 16 : 8;
  constexpr int LOG_SPW = ALPHA == 0 ? 4 : 3;
  constexpr int UNIT_SHIFT = ALPHA == 0 ? 6 : 5;  // symbols per 4-word (32-B) unit
  __shared__ uint8_t lut[256];
  lut[threadIdx.x] = c_ascii_to_dsym[ALPHA][threadIdx.x];
  __syncthreads();
  constexpr int LOG_PL = PL == 8 ? 3 : PL == 4 ? 2 : 1;
  const uint32_t sub = threadIdx.x & (PL - 1);
  const uint64_t ngroups = (gridDim.x * uint64_t(blockDim.x)) >> LOG_PL;
  for (uint64_t q = (blockIdx.x * uint64_t(blockDim.x) + threadIdx.x) >> LOG_PL; q < nq; q += ngroups) {
    const uint64_t o0 = qoff[q], o1 = qoff[q + 1];
    // offsets are caller data: a query outside the batch's byte range [b_lo, b_hi] (non-monotone offsets) is
    // refused before any load or store -- both buffers are sized from that range
    if (o0 < b_lo || o1 > b_hi || o1 < o0 || o1 - o0 >= (1ull << 32)) {
      if (sub == 0) atomicMin(first_bad, bad_query_code(q, BAD_OFFSETS));
      continue;
    }
    if (o1 == o0) {  // empty query
      if (sub == 0) atomicMin(first_bad, bad_query_code(q, BAD_QUERY));
      continue;
    }
    const uint32_t len = uint32_t(o1 - o0);
    const uint32_t nwords = (len + SPW - 1) >> LOG_SPW;
    uint64_t* const dst = qwords + 4 * (q + (o0 >> UNIT_SHIFT));
    const uint8_t* const src = qbytes + o0;
    bool bad = false;
#pragma unroll 4
    for (uint32_t wi = sub; wi < nwords; wi += PL) {
      const uint32_t first = wi << LOG_SPW;  // search-order index of this word's first symbol
      uint64_t word;
      bool done = false;
      if (ALPHA == 0 && len >= 16) {
        // 16 ASCII bases -> 16 nibbles without per-byte loads: 4-5 aligned 32-bit loads, funnel
        // shift to the byte offset, then ascii4_to_nibbles.  The query's final, partial word reuses the
        // first 16 bytes of the query and shifts the surplus symbols out.  Any byte that is not
        // one of ACGT/acgt sends the word down the table path.
        const uint32_t have = len - first;               // symbols left from `first` on
        const uint32_t drop = have >= 16 ? 0 : 16 - have;  // surplus symbols of a partial word
        const uint8_t* p = src + (have >= 16 ? have - 16 : 0);
        const uint32_t sh = uint32_t(reinterpret_cast<uintptr_t>(p) & 3);
        const uint32_t* a = reinterpret_cast<const uint32_t*>(p - sh);
        uint32_t u[5];
#pragma unroll
        for (int j = 0; j < 4; j++) u[j] = __ldg(a + j);
        u[4] = sh ? __ldg(a + 4) : 0u;  // only when it still overlaps the 16 bytes
        uint32_t nibs[4];
        bool clean = true;
#pragma unroll
        for (int j = 0; j < 4; j++) {
          uint32_t diff;
          nibs[j] = ascii4_to_nibbles(__funnelshift_r(u[j], u[j + 1], 8 * sh), diff);  // bytes 4j .. 4j+3
          clean &= diff == 0;
        }
        if (clean) {
          word = (uint64_t(nibs[1] | (nibs[0] << 16)) << 32) | uint64_t(nibs[3] | (nibs[2] << 16));
          word >>= 4 * drop;
          done = true;
        }
      }
      if (!done) word = pack_word_bytes<ALPHA>(src, len, first, lut, bad);
      dst[wi] = word;
    }
    if (bad) atomicMin(first_bad, bad_query_code(q, BAD_QUERY));
  }
}

cudaError_t launch_pack(int alphabet, const uint8_t* d_qbytes, const uint64_t* d_qoff, uint64_t nq,
                        uint64_t* d_qwords, uint64_t b_lo, uint64_t b_hi, unsigned long long* d_first_bad,
                        cudaStream_t s) {
  if (nq == 0) return cudaSuccess;
  // lanes per query: 4 for reads (10 words per 150-bp read: 0.60 against 0.85 ms per 10 M reads with 8 lanes, of which
  // the second round keeps 2 busy), 2 for short queries
  const uint64_t avg_len = b_hi != ~0ull && b_hi > b_lo ? (b_hi - b_lo) / nq : 150;
  const int pl = alphabet != 0 ? 8 : avg_len >= 48 ? 4 : 2;
  uint64_t threads = nq * uint64_t(pl);
  unsigned grid = unsigned(std::min<uint64_t>((threads + 255) / 256, 148 * 64));
  if (alphabet == 0 && pl == 4)
    pack_kernel<0, 4><<<grid, 256, 0, s>>>(d_qbytes, d_qoff, nq, d_qwords, b_lo, b_hi, d_first_bad);
  else if (alphabet == 0)
    pack_kernel<0, 2><<<grid, 256, 0, s>>>(d_qbytes, d_qoff, nq, d_qwords, b_lo, b_hi, d_first_bad);
  else
    pack_kernel<1, 8><<<grid, 256, 0, s>>>(d_qbytes, d_qoff, nq, d_qwords, b_lo, b_hi, d_first_bad);
  COUNT_LAUNCH();
  return cudaGetLastError();
}

// ---- 2-bit host-packed nucleotide queries -> 4-bit search-order words ----
// The host sends crumb i = (ascii[i] >> 1) & 3 (A0 C1 T2 G3) for every query byte of the chunk, four per
// byte in text order (hostpack.cpp), a quarter of the PCIe bytes of the ASCII form.  8 lanes per query as
// in pack_kernel; a word takes the 16 crumbs it covers with two 32-bit loads and a funnel shift, reverses
// their order (search order = last character first), swaps codes 2 <-> 3 (device symbols are A0 C1 G2 T3)
// and spreads each crumb to a nibble.  Bytes that were not ACGT (N, IUPAC codes, '$') come separately as
// exceptions and are patched in afterwards.
__device__ __forceinline__ uint32_t spread8_crumbs(uint32_t v) {  // 8 crumbs (16 bits) -> 8 nibbles
  v &= 0xffffu;
  v = (v | (v << 8)) & 0x00ff00ffu;
  v = (v | (v << 4)) & 0x0f0f0f0fu;
  v = (v | (v << 2)) & 0x33333333u;
  return v;
}

__global__ void __launch_bounds__(256)
    pack2_kernel(const uint32_t* __restrict__ crumbs, uint64_t base, const uint64_t* __restrict__ qoff, uint64_t nq,
                 uint64_t* __restrict__ qwords, uint64_t b_lo, uint64_t b_hi, unsigned long long* first_bad) {
  const uint32_t sub = threadIdx.x & 7;
  const uint64_t ngroups = (gridDim.x * uint64_t(blockDim.x)) >> 3;
  for (uint64_t q = (blockIdx.x * uint64_t(blockDim.x) + threadIdx.x) >> 3; q < nq; q += ngroups) {
    const uint64_t o0 = qoff[q], o1 = qoff[q + 1];
    if (o0 < b_lo || o1 > b_hi || o1 < o0 || o1 - o0 >= (1ull << 32)) {  // see pack_kernel
      if (sub == 0) atomicMin(first_bad, bad_query_code(q, BAD_OFFSETS));
      continue;
    }
    if (o1 == o0) {
      if (sub == 0) atomicMin(first_bad, bad_query_code(q, BAD_QUERY));
      continue;
    }
    const uint32_t len = uint32_t(o1 - o0);
    const uint32_t nwords = (len + 15) >> 4;
    uint64_t* const dst = qwords + 4 * (q + (o0 >> 6));
    const uint64_t c0 = o0 - base;  // crumb index of the query's first character
    for (uint32_t wi = sub; wi < nwords; wi += 8) {
      const uint32_t hi = len - 16 * wi;            // text positions [lo, hi) feed this word
      const uint32_t lo = hi >= 16 ? hi - 16 : 0;
      const uint32_t cnt = hi - lo;
      const uint64_t bit = 2 * (c0 + lo);
      const uint32_t* a = crumbs + (bit >> 5);
      uint32_t x = __funnelshift_r(__ldg(a), __ldg(a + 1), uint32_t(bit & 31));  // crumb j = text position lo + j
      x <<= 2 * (16 - cnt);                         // (cnt >= 1) drop what belongs to the next query
      uint32_t r = __brev(x);                        // reverses crumb order and the two bits of each crumb
      r = ((r & 0x55555555u) << 1) | ((r >> 1) & 0x55555555u);
      r ^= (r >> 1) & 0x55555555u;                   // codes 2 <-> 3
      dst[wi] = uint64_t(spread8_crumbs(r)) | (uint64_t(spread8_crumbs(r >> 16)) << 32);
    }
  }
}

// exceptions: ((byte position - exc_base) << 8) | ASCII byte, for bytes outside ACGTacgt
__global__ void patch_exceptions_kernel(const uint64_t* __restrict__ exc, uint64_t n_exc, uint64_t exc_base,
                                        const uint64_t* __restrict__ qoff, uint64_t nq, uint64_t* __restrict__ qwords,
                                        uint64_t b_lo, uint64_t b_hi, unsigned long long* first_bad) {
  uint64_t i = blockIdx.x * uint64_t(blockDim.x) + threadIdx.x;
  if (i >= n_exc) return;
  const uint64_t pos = exc_base + (exc[i] >> 8);
  const uint32_t d = c_ascii_to_dsym[0][exc[i] & 0xff];
  uint64_t lo = 0, hi = nq;  // last q with qoff[q] <= pos
  while (hi - lo > 1) {
    uint64_t mid = (lo + hi) >> 1;
    if (qoff[mid] <= pos)
      lo = mid;
    else
      hi = mid;
  }
  const uint64_t q = lo, o0 = qoff[q], o1 = qoff[q + 1];
  if (pos < o0 || pos >= o1) return;  // not inside any query of this chunk
  if (o0 < b_lo || o1 > b_hi || o1 - o0 >= (1ull << 32)) return;  // refused by pack2_kernel: its words do not exist
  if (d == uint32_t(DNA_SENTINEL)) {
    atomicMin(first_bad, bad_query_code(q, BAD_QUERY));
    return;
  }
  const uint32_t si = uint32_t(o1 - 1 - pos);  // search-order index
  unsigned long long* w = reinterpret_cast<unsigned long long*>(qwords + 4 * (q + (o0 >> 6)) + (si >> 4));
  const uint32_t sh = 4 * (si & 15);
  atomicAnd(w, ~(0xfull << sh));
  atomicOr(w, uint64_t(d) << sh);
}

cudaError_t launch_pack2(const uint32_t* d_crumbs, uint64_t base, const uint64_t* d_qoff, uint64_t nq, uint64_t* d_qwords,
                         const uint64_t* d_exc, uint64_t n_exc, uint64_t exc_base, uint64_t b_lo, uint64_t b_hi,
                         unsigned long long* d_first_bad, cudaStream_t s) {
  if (nq == 0) return cudaSuccess;
  uint64_t threads = nq * 8;
  unsigned grid = unsigned(std::min<uint64_t>((threads + 255) / 256, 148 * 64));
  pack2_kernel<<<grid, 256, 0, s>>>(d_crumbs, base, d_qoff, nq, d_qwords, b_lo, b_hi, d_first_bad);
  COUNT_LAUNCH();
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess || n_exc == 0) return e;
  patch_exceptions_kernel<<<unsigned((n_exc + 255) / 256), 256, 0, s>>>(d_exc, n_exc, exc_base, d_qoff, nq, d_qwords,
                                                                        b_lo, b_hi, d_first_bad);
  COUNT_LAUNCH();
  return cudaGetLastError();
}

__global__ void fill_offsets_kernel(uint64_t* __restrict__ qoff, uint64_t first, uint64_t len, uint64_t n) {
  const uint64_t i = blockIdx.x * uint64_t(blockDim.x) + threadIdx.x;
  if (i <= n) qoff[i] = first + i * len;
}
cudaError_t launch_fill_offsets(uint64_t* d_qoff, uint64_t first, uint64_t len, uint64_t n, cudaStream_t s) {
  fill_offsets_kernel<<<unsigned((n + 256) / 256), 256, 0, s>>>(d_qoff, first, len, n);
  COUNT_LAUNCH();
  return cudaGetLastError();
}

// ---- both strands: virtual offsets and words (kernels.hpp) ----
__global__ void strand_offsets_kernel(const uint64_t* __restrict__ qoff, uint64_t nq, uint64_t b_lo, uint64_t b_hi,
                                      uint64_t* __restrict__ voff) {
  const uint64_t q = blockIdx.x * uint64_t(blockDim.x) + threadIdx.x;
  if (q > nq) return;
  const uint64_t o0 = qoff[q];
  voff[2 * q] = 2 * o0;
  if (q == nq) return;
  const uint64_t o1 = qoff[q + 1];
  const bool ok = o0 >= b_lo && o1 <= b_hi && o1 >= o0 && o1 - o0 < (1ull << 32);  // checked_len's rule
  voff[2 * q + 1] = ok ? o0 + o1 : ~0ull;
}

cudaError_t launch_strand_offsets(const uint64_t* d_qoff, uint64_t nq, uint64_t b_lo, uint64_t b_hi, uint64_t* d_voff,
                                  cudaStream_t s) {
  strand_offsets_kernel<<<unsigned((nq + 256) / 256), 256, 0, s>>>(d_qoff, nq, b_lo, b_hi, d_voff);
  COUNT_LAUNCH();
  return cudaGetLastError();
}

// 16 nibbles -> the same 16 in reverse order
__device__ __forceinline__ uint64_t reverse_nibbles(uint64_t x) {
  x = ((x >> 4) & 0x0F0F0F0F0F0F0F0Full) | ((x & 0x0F0F0F0F0F0F0F0Full) << 4);
  const uint32_t lo = uint32_t(x), hi = uint32_t(x >> 32);
  return (uint64_t(__byte_perm(lo, 0, 0x0123)) << 32) | __byte_perm(hi, 0, 0x0123);
}

// 4 lanes per read; lane `sub` writes words sub, sub + 4, ... of both virtual queries.  Reverse-complement word w holds
// search-order symbols 16 w .. 16 w + 15 = the complements of the read's symbols L - 1 - 16 w down to L - 16 w - 16,
// which span at most two of the read's words.
__global__ void __launch_bounds__(256)
    strand_words_kernel(const uint64_t* __restrict__ qwords, const uint64_t* __restrict__ qoff, uint64_t nq,
                        ByteRange br, const uint64_t* __restrict__ voff, uint64_t* __restrict__ vwords) {
  const uint32_t sub = threadIdx.x & 3;
  const uint64_t ngroups = (gridDim.x * uint64_t(blockDim.x)) >> 2;
  for (uint64_t q = (blockIdx.x * uint64_t(blockDim.x) + threadIdx.x) >> 2; q < nq; q += ngroups) {
    const uint64_t o0 = qoff[q], o1 = qoff[q + 1];
    const uint32_t len = checked_len(o0, o1, br);
    if (len == 0) continue;  // refused by the prepass (its words do not exist) or empty
    const uint32_t nwords = (len + 15) >> 4;
    const uint64_t* const src = qwords + 4 * (q + (o0 >> 6));
    uint64_t* const fwd = vwords + 4 * (2 * q + (voff[2 * q] >> 6));
    uint64_t* const rev = vwords + 4 * (2 * q + 1 + (voff[2 * q + 1] >> 6));
    for (uint32_t w = sub; w < nwords; w += 4) {
      fwd[w] = src[w];
      // read symbols [a, a + 16) with a = L - 16 w - 16 (those below 0 do not exist)
      const int a = int(len) - 16 * int(w) - 16;
      uint64_t x;
      if (a >= 0) {
        const uint32_t wi = uint32_t(a) >> 4, sh = 4 * (uint32_t(a) & 15);
        const uint64_t lo = src[wi], hi = sh && 16 * (wi + 1) < len ? src[wi + 1] : 0ull;
        x = sh ? (lo >> sh) | (hi << (64 - sh)) : lo;
      } else {
        x = src[0] << (4 * uint32_t(-a));
      }
      x = reverse_nibbles(x);
      const uint64_t lt4 = ~(x >> 2) & 0x1111111111111111ull;  // codes below 4 (bit 2 clear)
      x ^= lt4 | (lt4 << 1);
      const uint32_t have = len - 16 * w;                       // symbols of this word (the rest stay 0)
      if (have < 16) x &= (1ull << (4 * have)) - 1;
      rev[w] = x;
    }
  }
}

cudaError_t launch_strand_words(const uint64_t* d_qwords, const uint64_t* d_qoff, uint64_t nq, uint64_t b_lo, uint64_t b_hi,
                                const uint64_t* d_voff, uint64_t* d_vwords, cudaStream_t s) {
  if (nq == 0) return cudaSuccess;
  const unsigned grid = unsigned(std::min<uint64_t>((nq * 4 + 255) / 256, 148 * 64));
  strand_words_kernel<<<grid, 256, 0, s>>>(d_qwords, d_qoff, nq, ByteRange{b_lo, b_hi}, d_voff, d_vwords);
  COUNT_LAUNCH();
  return cudaGetLastError();
}

// ------------------------------------------------------------------ backward search

// Start of a query: seed interval from the k-mer table when the last k symbols are all
// encoding symbols (replaces KmerLookupTable::get_range_for_kmer, kmer_lookup_table.rs:90-110,
// which recomputes the k-1 steps), else the single-symbol range (search.rs:43-48).
// Returns the number of symbols still to process.
template <int ALPHA>
__device__ __forceinline__ uint32_t begin_query(const IndexView& ix, const uint64_t* __restrict__ qwords,
                                                QueryStream<ALPHA>& qs, uint32_t len, uint32_t& sp,
                                                uint32_t& ep) {
  const uint32_t k = ix.kmer_len;
  if (k != 0 && len >= k) {
    uint64_t idx = 0;
    bool ok = true;
    if (ALPHA == 0) {
      uint64_t w = qs.w;  // k <= 16 symbols, all inside the first word
      uint64_t himask = 0xCCCCCCCCCCCCCCCCull >> (4 * (16 - k));
      ok = (w & himask) == 0;
      idx = kmer_index(w, k);
    } else {
      uint64_t w = qs.w, mult = 1;  // k <= 8
      for (uint32_t j = 0; j < k; j++) {
        uint32_t s = uint32_t(w >> (8 * j)) & 0xff;
        ok &= (s != AMINO_X) & (s != AMINO_SENTINEL);
        idx += uint64_t(s == 21 ? 19 : s - 1) * mult;
        mult *= 20;
      }
    }
    if (ok) {
      AWRY_CHK(idx < ix.n_table);
      uint2 r = __ldg(ix.table + idx);
      sp = r.x;
      ep = r.y;
      for (uint32_t j = 0; j < k; j++) qs.next(qwords);
      return len - k;
    }
  }
  uint32_t c = qs.next(qwords);
  if (c == (ALPHA == 0 ? uint32_t(DNA_SENTINEL) : uint32_t(AMINO_SENTINEL))) {
    sp = 1;
    ep = 0;
    return 0;
  }
  sp = ix.c_lo[c];
  ep = ix.c_hi[c];
  return len - 1;
}

// ---- scalar kernel: one thread per query (any alphabet) ----
// LIST: the queries to run are listed in defer[1 .. 1+defer[0]) (queries the cooperative kernels
// handed back because they contain an ambiguity symbol).
template <int ALPHA, int MODE, bool LIST>
__global__ void __launch_bounds__(256) search_scalar_kernel(IndexView ix, const uint64_t* __restrict__ qwords,
                                                            const uint64_t* __restrict__ qoff, uint64_t nq,
                                                            void* __restrict__ out,
                                                            const uint32_t* __restrict__ defer, ByteRange br) {
  uint64_t stride = gridDim.x * uint64_t(blockDim.x);
  uint64_t n = LIST ? uint64_t(defer[0]) : nq;
  for (uint64_t i = blockIdx.x * uint64_t(blockDim.x) + threadIdx.x; i < n; i += stride) {
    uint64_t q = LIST ? uint64_t(defer[1 + i]) : i;
    uint64_t o0 = qoff[q];
    uint32_t len = checked_len(o0, qoff[q + 1], br);
    uint32_t sp = 1, ep = 0;
    if (len != 0) {
      QueryStream<ALPHA> qs;
      qs.open(qwords, uint32_t(q), o0);
      uint32_t left = begin_query<ALPHA>(ix, qwords, qs, len, sp, ep);
      while (left != 0 && sp <= ep) {  // early break: fm_index.rs:409-416 / :425-433
        uint32_t c = qs.next(qwords);
        left--;
        if (c == (ALPHA == 0 ? uint32_t(DNA_SENTINEL) : uint32_t(AMINO_SENTINEL))) {
          sp = 1;
          ep = 0;
          break;
        }
        lf_update<ALPHA>(ix, sp, ep, c);
      }
    }
    store_result<MODE>(out, q, sp, ep);
  }
}

// ---- nucleotide kernel: LANES lanes cooperate on one query ----
// Each lane owns CH = 4/LANES chunks of the 64-B block (LANES=4: one LDG.128, LANES=2: one
// LDG.256, LANES=1: two LDG.256), computes its part of both inclusive ranks Occ(c,sp-1) and
// Occ(c,ep) from ONE block load whenever both fall in the same block, and the group reduces
// with LANES-wide xor shuffles.  Groups are persistent: when a query finishes (all symbols
// consumed or empty interval) the group moves to query q + G, so early exits refill lanes
// instead of idling them; all groups of a warp stay converged on the step body.
template <int LANES, int MODE, int TPB, int MINB>
__global__ void __launch_bounds__(TPB, MINB)
    search_dna_kernel(IndexView ix, const uint64_t* __restrict__ qwords,
                      const uint64_t* __restrict__ qoff, uint64_t nq, void* __restrict__ out, ByteRange br) {
  const uint32_t lane = threadIdx.x & 31;
  const uint32_t sub = lane % LANES;
  const uint32_t gmask = LANES == 1 ? (1u << lane) : (((1u << LANES) - 1u) << (lane - sub));
  const uint32_t G = (gridDim.x * blockDim.x) / LANES;  // nq < 2^32 per launch
  const uint32_t nq32 = uint32_t(nq);
  uint32_t q = (blockIdx.x * blockDim.x + threadIdx.x) / LANES;
  uint32_t cur = 0;
  bool have = false;
  uint32_t sp = 1, ep = 0, left = 0;
  QueryStream<0> qs;
  qs.w = qs.wnext = 0;
  qs.widx = 0;
  qs.inword = 0;

  for (;;) {
    if (left == 0 || sp > ep) {
      if (have && sub == 0) store_result<MODE>(out, cur, sp, ep);
      have = false;
      if (q >= nq32) break;
      cur = q;
      q = (q + G < q) ? 0xffffffffu : q + G;
      have = true;
      uint64_t o0 = qoff[cur];
      uint32_t len = checked_len(o0, qoff[cur + 1], br);
      sp = 1;
      ep = 0;
      left = 0;
      if (len != 0) {
        qs.open(qwords, cur, o0);
        left = begin_query<0>(ix, qwords, qs, len, sp, ep);
      }
      continue;
    }
    uint32_t c = qs.next(qwords);
    left--;
    uint32_t pa = sp - 1, pb = ep;
    uint32_t ba = pa >> 7, bb = pb >> 7;
    if (c < 4) {
      const uint4* blk = ix.blocks + size_t(ba) * DNA_BLOCK_UINT4;
      AWRY_CHK(uint64_t(ba) * DNA_BLOCK_UINT4 + 3 < ix.n_blocks_u4 && uint64_t(bb) * DNA_BLOCK_UINT4 + 3 < ix.n_blocks_u4);
      LaneChunks<LANES> x;
      x.load(blk, sub);
      uint32_t m0 = (c & 1) ? ~0u : 0u, m1 = (c & 2) ? ~0u : 0u;
      uint32_t ra = dna_partial_rank<LANES>(x, sub, pa & 127, c, m0, m1);
      if (bb != ba) x.load(ix.blocks + size_t(bb) * DNA_BLOCK_UINT4, sub);
      uint32_t rb = dna_partial_rank<LANES>(x, sub, pb & 127, c, m0, m1);
#pragma unroll
      for (int off = LANES / 2; off > 0; off >>= 1) {
        ra += __shfl_xor_sync(gmask, ra, off);
        rb += __shfl_xor_sync(gmask, rb, off);
      }
      uint32_t base = ix.c_lo[c];
      sp = base + ra;
      ep = base + rb - 1;
    } else if (c == DNA_N) {
      lf_update<0>(ix, sp, ep, c);  // rare: every lane of the group runs the scalar step
    } else {
      sp = 1;  // sentinel in a query: rejected by the prepass; keep the kernel well defined
      ep = 0;
    }
  }
}

template <int LANES, int MODE, int MINB>
static cudaError_t launch_search_dna_b(const IndexView& ix, const uint64_t* d_qwords, const uint64_t* d_qoff,
                                       uint64_t nq, void* d_out, int sm_count, int force_per_sm,
                                       cudaStream_t s, ByteRange br) {
  constexpr int TPB = 256;
  auto kern = search_dna_kernel<LANES, MODE, TPB, MINB>;
  int per_sm = 0;
  cudaError_t e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, TPB, 0);
  if (e != cudaSuccess) return e;
  if (per_sm < 1) per_sm = 1;
  if (force_per_sm > 0 && force_per_sm < per_sm) per_sm = force_per_sm;
  uint64_t max_blocks = uint64_t(sm_count) * uint64_t(per_sm);
  uint64_t need_blocks = (nq * LANES + TPB - 1) / TPB;
  unsigned grid = unsigned(std::max<uint64_t>(1, std::min(max_blocks, need_blocks)));
  kern<<<grid, TPB, 0, s>>>(ix, d_qwords, d_qoff, nq, d_out, br);
  COUNT_LAUNCH();
  return cudaGetLastError();
}

// blocks_per_sm picks the register budget the kernel was compiled for (launch bounds 256 x MINB)
template <int LANES, int MODE>
static cudaError_t launch_search_dna(const IndexView& ix, const uint64_t* d_qwords, const uint64_t* d_qoff,
                                     uint64_t nq, void* d_out, const SearchVariant& v, int sm_count,
                                     cudaStream_t s) {
  if (nq >= (1ull << 32)) return cudaErrorInvalidValue;
  switch (v.blocks_per_sm) {
    case 6: return launch_search_dna_b<LANES, MODE, 6>(ix, d_qwords, d_qoff, nq, d_out, sm_count, 0, s, ByteRange{v.b_lo, v.b_hi});
    case 8: return launch_search_dna_b<LANES, MODE, 8>(ix, d_qwords, d_qoff, nq, d_out, sm_count, 0, s, ByteRange{v.b_lo, v.b_hi});
    default:  // 0 / 4: no register cap (4 resident blocks); 1..3 run the same kernel on a smaller grid
      return launch_search_dna_b<LANES, MODE, 4>(ix, d_qwords, d_qoff, nq, d_out, sm_count, v.blocks_per_sm, s, ByteRange{v.b_lo, v.b_hi});
  }
}

// The k-mer seed table is read once per query at a random entry.  When it fits (amino k <= 5:
// 25.6 MB, nucleotide k <= 11: 32 MB) it is kept resident in L2 with a persisting access-policy
// window on the search launches.  Larger tables (nucleotide k = 13: 512 MB) get no window: setting
// L2 aside for a few percent of such a table was measured to slow the streaming pack kernel 2.5x
// (0.8 -> 2.0 ms) for no measurable gain in the search kernel.
struct TableWindow {
  const void* base = nullptr;
  size_t bytes = 0;
  float hit_ratio = 0.f;
};
static TableWindow table_window(const IndexView& ix) {
  TableWindow w;
  if (ix.table == nullptr || ix.kmer_len == 0) return w;
  size_t bytes = size_t(table_entries(int(ix.alphabet), ix.kmer_len)) * sizeof(uint2);
  int dev = 0, max_win = 0, max_persist = 0;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&max_win, cudaDevAttrMaxAccessPolicyWindowSize, dev);
  cudaDeviceGetAttribute(&max_persist, cudaDevAttrMaxPersistingL2CacheSize, dev);
  if (max_win <= 0 || max_persist <= 0 || bytes > size_t(max_win) || bytes > size_t(max_persist) / 2) return w;
  static thread_local int limit_set_for = -1;
  static thread_local size_t limit_bytes = 0;
  if (limit_set_for != dev || limit_bytes < bytes) {  // set aside just enough L2 for the table
    cudaDeviceSetLimit(cudaLimitPersistingL2CacheSize, bytes + (bytes >> 3));
    limit_set_for = dev;
    limit_bytes = bytes;
  }
  w.base = ix.table;
  w.bytes = bytes;
  w.hit_ratio = 1.0f;
  return w;
}

template <class Kern, class... Args>
static cudaError_t launch_with_table_window(Kern kern, unsigned grid, unsigned block, cudaStream_t s,
                                            const IndexView& ix, Args... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(grid);
  cfg.blockDim = dim3(block);
  cfg.dynamicSmemBytes = 0;
  cfg.stream = s;
  cudaLaunchAttribute attr[1];
  TableWindow w = table_window(ix);
  unsigned n_attr = 0;
  if (w.base != nullptr) {
    attr[0].id = cudaLaunchAttributeAccessPolicyWindow;
    attr[0].val.accessPolicyWindow.base_ptr = const_cast<void*>(w.base);
    attr[0].val.accessPolicyWindow.num_bytes = w.bytes;
    attr[0].val.accessPolicyWindow.hitRatio = w.hit_ratio;
    attr[0].val.accessPolicyWindow.hitProp = cudaAccessPropertyPersisting;
    attr[0].val.accessPolicyWindow.missProp = cudaAccessPropertyStreaming;
    n_attr = 1;
  }
  cfg.attrs = attr;
  cfg.numAttrs = n_attr;
  return cudaLaunchKernelEx(&cfg, kern, args...);
}

// ---- nucleotide pair kernel: 4 lanes per query, two query symbols per 128-B block access ----
// While at least two symbols remain the group reads ONE pair block (4 x LDG.256; fetching only the
// sectors a rank needs was measured and is NOT faster -- the line request is the unit of cost) and applies two
// backward-search steps at once; a lone last symbol uses the 1-step block (4 x LDG.128).
// Queries holding an ambiguity symbol (N) are handed to the scalar kernel through `defer`
// (defer[0] = count, then the query numbers), which keeps this kernel's register budget small.
// Same persistent-group refill as above.
// Which lane slice / 32-bit word of a pair block holds the count of pair p (see layout.cuh):
// p 0-2 -> slice 0, 3-5 -> 1, 6-8 -> 2 (words 5..7), 9-15 -> slice 3 (words 0..6).
__device__ __forceinline__ uint32_t pair_count_lane(uint32_t p) {
  constexpr uint32_t LUT = (1u << 6) | (1u << 8) | (1u << 10) | (2u << 12) | (2u << 14) | (2u << 16) |
                           (3u << 18) | (3u << 20) | (3u << 22) | (3u << 24) | (3u << 26) | (3u << 28) | (3u << 30);
  return (LUT >> (2 * p)) & 3u;
}

// One pair block slice in registers: the rows of this lane's 32-row chunk that hold `pair`
// (0 for slice 3) and this lane's share of the block-start count (0 unless it owns the slot).
struct PairSlice {
  uint32_t match, count;
};
__device__ __forceinline__ PairSlice pair_slice(const u32x8& x, uint32_t sub, uint32_t pair) {
  PairSlice r;
  uint32_t m = ~x.v[4];
#pragma unroll
  for (int p = 0; p < 4; p++) m &= ((pair >> p) & 1u) ? x.v[p] : ~x.v[p];
  r.match = sub < 3 ? m : 0u;
  const uint32_t lane = pair_count_lane(pair);
  const uint32_t word = lane < 3 ? pair + 5 - 3 * lane : pair - 9;
  const uint32_t t0 = (word & 1) ? x.v[1] : x.v[0], t1 = (word & 1) ? x.v[3] : x.v[2];
  const uint32_t t2 = (word & 1) ? x.v[5] : x.v[4], t3 = (word & 1) ? x.v[7] : x.v[6];
  const uint32_t u0 = (word & 2) ? t1 : t0, u1 = (word & 2) ? t3 : t2;
  const uint32_t c = (word & 4) ? u1 : u0;
  r.count = sub == lane ? c : 0u;
  return r;
}


// VFY ("finish in the text", count mode, needs ix.full_sa and ix.rtext): once the interval has narrowed to ONE
// row and at least VERIFY_MIN_LEFT symbols remain, the group stops stepping: SA[row] says where in the text
// the matched suffix stands, and the remaining symbols are compared with the text in front of it -- one suffix
// array read and one or two lines of text (4 x LDG.256 of the reversed, 4-bit-per-symbol copy, layout.cuh)
// instead of one block read per two symbols.  The count is the one backward search arrives at: a one-row
// interval can only stay one row (the row of the suffix `left` positions further left, when the text there
// spells the rest of the query) or become empty (fm_index.rs:409-416 with update_range_with_symbol, :559-582).
constexpr uint32_t VERIFY_MIN_LEFT = 8;

// LIST: the queries to run are the ones search_dna_wave_kernel left over (defer + nq + 2: count, ticket counter,
// then the query numbers), handed out from that ticket counter.
template <int MODE, int TPB, int MINB, bool VFY = false, bool LIST = false>
__global__ void __launch_bounds__(TPB, MINB)
    search_dna_pair_kernel(IndexView ix, const uint64_t* __restrict__ qwords,
                           const uint64_t* __restrict__ qoff, uint64_t nq, void* __restrict__ out,
                           uint32_t* __restrict__ defer, uint32_t ticket_sz, ByteRange br) {
  constexpr int LANES = 4;
  constexpr uint32_t NONE = 0xffffffffu, FULL = 0xffffffffu;
  // The group's packed query is staged in shared memory (a 16-word ring = 256 symbols, refilled
  // 8 words at a time for longer queries): one aligned 128-B global read per query instead of one
  // 8-byte read per 16 symbols, which matters because random LINE REQUESTS are the scarce resource.
  __shared__ uint64_t s_q[TPB / LANES][16];
  const uint32_t sub = threadIdx.x & 3;
  const uint32_t gbase = (threadIdx.x & 31) - sub;
  const uint32_t gmask = 0xfu << gbase;
  uint64_t* const ring = s_q[threadIdx.x / LANES];
  const uint32_t* const rest = defer + nq + 2;
  const uint32_t nq32 = LIST ? rest[0] : uint32_t(nq);
  // Queries are handed out dynamically from a counter behind the deferred list (defer[nq + 1]): with a
  // static stride every SM gets the same share and the kernel ends when the slowest SM does -- on B200 the
  // SMs do not all see the same random-access throughput (the gather probe's SMs are busy between 52 % and
  // 100 % of the time under a static split).  The hand-out is per WARP: the warp keeps a pool [pn, pe) of
  // query numbers in registers (identical in all lanes), the groups that need a query in an iteration are
  // counted with one ballot and numbered by rank, and lane 0 tops the pool up with ONE atomic per
  // `ticket_sz` queries.  So the counter sees one atomic per warp-ticket however the 8 groups of the warp
  // drift apart (a per-group grab collapses once reads that end early dephase the groups: same-address
  // atomics retire at ~0.5 G/s), and at the end of the batch at most ticket_sz - 1 queries wait in a pool.
  uint32_t* const ticket = LIST ? defer + nq + 3 : defer + nq + 1;
  const uint32_t lane = threadIdx.x & 31;
  uint32_t pn = 0, pe = 0;  // the warp's pool of query numbers
  bool more = true;         // the counter has not run past nq yet
  uint32_t cur = NONE;      // query in flight
  uint32_t sp = 1, ep = 0, left = 0, len = 0, nwords = 0;
  uint32_t ubase = 0;  // word index of the query's packed symbols
  uint32_t wlim = 8;   // word index at which the ring slides by 8 words
  // VFY: a query lives for ~8 loads, so the latency of the ticket atomic was 16 % of the warp-stall samples
  // (profiles/r02p_search_text_full.md): the warp draws its NEXT ticket when it starts on the current one and
  // looks at the result only when the pool runs dry (lane 0 holds it)
  uint32_t ahead = 0;
  if (VFY && lane == 0) ahead = atomicAdd(ticket, ticket_sz);

  // Every lane of the warp runs every iteration (the loop exit is a warp vote), so the rank
  // reduction can use full-mask shuffles; a group whose query ended refills in the same iteration.
  for (;;) {
    const bool want = left == 0 || sp > ep;
    const uint32_t wmask = __ballot_sync(FULL, want && sub == 0);  // one bit per group that needs a query
    uint32_t next_q = NONE;
    if (wmask) {  // warp-uniform
      const uint32_t n_want = __popc(wmask), avail = pe - pn;
      uint32_t b = 0, got = 0;
      if (n_want > avail && more) {
        uint32_t t = 0;
        if (VFY) {
          t = ahead;
          if (lane == 0 && t < nq32) ahead = atomicAdd(ticket, ticket_sz);
        } else if (lane == 0) {
          t = atomicAdd(ticket, ticket_sz);
        }
        t = __shfl_sync(FULL, t, 0);
        b = t;
        got = t < nq32 ? (nq32 - t < ticket_sz ? nq32 - t : ticket_sz) : 0u;
        more = got == ticket_sz;
      }
      const uint32_t r = __popc(wmask & ((1u << gbase) - 1u));  // this group's rank among the needy ones
      if (want) next_q = r < avail ? pn + r : (r - avail < got ? b + (r - avail) : NONE);
      if (n_want <= avail) {
        pn += n_want;
      } else if (got) {
        const uint32_t used = n_want - avail < got ? n_want - avail : got;
        pn = b + used;
        pe = b + got;
      } else {
        pn = pe;
      }
    }
    if (want) {
      if (cur != NONE && sub == 0) store_result<MODE>(out, cur, sp, ep);
      cur = NONE;
      left = 0;
      if (next_q != NONE) {
        cur = LIST ? rest[2 + next_q] : next_q;
        uint64_t ov = qoff[cur + (sub & 1)];  // lanes 0/1 fetch both ends with one request
        uint64_t o0 = __shfl_sync(gmask, ov, gbase), o1 = __shfl_sync(gmask, ov, gbase + 1);
        len = checked_len(o0, o1, br);
        sp = 1;
        ep = 0;
        if (len != 0) {
          ubase = 4 * (cur + uint32_t(o0 >> 6));
          nwords = (len + 15) >> 4;
          // ambiguity symbols (code >= 4) are looked for once, while the query is staged, not per step;
          // unused nibbles of the last word are 0
          uint32_t amb = 0;
          __syncwarp(gmask);
          if (4 * sub < nwords) {
            AWRY_CHK_QWORDS(ubase + 4 * sub, br, nq, 6);
            u32x8 t = ldg256(qwords + ubase + 4 * sub);
#pragma unroll
            for (int j = 0; j < 4; j++) {
              ring[4 * sub + j] = uint64_t(t.v[2 * j]) | (uint64_t(t.v[2 * j + 1]) << 32);
              if (4 * sub + j < nwords) amb |= (t.v[2 * j] | t.v[2 * j + 1]) & 0xCCCCCCCCu;
            }
          }
          const bool clean = !__any_sync(gmask, amb != 0);
          __syncwarp(gmask);
          wlim = 8;
          if (!clean) {  // hand the whole query to the scalar kernel
            if (sub == 0) defer[1 + atomicAdd(defer, 1u)] = cur;
            cur = NONE;
          } else {
            const uint32_t k = ix.kmer_len;
            const uint64_t w = ring[0];
            if (k != 0 && len >= k) {  // k <= 16: inside word 0
              uint64_t idx = 0;
              idx = kmer_index(w, k);
              AWRY_CHK(idx < ix.n_table);
      uint2 r = __ldg(ix.table + idx);
              sp = r.x;
              ep = r.y;
              left = len - k;
            } else {
              uint32_t c = uint32_t(w) & 15u;
              sp = ix.c_lo[c];
              ep = ix.c_hi[c];
              left = len - 1;
            }
          }
        }
      }
    }
    if (__all_sync(FULL, cur == NONE && pn == pe && !more)) break;

    bool active = left != 0 && sp <= ep;  // (a query that just ended is stored next iteration)
    const uint32_t pos = len - left;      // search-order index of the next symbol
    if (active && (pos >> 4) >= wlim) {   // long query: bring in words [wlim+8, wlim+16)
      uint32_t amb = 0;
      __syncwarp(gmask);
      if (sub < 2) {
        AWRY_CHK_QWORDS(ubase + wlim + 8 + 4 * sub, br, nq, 6);
        u32x8 t = ldg256(qwords + ubase + wlim + 8 + 4 * sub);  // in bounds: buffer padded by 32 words
#pragma unroll
        for (int j = 0; j < 4; j++) {
          ring[(wlim + 8 + 4 * sub + j) & 15] = uint64_t(t.v[2 * j]) | (uint64_t(t.v[2 * j + 1]) << 32);
          if (wlim + 8 + 4 * sub + j < nwords) amb |= (t.v[2 * j] | t.v[2 * j + 1]) & 0xCCCCCCCCu;
        }
      }
      const bool clean = !__any_sync(gmask, amb != 0);
      __syncwarp(gmask);
      wlim += 8;
      if (!clean) {  // ambiguity symbol further on: the scalar kernel redoes the whole query
        if (sub == 0) defer[1 + atomicAdd(defer, 1u)] = cur;
        cur = NONE;
        left = 0;
        active = false;
      }
    }
    // A pair step always starts on an EVEN symbol index (an odd start takes one single-symbol step
    // first), so both symbols are one byte of the ring: low nibble = symbol pos, high nibble = pos + 1.
    const uint32_t qb = reinterpret_cast<const uint8_t*>(ring)[(pos >> 1) & 127];
    // VFY: a query takes two or three steps in all, so the single-symbol step an odd seed length asks for would
    // be one of its ~8 dependent loads; there the two symbols are cut out of two ring bytes instead (the word
    // behind the current one is always in the ring: it slides only when `pos` enters word wlim)
    const bool two = VFY ? left >= 2 : (left >= 2 && (pos & 1) == 0);
    const uint32_t pa = sp - 1, pb = ep;
    uint32_t ra = 0, rb = 0, base = 0;
    if (active) {
      if (two) {
        uint32_t q2 = qb;
        if (VFY) q2 = ((qb | (uint32_t(reinterpret_cast<const uint8_t*>(ring)[((pos >> 1) + 1) & 127]) << 8)) >> (4 * (pos & 1))) & 0xffu;
        const uint32_t pair = ((q2 & 3u) << 2) | (q2 >> 4);
        const uint32_t ba = __umulhi(pa, 0xAAAAAAABu) >> 6;  // / 96
        const uint32_t la = pa - ba * PAIR_ROWS_PER_BLOCK, lb = pb - ba * PAIR_ROWS_PER_BLOCK;
        AWRY_CHK(uint64_t(ba) * PAIR_BLOCK_UINT4 + 7 < ix.n_pair_u4);
        u32x8 x = ldg256(ix.pair_blocks + size_t(ba) * PAIR_BLOCK_UINT4 + 2 * sub);
        PairSlice s = pair_slice(x, sub, pair);
        ra = __popc(s.match & low_mask(int(la) + 1 - int(32 * sub))) + s.count;
        if (lb < PAIR_ROWS_PER_BLOCK) {
          rb = __popc(s.match & low_mask(int(lb) + 1 - int(32 * sub))) + s.count;
        } else {  // the interval straddles two blocks (only while it is still wide): a real branch
          const uint32_t bb = __umulhi(pb, 0xAAAAAAABu) >> 6;
          AWRY_CHK(uint64_t(bb) * PAIR_BLOCK_UINT4 + 7 < ix.n_pair_u4);
          x = ldg256(ix.pair_blocks + size_t(bb) * PAIR_BLOCK_UINT4 + 2 * sub);
          s = pair_slice(x, sub, pair);
          rb = __popc(s.match & low_mask(int(pb - bb * PAIR_ROWS_PER_BLOCK) + 1 - int(32 * sub))) + s.count;
        }
        base = ix.c2[pair];
      } else {
        const uint32_t c1 = (qb >> (4 * (pos & 1))) & 15u;
        const uint32_t ba = pa >> 7, bb = pb >> 7;
        LaneChunks<4> y;
        AWRY_CHK(uint64_t(ba) * DNA_BLOCK_UINT4 + 3 < ix.n_blocks_u4 && uint64_t(bb) * DNA_BLOCK_UINT4 + 3 < ix.n_blocks_u4);
        y.load(ix.blocks + size_t(ba) * DNA_BLOCK_UINT4, sub);
        const uint32_t m0 = (c1 & 1) ? ~0u : 0u, m1 = (c1 & 2) ? ~0u : 0u;
        ra = dna_partial_rank<4>(y, sub, pa & 127, c1, m0, m1);
        if (bb != ba) y.load(ix.blocks + size_t(bb) * DNA_BLOCK_UINT4, sub);
        rb = dna_partial_rank<4>(y, sub, pb & 127, c1, m0, m1);
        base = ix.c_lo[c1];
      }
    }
    ra += __shfl_xor_sync(FULL, ra, 1);
    rb += __shfl_xor_sync(FULL, rb, 1);
    ra += __shfl_xor_sync(FULL, ra, 2);
    rb += __shfl_xor_sync(FULL, rb, 2);
    if (active) {
      sp = base + ra;
      ep = base + rb - 1;
      left -= two ? 2 : 1;
    }
    if (VFY) {
      // the unconsumed symbols [len - left, len) are compared out of the ring when it holds them all (always, for
      // queries of <= 256 symbols), else out of the packed words in global memory
      if (active && sp == ep && left >= VERIFY_MIN_LEFT) {
        const bool in_ring = nwords <= wlim + 8;
        AWRY_CHK(sp < ix.n_full_sa);
        const uint32_t p = __ldg(ix.full_sa + sp);  // the matched suffix stands at text[p ..]
        bool ok = p >= left;                          // else the rest of the query would start before the text
        if (ok) {
          const uint32_t done = len - left;
          // reversed text: rtext[i] = text[n - 1 - i], so the symbol of search-order index j (compared with
          // text[p + done - 1 - j]) is rtext[rb0 + j]
          const uint32_t rb0 = ix.bwt_len - p - done;
          const uint32_t s_first = (rb0 + done) >> 6, s_last = (rb0 + len - 1) >> 6;  // 32-B sectors = 64 symbols
          uint32_t bad = 0;
          for (uint32_t sec = s_first + sub; sec <= s_last; sec += 4) {
            AWRY_CHK(uint64_t(sec) * 32 + 31 < ix.n_rtext);
            const u32x8 t = ldg256(ix.rtext + size_t(sec) * 32);
            bad |= in_ring ? text_sector_mismatch<true>(t, ring, sec, rb0, done, len)
                           : text_sector_mismatch<false>(t, qwords + ubase, sec, rb0, done, len);
          }
          ok = !__any_sync(gmask, bad != 0u);
        }
        // finished either way -- one hit or none -- and stored here: the group draws a new query next iteration
        if (sub == 0) {
          if (MODE == OUT_COUNT_U64)
            reinterpret_cast<uint64_t*>(out)[cur] = ok ? 1ull : 0ull;
          else  // OUT_SP_CNT_U32 for a gather pass 2: the hit's text position itself
            reinterpret_cast<uint2*>(out)[cur] = ok ? make_uint2(p - left, CNT_AT_TEXT_POS) : make_uint2(1u, 0u);
        }
        cur = NONE;
        left = 0;
      }
    }
  }
}

// ---- nucleotide wave kernel (count / locate pass 1 with the text on the device) ----
// With "finish in the text" a 150-bp read is a chain of ~8 dependent loads of seven kinds -- its offsets, its
// packed words, its seed entry, two or three pair blocks, one suffix-array element, one or two lines of text --
// and search_dna_pair_kernel<VFY>, whose lane groups refill one by one, spends its time with the 8 groups of a
// warp in 8 different phases: every phase's load is issued alone, inside a branch the other groups wait behind
// (13.7 of 32 lanes active per instruction, 19 warps per issue slot waiting on a load,
// profiles/r02p_search_text_full.md).  Here a warp takes 8 queries at a time and walks them through the phases
// TOGETHER: every phase is one straight piece of code whose 8 loads go out side by side, the votes are full-warp
// ballots, and nothing is refilled in between -- the queries of a wave need the same few steps, so a wave ends
// together.  Queries that do not fit the pattern are handed on instead of stalling their wave: more than
// WAVE_MAX_STEPS steps with the interval still wider than one row (repeats), or more than 256 symbols -> the
// `rest` list, searched afterwards by search_dna_pair_kernel<VFY, LIST>; an ambiguity symbol -> the scalar kernel.
// Both block reads of an interval that straddles two blocks are issued before either is used.
// ASCII: the kernel reads the caller's query bytes (qbytes, indexed by the absolute offsets) instead of the words of
// pack_kernel and is its own prepass: it latches what pack_kernel latches into *first_bad, stages each read into the
// ring straight from its bytes (stage_ascii_ring), and writes the packed words of every query it hands on to `qw_out`
// (biased like `qwords`, which it does not read), so that the list kernels find them where they always do.
constexpr int WAVE_MAX_STEPS = 6;

// Query bytes [b, e) (addresses, at most 256 of them) -> the group's ring: every nibble of the read as pack_kernel
// writes it (nibbles past the read's length are left as they come: the search never reads them).  The read's 32-byte
// sectors are counted from its END: sector k holds bytes [end32 - 32 (k + 1), end32 - 32 k), end32 = e rounded up to
// 32, and converts to the 32 nibbles [32 k, 32 k + 32) of a sector-aligned stream in search order whose nibble j + pad
// is ring nibble j (pad = end32 - e).  Lane `sub` converts sectors sub, sub + 4, sub + 8 (aligned LDG.256) and writes
// the four 32-bit ring halves that start in its sector; the last of them needs the first half of sector k + 1, which
// the next lane holds (lane 3: lane 0 in the round before -- rounds run from the last sector down).  Returns non-zero
// when a byte of the sectors is not one of ACGT/acgt -- bytes of the neighbouring reads included (see the caller).
__device__ __forceinline__ uint32_t stage_ascii_ring(uintptr_t b, uintptr_t e, bool run, uint32_t sub, uint32_t gbase,
                                                     uint64_t* ring) {
  constexpr uint32_t FULL = 0xffffffffu;
  const uint32_t nsec = run ? uint32_t(((e - 1) >> 5) - (b >> 5)) + 1 : 0u;
  const uintptr_t end32 = (e + 31) & ~uintptr_t(31);
  const uint32_t pad = uint32_t(end32 - e), ph = pad >> 3, pl4 = 4 * (pad & 7);
  uint32_t* const r32 = reinterpret_cast<uint32_t*>(ring);
  uint32_t dirty = 0, carry = 0;
  const int rounds = int(__reduce_max_sync(FULL, (nsec + 3) >> 2));
#pragma unroll 1
  for (int i = rounds - 1; i >= 0; i--) {
    const uint32_t k = sub + 4u * uint32_t(i);
    uint32_t h[5] = {0u, 0u, 0u, 0u, 0u};
    if (k < nsec) {
      const u32x8 t = ldg256(reinterpret_cast<const void*>(end32 - 32 * uintptr_t(k + 1)));
      uint32_t nib[8];
#pragma unroll
      for (int j = 0; j < 8; j++) {
        uint32_t diff;
        nib[j] = ascii4_to_nibbles(t.v[j], diff);
        dirty |= diff;
      }
      h[0] = nib[7] | (nib[6] << 16);
      h[1] = nib[5] | (nib[4] << 16);
      h[2] = nib[3] | (nib[2] << 16);
      h[3] = nib[1] | (nib[0] << 16);
    }
    const uint32_t x = __shfl_sync(FULL, h[0], gbase + ((sub + 1) & 3));
    h[4] = sub == 3 ? carry : x;
    carry = x;
    if (k < nsec) {
#pragma unroll
      for (int j = 0; j < 4; j++) {
        const int m = int(4 * k) - int(ph) + j;
        if (m >= 0 && m < 32) r32[m] = __funnelshift_r(h[j], h[j + 1], pl4);
      }
    }
  }
  return dirty;
}

// The same for the strand flavour, whose lanes with `rc` set stage the ring of the read's reverse complement: its
// search order is the read's text order with every code complemented.  Their sectors are counted from the read's START
// (sector k holds bytes [b32 + 32 k, b32 + 32 k + 32), b32 = b rounded down to 32, pad = b - b32) and convert without
// the byte reversal, XOR 3 per code; the ring halves and the hand-over between lanes are the same, so both strands of a
// read load the same sectors.  (A function of its own: the single-strand kernels keep their code as it was.)
__device__ __forceinline__ uint32_t stage_strand_ring(uintptr_t b, uintptr_t e, bool run, uint32_t sub, uint32_t gbase,
                                                      uint64_t* ring, bool r) {
  constexpr uint32_t FULL = 0xffffffffu;
  const uint32_t nsec = run ? uint32_t(((e - 1) >> 5) - (b >> 5)) + 1 : 0u;
  const uintptr_t end32 = (e + 31) & ~uintptr_t(31), b32 = b & ~uintptr_t(31);
  const uint32_t pad = r ? uint32_t(b - b32) : uint32_t(end32 - e), ph = pad >> 3, pl4 = 4 * (pad & 7);
  uint32_t* const r32 = reinterpret_cast<uint32_t*>(ring);
  uint32_t dirty = 0, carry = 0;
  const int rounds = int(__reduce_max_sync(FULL, (nsec + 3) >> 2));
#pragma unroll 1
  for (int i = rounds - 1; i >= 0; i--) {
    const uint32_t k = sub + 4u * uint32_t(i);
    uint32_t h[5] = {0u, 0u, 0u, 0u, 0u};
    if (k < nsec) {
      const uintptr_t at = r ? b32 + 32 * uintptr_t(k) : end32 - 32 * uintptr_t(k + 1);
      const u32x8 t = ldg256(reinterpret_cast<const void*>(at));
      uint32_t nib[8];
#pragma unroll
      for (int j = 0; j < 8; j++) {
        uint32_t diff;
        nib[j] = ascii4_codes(__byte_perm(t.v[j], 0, r ? 0x3210u : 0x0123u), diff) ^ (r ? 0x3333u : 0u);
        dirty |= diff;
      }
#pragma unroll
      for (int j = 0; j < 4; j++)
        h[j] = r ? nib[2 * j] | (nib[2 * j + 1] << 16) : nib[7 - 2 * j] | (nib[6 - 2 * j] << 16);
    }
    const uint32_t x = __shfl_sync(FULL, h[0], gbase + ((sub + 1) & 3));
    h[4] = sub == 3 ? carry : x;
    carry = x;
    if (k < nsec) {
#pragma unroll
      for (int j = 0; j < 4; j++) {
        const int m = int(4 * k) - int(ph) + j;
        if (m >= 0 && m < 32) r32[m] = __funnelshift_r(h[j], h[j + 1], pl4);
      }
    }
  }
  return dirty;
}

// whether bytes [src, src + len) hold anything but ACGT/acgt (the group's 4 lanes take every 4th byte)
__device__ __forceinline__ uint32_t read_is_dirty(const uint8_t* src, uint32_t len, uint32_t sub) {
  uint32_t dirty = 0;
  for (uint32_t i = sub; i < len; i += 4) {
    uint32_t diff;
    ascii4_to_nibbles(0x41414100u | src[i], diff);  // the byte and three 'A'
    dirty |= diff;
  }
  return dirty;
}

// a query the ASCII wave kernel hands on without a ring: its words by pack_kernel's table path, which also latches a
// sentinel (the group's 4 lanes take words sub, sub + 4, ...); rc: the words of its reverse complement
template <bool STRAND = false>
__device__ __forceinline__ void pack_query_lut(const uint8_t* src, uint32_t len, uint32_t nwords, uint64_t* dst,
                                               uint32_t sub, const uint8_t* lut, uint64_t q, unsigned long long* first_bad,
                                               bool rc = false) {
  bool bad = false;
  for (uint32_t wi = sub; wi < nwords; wi += 4)
    dst[wi] = STRAND && rc ? pack_word_bytes<0, true>(src, len, wi << 4, lut, bad) : pack_word_bytes<0>(src, len, wi << 4, lut, bad);
  if (bad) atomicMin(first_bad, bad_query_code(q, BAD_QUERY));
}

// STRAND (ASCII flavour for both strands, launch_search_ascii with strands): the kernel hands out the batch's VIRTUAL
// queries v = 2q (read q) and v = 2q + 1 (its reverse complement); `qoff` and `br` are the virtual offsets of
// launch_strand_offsets and their byte range, from which the read's own ends are recovered (qoff[2q] / 2,
// qoff[2q + 2] / 2; a refused read has qoff[2q + 1] = ~0).  The two strands of a read sit in neighbouring lane groups
// of a warp (tickets and waves start at even v) and stage their rings from the same sectors; results, lists and
// handed-on words are per virtual query, what the kernel latches names the read.
template <int MODE, int TPB, bool ASCII, bool STRAND>
__device__ __forceinline__ void search_dna_wave(const IndexView& ix, const uint64_t* __restrict__ qwords,
                                                const uint64_t* __restrict__ qoff, uint64_t nq, void* __restrict__ out,
                                                uint32_t* __restrict__ defer, uint32_t ticket_sz, const ByteRange& br,
                                                const uint8_t* __restrict__ qbytes, uint64_t* qw_out,
                                                unsigned long long* first_bad) {
  static_assert(ASCII || !STRAND, "the strand flavour reads the caller's bytes");
  constexpr uint32_t FULL = 0xffffffffu;
  enum : uint32_t { W_NONE = 0, W_RUN = 1, W_EMPTY = 2 };  // no query (or handed on) / in progress / refused by the prepass
  __shared__ uint64_t s_q[TPB / 4][16];
  __shared__ uint8_t s_lut[ASCII ? 256 : 1];
  if (ASCII) {
    s_lut[threadIdx.x] = c_ascii_to_dsym[0][threadIdx.x];
    __syncthreads();
  }
  const uint32_t lane = threadIdx.x & 31, sub = lane & 3, gbase = lane - sub, gmask = 0xfu << gbase, grp = lane >> 2;
  uint64_t* const ring = s_q[threadIdx.x >> 2];
  const uint32_t nq32 = uint32_t(nq);
  uint32_t* const ticket = defer + nq + 1;
  uint32_t* const rest = defer + nq + 2;  // rest[0] = count, rest[2 ..] = query numbers
  uint32_t pn = 0, pe = 0;                // the warp's pool of query numbers (identical in all lanes)
  uint32_t ahead = 0;                     // the warp's NEXT ticket, drawn while the current one is worked on (lane 0)
  if (lane == 0) ahead = atomicAdd(ticket, ticket_sz);
  for (;;) {
    if (pn == pe) {  // warp-uniform
      uint32_t t = ahead;
      if (lane == 0 && t < nq32) ahead = atomicAdd(ticket, ticket_sz);
      t = __shfl_sync(FULL, t, 0);
      if (t >= nq32) break;
      pn = t;
      pe = t + (nq32 - t < ticket_sz ? nq32 - t : ticket_sz);
    }
    const uint32_t q = pn + grp;
    uint32_t st = q < pe ? W_RUN : W_NONE;
    pn = pe - pn > 8u ? pn + 8u : pe;

    // ---- offsets
    uint64_t ov = 0;
    if (STRAND) {  // lanes 0/1/2: qoff[2r], qoff[2r + 1], qoff[2r + 2] of read r = q / 2
      if (st == W_RUN && sub < 3) ov = __ldg(qoff + (q & ~1u) + sub);
    } else if (st == W_RUN) {
      ov = __ldg(qoff + q + (sub & 1));  // lanes 0/1 fetch both ends with one request
    }
    const uint64_t x0 = __shfl_sync(FULL, ov, gbase), x1 = __shfl_sync(FULL, ov, gbase + 1);
    const uint64_t x2 = STRAND ? __shfl_sync(FULL, ov, gbase + 2) : 0ull;
    const bool rc = STRAND && (q & 1u), refused = STRAND && x1 == ~0ull;
    const uint64_t o0 = STRAND ? x0 >> 1 : x0, o1 = STRAND ? x2 >> 1 : x1;  // the read's bytes
    const uint64_t vo0 = rc ? x1 : x0;                                      // the query's own offset (its word slot)
    const uint32_t rq = STRAND ? q >> 1 : q;                                // the read (what is latched)
    const ByteRange rbr = STRAND ? ByteRange{br.lo >> 1, br.hi >> 1} : br;
    const uint32_t len = st == W_RUN && !refused ? checked_len(o0, o1, rbr) : 0u;
    if (st == W_RUN && len == 0) {
      st = W_EMPTY;
      if (ASCII && sub == 0)  // as pack_kernel: offsets outside [b_lo, b_hi] first, else the query is empty
        atomicMin(first_bad,
                  bad_query_code(rq, !refused && o1 == o0 && o0 >= rbr.lo && o1 <= rbr.hi ? BAD_QUERY : BAD_OFFSETS));
    }
    const uint32_t nwords = (len + 15) >> 4;
    const uint32_t ubase = 4 * (q + uint32_t(vo0 >> 6));
    if (st == W_RUN && nwords > 16) {  // longer than the ring: the refilling kernel slides it
      if (ASCII) pack_query_lut<STRAND>(qbytes + o0, len, nwords, qw_out + ubase, sub, s_lut, rq, first_bad, rc);
      if (sub == 0) rest[2 + atomicAdd(rest, 1u)] = q;
      st = W_NONE;
    }
    // ---- query -> ring; ambiguity symbols (code >= 4; ASCII: any byte but ACGT/acgt) are looked for here, once
    uint32_t amb = 0;
    __syncwarp();  // the previous wave's ring reads are done
    if (ASCII) {
      if (STRAND)
        amb = stage_strand_ring(uintptr_t(qbytes + o0), uintptr_t(qbytes + o1), st == W_RUN, sub, gbase, ring, rc);
      else
        amb = stage_ascii_ring(uintptr_t(qbytes + o0), uintptr_t(qbytes + o1), st == W_RUN, sub, gbase, ring);
      // the first and last sector also hold bytes of the neighbouring reads: a group that saw a byte outside ACGT/acgt
      // looks again at its read's bytes alone (rare: a batch of clean reads never comes here)
      const uint32_t dirty_groups = __ballot_sync(FULL, amb != 0);
      if (dirty_groups) amb = st == W_RUN && (dirty_groups & gmask) ? read_is_dirty(qbytes + o0, len, sub) : 0u;
    } else if (st == W_RUN && 4 * sub < nwords) {
      AWRY_CHK_QWORDS(ubase + 4 * sub, br, nq, 6);
      const u32x8 t = ldg256(qwords + ubase + 4 * sub);
#pragma unroll
      for (int j = 0; j < 4; j++) {
        ring[4 * sub + j] = uint64_t(t.v[2 * j]) | (uint64_t(t.v[2 * j + 1]) << 32);
        if (4 * sub + j < nwords) amb |= (t.v[2 * j] | t.v[2 * j + 1]) & 0xCCCCCCCCu;
      }
    }
    const uint32_t amb_groups = __ballot_sync(FULL, amb != 0);
    __syncwarp();
    if (st == W_RUN && (amb_groups & gmask) != 0) {  // the scalar kernel takes the whole query
      if (ASCII) pack_query_lut<STRAND>(qbytes + o0, len, nwords, qw_out + ubase, sub, s_lut, rq, first_bad, rc);
      if (sub == 0) defer[1 + atomicAdd(defer, 1u)] = q;
      st = W_NONE;
    }
    // ---- seed
    uint32_t sp = 1, ep = 0, left = 0;
    if (st == W_RUN) {
      const uint32_t k = ix.kmer_len;
      const uint64_t w = ring[0];
      if (k != 0 && len >= k) {  // k <= 16: inside word 0
        const uint64_t idx = kmer_index(w, k);
        AWRY_CHK(idx < ix.n_table);
        const uint2 r = __ldg(ix.table + idx);
        sp = r.x;
        ep = r.y;
        left = len - k;
      } else {
        const uint32_t c = uint32_t(w) & 15u;
        sp = ix.c_lo[c];
        ep = ix.c_hi[c];
        left = len - 1;
      }
    }
    // ---- steps, until every interval of the wave is one row wide (or empty, or its query is used up)
#pragma unroll 1
    for (int it = 0; it <= WAVE_MAX_STEPS; it++) {
      const bool active = st == W_RUN && left != 0 && sp <= ep && !(sp == ep && left >= VERIFY_MIN_LEFT);
      if (!__any_sync(FULL, active)) break;
      if (it == WAVE_MAX_STEPS) {  // still wide: a repeat -- handed on, searched from its start by the refilling kernel
        if (active) {
          if (ASCII) {  // its words are the ring, with the nibbles past its length set to 0
#pragma unroll
            for (uint32_t j = 4 * sub; j < 4 * sub + 4; j++) {
              if (j < nwords) {
                AWRY_CHK_QWORDS(ubase + j, br, nq, 6);
                const uint32_t tail = len - 16 * j;
                qw_out[ubase + j] = tail >= 16 ? ring[j] : ring[j] & ((1ull << (4 * tail)) - 1);
              }
            }
          }
          if (sub == 0) rest[2 + atomicAdd(rest, 1u)] = q;
          st = W_NONE;
        }
        break;
      }
      const uint32_t pos = len - left;  // search-order index of the next symbol
      const uint8_t* const rb8 = reinterpret_cast<const uint8_t*>(ring);
      const uint32_t qb = rb8[(pos >> 1) & 127];
      const bool two = left >= 2;
      const uint32_t pa = sp - 1, pb = ep;
      uint32_t ra = 0, rb = 0, base = 0;
      if (active) {
        if (two) {  // (the word behind the current one is in the ring: it holds the whole query)
          const uint32_t q2 = ((qb | (uint32_t(rb8[((pos >> 1) + 1) & 127]) << 8)) >> (4 * (pos & 1))) & 0xffu;
          const uint32_t pair = ((q2 & 3u) << 2) | (q2 >> 4);
          const uint32_t ba = __umulhi(pa, 0xAAAAAAABu) >> 6, bb = __umulhi(pb, 0xAAAAAAABu) >> 6;  // / 96
          AWRY_CHK(uint64_t(ba) * PAIR_BLOCK_UINT4 + 7 < ix.n_pair_u4 && uint64_t(bb) * PAIR_BLOCK_UINT4 + 7 < ix.n_pair_u4);
          const u32x8 x = ldg256(ix.pair_blocks + size_t(ba) * PAIR_BLOCK_UINT4 + 2 * sub);
          u32x8 y = x;
          if (bb != ba) y = ldg256(ix.pair_blocks + size_t(bb) * PAIR_BLOCK_UINT4 + 2 * sub);
          PairSlice s = pair_slice(x, sub, pair);
          ra = __popc(s.match & low_mask(int(pa - ba * PAIR_ROWS_PER_BLOCK) + 1 - int(32 * sub))) + s.count;
          if (bb != ba) s = pair_slice(y, sub, pair);
          rb = __popc(s.match & low_mask(int(pb - bb * PAIR_ROWS_PER_BLOCK) + 1 - int(32 * sub))) + s.count;
          base = ix.c2[pair];
        } else {
          const uint32_t c1 = (qb >> (4 * (pos & 1))) & 15u;
          const uint32_t ba = pa >> 7, bb = pb >> 7;
          LaneChunks<4> y;
          AWRY_CHK(uint64_t(ba) * DNA_BLOCK_UINT4 + 3 < ix.n_blocks_u4 && uint64_t(bb) * DNA_BLOCK_UINT4 + 3 < ix.n_blocks_u4);
          y.load(ix.blocks + size_t(ba) * DNA_BLOCK_UINT4, sub);
          const uint32_t m0 = (c1 & 1) ? ~0u : 0u, m1 = (c1 & 2) ? ~0u : 0u;
          ra = dna_partial_rank<4>(y, sub, pa & 127, c1, m0, m1);
          if (bb != ba) y.load(ix.blocks + size_t(bb) * DNA_BLOCK_UINT4, sub);
          rb = dna_partial_rank<4>(y, sub, pb & 127, c1, m0, m1);
          base = ix.c_lo[c1];
        }
      }
      ra += __shfl_xor_sync(FULL, ra, 1);
      rb += __shfl_xor_sync(FULL, rb, 1);
      ra += __shfl_xor_sync(FULL, ra, 2);
      rb += __shfl_xor_sync(FULL, rb, 2);
      if (active) {
        sp = base + ra;
        ep = base + rb - 1;
        left -= two ? 2 : 1;
      }
    }
    // ---- finish in the text: a one-row interval with symbols left (see search_dna_pair_kernel<VFY>)
    const bool need = st == W_RUN && left != 0 && sp <= ep;  // (then sp == ep and left >= VERIFY_MIN_LEFT)
    uint32_t p = 0;
    if (need) {
      AWRY_CHK(sp < ix.n_full_sa);
      p = __ldg(ix.full_sa + sp);  // the matched suffix stands at text[p ..]
    }
    bool ok = need && p >= left;   // else the rest of the query would start before the text
    uint32_t bad = 0;
    if (ok) {
      const uint32_t done = len - left;
      const uint32_t rb0 = ix.bwt_len - p - done;  // reversed-text index of search-order symbol 0
      const uint32_t s_first = (rb0 + done) >> 6, s_last = (rb0 + len - 1) >> 6;  // 32-B sectors = 64 symbols
      for (uint32_t sec = s_first + sub; sec <= s_last; sec += 4) {
        AWRY_CHK(uint64_t(sec) * 32 + 31 < ix.n_rtext);
        const u32x8 t = ldg256(ix.rtext + size_t(sec) * 32);
        bad |= text_sector_mismatch(t, ring, sec, rb0, done, len);
      }
    }
    const uint32_t bad_groups = __ballot_sync(FULL, bad != 0);
    ok = ok && (bad_groups & gmask) == 0;
    // ---- results
    if (sub == 0) {
      if (st == W_EMPTY) {
        store_result<MODE>(out, q, 1u, 0u);
      } else if (st == W_RUN && !need) {
        store_result<MODE>(out, q, sp, ep);
      } else if (st == W_RUN) {  // one hit or none
        if (MODE == OUT_COUNT_U64)
          reinterpret_cast<uint64_t*>(out)[q] = ok ? 1ull : 0ull;
        else  // OUT_SP_CNT_U32 for a gather pass 2: the hit's text position itself
          reinterpret_cast<uint2*>(out)[q] = ok ? make_uint2(p - left, CNT_AT_TEXT_POS) : make_uint2(1u, 0u);
      }
    }
  }
}

template <int MODE, int TPB, int MINB, bool ASCII = false>
__global__ void __launch_bounds__(TPB, MINB)
    search_dna_wave_kernel(IndexView ix, const uint64_t* __restrict__ qwords, const uint64_t* __restrict__ qoff,
                           uint64_t nq, void* __restrict__ out, uint32_t* __restrict__ defer, uint32_t ticket_sz,
                           ByteRange br, const uint8_t* __restrict__ qbytes, uint64_t* qw_out,
                           unsigned long long* first_bad) {
  search_dna_wave<MODE, TPB, ASCII, false>(ix, qwords, qoff, nq, out, defer, ticket_sz, br, qbytes, qw_out, first_bad);
}

template <int MODE, int TPB, int MINB>
__global__ void __launch_bounds__(TPB, MINB)
    search_dna_strand_wave_kernel(IndexView ix, const uint64_t* __restrict__ qwords, const uint64_t* __restrict__ qoff,
                                  uint64_t nq, void* __restrict__ out, uint32_t* __restrict__ defer, uint32_t ticket_sz,
                                  ByteRange br, const uint8_t* __restrict__ qbytes, uint64_t* qw_out,
                                  unsigned long long* first_bad) {
  search_dna_wave<MODE, TPB, true, true>(ix, qwords, qoff, nq, out, defer, ticket_sz, br, qbytes, qw_out, first_bad);
}

// ---- nucleotide pair kernel, NS queries per lane group, every load of a query's life in the same slot of
// the instruction stream ("state machine") ----
// search_dna_pair_kernel above has two costs the block reads do not explain.  (1) A query's start is a chain
// of three dependent loads (its offsets -> its packed words -> its seed-table entry) that runs inside a
// divergent branch: while ONE lane group of a warp starts a query, the other seven wait for all three
// latencies, so reads that end early (dephasing the groups) cost far more than the steps they save.
// (2) One block read in flight per lane group: 384 per SM at 6 x 256 threads.
// Here a lane group owns NS query SLOTS, and every slot is in one of five states whose load is issued at
// the same point of the loop -- ST_OFFS (its two offsets), ST_WORDS (its packed symbols, into the
// shared-memory ring), ST_SEED (its k-mer table entry), ST_STEP (one pair block = two LF steps, or a
// one-symbol block), ST_RING (8 more words of a long query) -- then all slots consume.  A group that starts
// a query spends three iterations on it without holding anyone up, the loads of the NS slots of a lane
// overlap, and the warp-level bookkeeping (hand-out ballot, exit vote, loop) is paid once per NS block reads.
// Everything else is as above: 4 lanes per query, per-warp pool of query numbers topped up with one atomic,
// queries with an ambiguity symbol go to the scalar kernel through `defer`, full-mask xor-shuffles.
// MEASURED (profiles/r02_s1_ab_state_machine_*.log, 10 launches back to back, 10 M x 150 bp): it LOSES --
// 19.6 ms (1 slot, 8 x 256 threads/SM) and 18.7 ms (2 slots, 5 x 256) against 17.8 ms for the branching kernel,
// 21.8 / 20.6 against 19.1 ms with 10 % mismatching reads, 0.58 / 0.57 against 0.54 ms for 1 M x 50 bp.
// The state dispatch adds ~20 % instructions per block read, and at ~41 G block reads/s the part sits at its
// power cap (sw_power_cap in every bench line): what a launch costs follows the instructions it issues, not
// the loads it has in flight, so more memory-level parallelism per lane buys nothing here.  The default stays
// search_dna_pair_kernel; this one is bit-exact (the GPU suite passes with AWRY_B200_SLOTS=1 and =2) and
// selectable (awry_set_search_variant(81 / 82)) so the comparison can be repeated.
// VFY (count mode, see search_dna_pair_kernel): two more states -- ST_SA (the suffix-array element of a one-row
// interval) and ST_TEXT (the sectors of the reversed text the rest of the query is compared with; at most 4, so
// it is entered with at most 193 symbols left).  With the comparison a 150-bp read is ~8 dependent loads of
// seven different kinds instead of ~70 block reads, which is the workload this kernel was written for.
template <int MODE, int TPB, int MINB, int NS, bool VFY = false>
__global__ void __launch_bounds__(TPB, MINB)
    search_dna_pairx_kernel(IndexView ix, const uint64_t* __restrict__ qwords,
                            const uint64_t* __restrict__ qoff, uint64_t nq, void* __restrict__ out,
                            uint32_t* __restrict__ defer, uint32_t ticket_sz, ByteRange br) {
  constexpr uint32_t NONE = 0xffffffffu, FULL = 0xffffffffu;
  enum : uint32_t { ST_IDLE = 0, ST_OFFS = 1, ST_WORDS = 2, ST_SEED = 3, ST_STEP = 4, ST_RING = 5, ST_SA = 6, ST_TEXT = 7 };
  constexpr uint32_t PC_STEP = 0x200u, PC_TWO = 0x100u;  // pc: "this slot issued a step" | "a two-symbol step" | symbols
  __shared__ uint64_t s_q[NS][TPB / 4][16];
  __shared__ uint32_t s_amb[NS][TPB / 4];  // an ambiguity symbol was seen while staging (set by any lane of the group)
  const uint32_t lane = threadIdx.x & 31, sub = lane & 3, gbase = lane - sub;
  const uint32_t gmask = 0xfu << gbase;
  const uint32_t grp = threadIdx.x >> 2;
  const uint32_t nq32 = uint32_t(nq);
  uint32_t* const ticket = defer + nq + 1;
  uint32_t pn = 0, pe = 0;  // the warp's pool of query numbers (see search_dna_pair_kernel)
  bool more = true;
  uint32_t st[NS], cur[NS], sp[NS], ep[NS], left[NS], len[NS], ubase[NS], wlim[NS];
#pragma unroll
  for (int s = 0; s < NS; s++) {
    st[s] = ST_IDLE;
    cur[s] = NONE;
    sp[s] = 1;
    ep[s] = 0;
    left[s] = len[s] = ubase[s] = 0;
    wlim[s] = 8;
  }

  for (;;) {
    // ---- hand-out: lane `s` of a group reports slot s (NS <= 4), one ballot for the warp
    bool want_here = false;
#pragma unroll
    for (int s = 0; s < NS; s++) want_here |= (sub == uint32_t(s)) && st[s] == ST_IDLE;
    const uint32_t wmask = __ballot_sync(FULL, want_here);
    if (wmask != 0 && (pn != pe || more)) {  // warp-uniform
      const uint32_t n_want = __popc(wmask), avail = pe - pn;
      uint32_t b = 0, got = 0;
      if (n_want > avail && more) {
        uint32_t t = 0;
        if (lane == 0) t = atomicAdd(ticket, ticket_sz);
        t = __shfl_sync(FULL, t, 0);
        b = t;
        got = t < nq32 ? (nq32 - t < ticket_sz ? nq32 - t : ticket_sz) : 0u;
        more = got == ticket_sz;
      }
#pragma unroll
      for (int s = 0; s < NS; s++) {
        if (st[s] == ST_IDLE) {
          const uint32_t r = __popc(wmask & ((1u << (gbase + s)) - 1u));  // this slot's rank among the needy ones
          const uint32_t nx = r < avail ? pn + r : (r - avail < got ? b + (r - avail) : NONE);
          if (nx != NONE) {
            cur[s] = nx;
            st[s] = ST_OFFS;
          }
        }
      }
      if (n_want <= avail) {
        pn += n_want;
      } else if (got) {
        const uint32_t used = n_want - avail < got ? n_want - avail : got;
        pn = b + used;
        pe = b + got;
      } else {
        pn = pe;
      }
    }
    bool idle = true;
#pragma unroll
    for (int s = 0; s < NS; s++) idle &= st[s] == ST_IDLE;
    if (__all_sync(FULL, idle)) break;  // a slot still idle after the hand-out: the batch has been given out

    // ---- issue: one load per slot
    u32x8 x[NS];
    uint32_t pc[NS];
#pragma unroll
    for (int s = 0; s < NS; s++) {
      pc[s] = 0;
#pragma unroll
      for (int i = 0; i < 8; i++) x[s].v[i] = 0;
      if (st[s] == ST_STEP) {
        const uint32_t pos = len[s] - left[s];       // search-order index of the next symbol
        if ((pos >> 4) >= wlim[s]) st[s] = ST_RING;  // long query: the ring has to slide first
      }
      if (st[s] == ST_STEP) {
        const uint32_t pos = len[s] - left[s];
        // A pair step always starts on an EVEN symbol index (an odd start takes one single-symbol step
        // first), so both symbols are one byte of the ring: low nibble = symbol pos, high nibble = pos + 1.
        const uint32_t qb = reinterpret_cast<const uint8_t*>(s_q[s][grp])[(pos >> 1) & 127];
        const uint32_t pa = sp[s] - 1;
        if (left[s] >= 2 && (pos & 1) == 0) {
          pc[s] = PC_STEP | PC_TWO | ((qb & 3u) << 2) | (qb >> 4);
          const uint32_t ba = __umulhi(pa, 0xAAAAAAABu) >> 6;  // / 96
          AWRY_CHK(uint64_t(ba) * PAIR_BLOCK_UINT4 + 7 < ix.n_pair_u4);
          x[s] = ldg256(ix.pair_blocks + size_t(ba) * PAIR_BLOCK_UINT4 + 2 * sub);
        } else {
          pc[s] = PC_STEP | ((qb >> (4 * (pos & 1))) & 15u);
          AWRY_CHK(uint64_t(pa >> 7) * DNA_BLOCK_UINT4 + 3 < ix.n_blocks_u4);
          const uint4 c = ldg128(ix.blocks + size_t(pa >> 7) * DNA_BLOCK_UINT4 + sub);
          x[s].v[0] = c.x;
          x[s].v[1] = c.y;
          x[s].v[2] = c.z;
          x[s].v[3] = c.w;
        }
      } else if (st[s] == ST_OFFS) {
        const uint64_t ov = __ldg(qoff + cur[s] + (sub & 1));  // lanes 0/1 fetch both ends with one request
        x[s].v[0] = uint32_t(ov);
        x[s].v[1] = uint32_t(ov >> 32);
      } else if (st[s] == ST_WORDS) {
        if (4 * sub < ((len[s] + 15) >> 4)) {
          AWRY_CHK_QWORDS(ubase[s] + 4 * sub, br, nq, 6);
          x[s] = ldg256(qwords + ubase[s] + 4 * sub);
        }
      } else if (st[s] == ST_SEED) {
        const uint32_t k = ix.kmer_len;
        const uint64_t w = s_q[s][grp][0];  // k <= 16: inside word 0
        uint64_t idx = 0;
        idx = kmer_index(w, k);
        AWRY_CHK(idx < ix.n_table);
        const uint2 r = __ldg(ix.table + idx);
        x[s].v[0] = r.x;
        x[s].v[1] = r.y;
      } else if (st[s] == ST_RING) {
        if (sub < 2) {
          AWRY_CHK_QWORDS(ubase[s] + wlim[s] + 8 + 4 * sub, br, nq, 6);
          x[s] = ldg256(qwords + ubase[s] + wlim[s] + 8 + 4 * sub);  // in bounds: buffer padded by 32 words
        }
      } else if (VFY && st[s] == ST_SA) {
        AWRY_CHK(sp[s] < ix.n_full_sa);
        x[s].v[0] = __ldg(ix.full_sa + sp[s]);
      } else if (VFY && st[s] == ST_TEXT) {  // ubase = reversed-text index of search-order symbol 0 (set by ST_SA)
        const uint32_t done = len[s] - left[s];
        const uint32_t sec = ((ubase[s] + done) >> 6) + sub;
        if (sec <= ((ubase[s] + len[s] - 1) >> 6)) {
          AWRY_CHK(uint64_t(sec) * 32 + 31 < ix.n_rtext);
          x[s] = ldg256(ix.rtext + size_t(sec) * 32);
        }
      }
    }

    // ---- consume
    uint32_t ra[NS], rb[NS];
#pragma unroll
    for (int s = 0; s < NS; s++) {
      ra[s] = rb[s] = 0;
      uint64_t* const ring = s_q[s][grp];
      if (st[s] == ST_STEP) {
        const uint32_t pa = sp[s] - 1, pb = ep[s];
        if (pc[s] & PC_TWO) {
          const uint32_t pair = pc[s] & 15u;
          const uint32_t ba = __umulhi(pa, 0xAAAAAAABu) >> 6;
          const uint32_t la = pa - ba * PAIR_ROWS_PER_BLOCK, lb = pb - ba * PAIR_ROWS_PER_BLOCK;
          PairSlice sl = pair_slice(x[s], sub, pair);
          ra[s] = __popc(sl.match & low_mask(int(la) + 1 - int(32 * sub))) + sl.count;
          if (lb < PAIR_ROWS_PER_BLOCK) {
            rb[s] = __popc(sl.match & low_mask(int(lb) + 1 - int(32 * sub))) + sl.count;
          } else {  // the interval straddles two blocks (only while it is still wide): a real branch
            const uint32_t bb = __umulhi(pb, 0xAAAAAAABu) >> 6;
            AWRY_CHK(uint64_t(bb) * PAIR_BLOCK_UINT4 + 7 < ix.n_pair_u4);
            const u32x8 y = ldg256(ix.pair_blocks + size_t(bb) * PAIR_BLOCK_UINT4 + 2 * sub);
            sl = pair_slice(y, sub, pair);
            rb[s] = __popc(sl.match & low_mask(int(pb - bb * PAIR_ROWS_PER_BLOCK) + 1 - int(32 * sub))) + sl.count;
          }
        } else {
          const uint32_t c1 = pc[s] & 15u;
          const uint32_t ba = pa >> 7, bb = pb >> 7;
          LaneChunks<4> y;
          y.c[0] = make_uint4(x[s].v[0], x[s].v[1], x[s].v[2], x[s].v[3]);
          const uint32_t m0 = (c1 & 1) ? ~0u : 0u, m1 = (c1 & 2) ? ~0u : 0u;
          ra[s] = dna_partial_rank<4>(y, sub, pa & 127, c1, m0, m1);
          AWRY_CHK(uint64_t(bb) * DNA_BLOCK_UINT4 + 3 < ix.n_blocks_u4);
          if (bb != ba) y.load(ix.blocks + size_t(bb) * DNA_BLOCK_UINT4, sub);
          rb[s] = dna_partial_rank<4>(y, sub, pb & 127, c1, m0, m1);
        }
      } else if (st[s] == ST_OFFS) {
        const uint64_t ov = uint64_t(x[s].v[0]) | (uint64_t(x[s].v[1]) << 32);
        const uint64_t o0 = __shfl_sync(gmask, ov, gbase), o1 = __shfl_sync(gmask, ov, gbase + 1);
        len[s] = checked_len(o0, o1, br);
        sp[s] = 1;
        ep[s] = 0;
        left[s] = 0;
        wlim[s] = 8;
        if (len[s] == 0) {  // refused by the prepass: an empty result, the call fails anyway
          if (sub == 0) store_result<MODE>(out, cur[s], 1u, 0u);
          st[s] = ST_IDLE;
        } else {
          ubase[s] = 4 * (cur[s] + uint32_t(o0 >> 6));
          if (sub == 0) s_amb[s][grp] = 0;
          st[s] = ST_WORDS;
        }
      } else if (st[s] == ST_WORDS) {
        // ambiguity symbols (code >= 4) are looked for once, while the query is staged, not per step;
        // unused nibbles of the last word are 0
        const uint32_t nwords = (len[s] + 15) >> 4;
        uint32_t amb = 0;
        __syncwarp(gmask);  // the previous query's last ring reads, and the flag's reset, are done
        if (4 * sub < nwords) {
#pragma unroll
          for (int j = 0; j < 4; j++) {
            ring[4 * sub + j] = uint64_t(x[s].v[2 * j]) | (uint64_t(x[s].v[2 * j + 1]) << 32);
            if (4 * sub + j < nwords) amb |= (x[s].v[2 * j] | x[s].v[2 * j + 1]) & 0xCCCCCCCCu;
          }
        }
        if (amb) s_amb[s][grp] = 1;
        __syncwarp(gmask);
        if (s_amb[s][grp]) {  // hand the whole query to the scalar kernel
          if (sub == 0) defer[1 + atomicAdd(defer, 1u)] = cur[s];
          st[s] = ST_IDLE;
        } else if (ix.kmer_len != 0 && len[s] >= ix.kmer_len) {
          st[s] = ST_SEED;
        } else {
          const uint32_t c = uint32_t(ring[0]) & 15u;
          sp[s] = ix.c_lo[c];
          ep[s] = ix.c_hi[c];
          left[s] = len[s] - 1;
          st[s] = ST_STEP;
        }
      } else if (st[s] == ST_SEED) {
        sp[s] = x[s].v[0];
        ep[s] = x[s].v[1];
        left[s] = len[s] - ix.kmer_len;
        st[s] = ST_STEP;
      } else if (st[s] == ST_RING) {
        const uint32_t nwords = (len[s] + 15) >> 4;
        uint32_t amb = 0;
        __syncwarp(gmask);
        if (sub < 2) {
#pragma unroll
          for (int j = 0; j < 4; j++) {
            ring[(wlim[s] + 8 + 4 * sub + j) & 15] = uint64_t(x[s].v[2 * j]) | (uint64_t(x[s].v[2 * j + 1]) << 32);
            if (wlim[s] + 8 + 4 * sub + j < nwords) amb |= (x[s].v[2 * j] | x[s].v[2 * j + 1]) & 0xCCCCCCCCu;
          }
        }
        if (amb) s_amb[s][grp] = 1;
        __syncwarp(gmask);
        wlim[s] += 8;
        if (s_amb[s][grp]) {  // ambiguity symbol further on: the scalar kernel redoes the whole query
          if (sub == 0) defer[1 + atomicAdd(defer, 1u)] = cur[s];
          st[s] = ST_IDLE;
        } else {
          st[s] = ST_STEP;
        }
      } else if (VFY && st[s] == ST_SA) {
        const uint32_t p = x[s].v[0];  // the matched suffix stands at text[p ..]
        if (p < left[s]) {             // the rest of the query would start before the text
          if (sub == 0) store_result<MODE>(out, cur[s], 1u, 0u);
          st[s] = ST_IDLE;
        } else {
          ubase[s] = ix.bwt_len - p - (len[s] - left[s]);  // (the ring needs no more words: ubase is free)
          st[s] = ST_TEXT;
        }
      } else if (VFY && st[s] == ST_TEXT) {
        const uint32_t done = len[s] - left[s], rb0 = ubase[s];
        const uint32_t sec = ((rb0 + done) >> 6) + sub;
        uint32_t bad = 0;
        if (sec <= ((rb0 + len[s] - 1) >> 6)) bad = text_sector_mismatch(x[s], ring, sec, rb0, done, len[s]);
        const bool ok = !__any_sync(gmask, bad != 0u);
        if (sub == 0) store_result<MODE>(out, cur[s], ok ? sp[s] : 1u, ok ? ep[s] : 0u);  // one row, or empty
        st[s] = ST_IDLE;
      }
    }
    // rank reduction over the 4 lanes of every group, all slots, full-mask shuffles (every lane is here)
#pragma unroll
    for (int s = 0; s < NS; s++) {
      ra[s] += __shfl_xor_sync(FULL, ra[s], 1);
      rb[s] += __shfl_xor_sync(FULL, rb[s], 1);
    }
#pragma unroll
    for (int s = 0; s < NS; s++) {
      ra[s] += __shfl_xor_sync(FULL, ra[s], 2);
      rb[s] += __shfl_xor_sync(FULL, rb[s], 2);
    }
    // ---- apply the steps; a query that ends (all symbols consumed, or an empty interval: the early break
    // of fm_index.rs:409-416 / :425-433) is stored and its slot draws a new query in the next iteration
#pragma unroll
    for (int s = 0; s < NS; s++) {
      if (pc[s] & PC_STEP) {
        const uint32_t base = (pc[s] & PC_TWO) ? ix.c2[pc[s] & 15u] : ix.c_lo[pc[s] & 15u];
        sp[s] = base + ra[s];
        ep[s] = base + rb[s] - 1;
        left[s] -= (pc[s] & PC_TWO) ? 2 : 1;
      }
      if (st[s] == ST_STEP && (left[s] == 0 || sp[s] > ep[s])) {  // (also: a query no longer than its seed)
        if (sub == 0) store_result<MODE>(out, cur[s], sp[s], ep[s]);
        st[s] = ST_IDLE;
      }
      // one row left and the unconsumed symbols all in the ring, within four text sectors: finish in the text
      if (VFY && st[s] == ST_STEP && sp[s] == ep[s] && left[s] >= VERIFY_MIN_LEFT && left[s] <= 193u &&
          ((len[s] + 15) >> 4) <= wlim[s] + 8)
        st[s] = ST_SA;
    }
  }
}

template <int MODE, int MINB, bool VFY = false>
static cudaError_t launch_search_pair_b(const IndexView& ix, const uint64_t* d_qwords, const uint64_t* d_qoff,
                                        uint64_t nq, void* d_out, uint32_t* d_defer, int force_per_sm,
                                        int sm_count, cudaStream_t s, uint32_t avg_len, ByteRange br) {
  constexpr int TPB = 256;
  auto kern = search_dna_pair_kernel<MODE, TPB, MINB, VFY>;
  int per_sm = 0;
  cudaError_t e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, TPB, 0);
  if (e != cudaSuccess) return e;
  if (per_sm < 1) per_sm = 1;
  if (force_per_sm > 0 && force_per_sm < per_sm) per_sm = force_per_sm;
  uint64_t max_blocks = uint64_t(sm_count) * uint64_t(per_sm);
  uint64_t need_blocks = (nq * 4 + TPB - 1) / TPB;
  unsigned grid = unsigned(std::max<uint64_t>(1, std::min(max_blocks, need_blocks)));
  static const uint32_t ticket_env = [] {  // AWRY_B200_TICKET: fixed ticket size (experiments)
    if (const char* e = getenv("AWRY_B200_TICKET")) return uint32_t(std::min(1024l, std::max(1l, strtol(e, nullptr, 10))));
    return 0u;
  }();
  // per-WARP ticket of the pair kernel (8 lane groups): one query per group for 150-bp reads, more for
  // short queries; a small batch gets small tickets whatever the length, so that every warp still draws
  // several (a 256 k-query chunk of 50-bp queries with 32-query tickets is 1.15 tickets per warp).  Measured
  // effect: small -- 1 M x 50-bp queries 0.567 -> 0.553 ms, a 256 k-query chunk 0.34 ms either way (there the
  // fixed cost of filling and draining the persistent grid dominates, profiles/r01_s50_locate_gpu_timeline.log)
  uint32_t per_group = avg_len == 0 ? 2u : std::min(8u, std::max(1u, 200u / avg_len));
  per_group = ticket_cap(per_group, nq, uint64_t(grid) * (TPB / 4), avg_len);
  const uint32_t ticket_sz = ticket_env ? ticket_env : 8u * per_group;
  e = launch_with_table_window(kern, grid, TPB, s, ix, ix, d_qwords, d_qoff, nq, d_out, d_defer, ticket_sz, br);
  COUNT_LAUNCH();
  if (e != cudaSuccess) return e;
  // queries with ambiguity symbols: scalar kernel over the deferred list (empty for clean batches)
  search_scalar_kernel<0, MODE, true><<<unsigned(sm_count) * 2, 256, 0, s>>>(ix, d_qwords, d_qoff, nq, d_out, d_defer, br);
  COUNT_LAUNCH();
  return cudaGetLastError();
}

// the wave kernel, then the refilling kernel over the queries it handed on, then the scalar kernel over the
// queries with ambiguity symbols (both lists are empty for a batch of clean sequencer reads)
// ASCII flavour (launch_search_ascii): where the kernel reads the query bytes, writes the words it hands on, latches
struct AsciiQueries {
  const uint8_t* qbytes = nullptr;
  uint64_t* qwords = nullptr;
  unsigned long long* first_bad = nullptr;
};

template <int MODE, bool ASCII = false, bool STRAND = false>
static cudaError_t launch_search_wave(const IndexView& ix, const uint64_t* d_qwords, const uint64_t* d_qoff, uint64_t nq,
                                      void* d_out, uint32_t* d_defer, int sm_count, cudaStream_t s, uint32_t avg_len,
                                      ByteRange br, const AsciiQueries& a = AsciiQueries()) {
  // 6 x 256 threads/SM (40 registers, 8-16 bytes of spill) beat 5 x 256 (47 registers, none): 1.70 against 1.80 ms
  // per 10 M x 150-bp reads with a k = 13 seed table
  constexpr int TPB = 256, MINB = 6;
  cudaError_t e = cudaMemsetAsync(d_defer + nq + 2, 0, 8, s);  // count of the rest list, its ticket counter
  if (e != cudaSuccess) return e;
  auto kern = STRAND ? search_dna_strand_wave_kernel<MODE, TPB, MINB> : search_dna_wave_kernel<MODE, TPB, MINB, ASCII>;
  auto kern_rest = search_dna_pair_kernel<MODE, TPB, 4, true, true>;  // (64 registers: the list-driven flavour spills at 48)
  int per_sm = 0, per_sm_rest = 0;
  if ((e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, TPB, 0)) != cudaSuccess) return e;
  if ((e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm_rest, kern_rest, TPB, 0)) != cudaSuccess) return e;
  const uint64_t need_blocks = (nq * 4 + TPB - 1) / TPB;
  const unsigned grid = unsigned(std::max<uint64_t>(1, std::min<uint64_t>(uint64_t(sm_count) * std::max(1, per_sm), need_blocks)));
  const unsigned grid_rest = unsigned(std::max<uint64_t>(1, std::min<uint64_t>(uint64_t(sm_count) * std::max(1, per_sm_rest), need_blocks)));
  static const uint32_t ticket_env = [] {  // AWRY_B200_TICKET: fixed ticket size (experiments)
    if (const char* e = getenv("AWRY_B200_TICKET")) return uint32_t(std::min(1024l, std::max(8l, strtol(e, nullptr, 10)))) & ~7u;
    return 0u;
  }();
  // a ticket = 4 waves of 8 queries per warp; small batches get one wave per ticket so that every warp draws some
  // (tickets are multiples of 8: the strand flavour relies on waves that start at an even query)
  uint32_t ticket_sz = nq >= uint64_t(grid) * (TPB / 32) * 128 ? 32u : 8u;
  if (ticket_env) ticket_sz = ticket_env;
  e = launch_with_table_window(kern, grid, TPB, s, ix, ix, d_qwords, d_qoff, nq, d_out, d_defer, ticket_sz, br, a.qbytes,
                               a.qwords, a.first_bad);
  COUNT_LAUNCH();
  if (e != cudaSuccess) return e;
  uint32_t per_group = avg_len == 0 ? 2u : std::min(8u, std::max(1u, 200u / avg_len));
  e = launch_with_table_window(kern_rest, grid_rest, TPB, s, ix, ix, d_qwords, d_qoff, nq, d_out, d_defer, 8u * per_group, br);
  COUNT_LAUNCH();
  if (e != cudaSuccess) return e;
  search_scalar_kernel<0, MODE, true><<<unsigned(sm_count) * 2, 256, 0, s>>>(ix, d_qwords, d_qoff, nq, d_out, d_defer, br);
  COUNT_LAUNCH();
  return cudaGetLastError();
}

// the state-machine kernel: NS query slots per lane group, `per_sm` resident 256-thread blocks (register budget)
template <int MODE, int MINB, int NS, bool VFY = false>
static cudaError_t launch_search_pairx_b(const IndexView& ix, const uint64_t* d_qwords, const uint64_t* d_qoff,
                                         uint64_t nq, void* d_out, uint32_t* d_defer, int sm_count, cudaStream_t s,
                                         uint32_t avg_len, ByteRange br) {
  constexpr int TPB = 256;
  auto kern = search_dna_pairx_kernel<MODE, TPB, MINB, NS, VFY>;
  int per_sm = 0;
  cudaError_t e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, TPB, 0);
  if (e != cudaSuccess) return e;
  if (per_sm < 1) per_sm = 1;
  const uint64_t max_blocks = uint64_t(sm_count) * uint64_t(per_sm);
  const uint64_t need_blocks = (nq * 4 + uint64_t(TPB) * NS - 1) / (uint64_t(TPB) * NS);
  const unsigned grid = unsigned(std::max<uint64_t>(1, std::min(max_blocks, need_blocks)));
  static const uint32_t ticket_env = [] {  // AWRY_B200_TICKET: fixed ticket size (experiments)
    if (const char* e = getenv("AWRY_B200_TICKET")) return uint32_t(std::min(1024l, std::max(1l, strtol(e, nullptr, 10))));
    return 0u;
  }();
  // per-WARP ticket: one query per slot (8 groups x NS slots) for 150-bp reads, more for short queries; small
  // batches get small tickets so that every warp still draws several (see launch_search_pair_b)
  uint32_t per_slot = avg_len == 0 ? 2u : std::min(8u, std::max(1u, 200u / avg_len));
  per_slot = ticket_cap(per_slot, nq, uint64_t(grid) * (TPB / 4) * NS, avg_len);
  const uint32_t ticket_sz = ticket_env ? ticket_env : 8u * NS * per_slot;
  e = launch_with_table_window(kern, grid, TPB, s, ix, ix, d_qwords, d_qoff, nq, d_out, d_defer, ticket_sz, br);
  COUNT_LAUNCH();
  if (e != cudaSuccess) return e;
  search_scalar_kernel<0, MODE, true><<<unsigned(sm_count) * 2, 256, 0, s>>>(ix, d_qwords, d_qoff, nq, d_out, d_defer, br);
  COUNT_LAUNCH();
  return cudaGetLastError();
}

static int slots_default() {
  static const int d = [] {
    if (const char* e = getenv("AWRY_B200_SLOTS")) return std::max(0, std::min(4, atoi(e)));
    return 0;
  }();
  return d;
}

// With the text on the device one-row intervals are finished by comparing with it (see the kernels): count mode,
// and locate pass 1 for a gather pass 2 (the hit stored as its text position).
static bool finishes_in_text(const IndexView& ix, SearchOut mode, const SearchVariant& v) {
  return v.finish_in_text && ix.rtext != nullptr && ix.full_sa != nullptr &&
         (mode == OUT_COUNT_U64 || (mode == OUT_SP_CNT_U32 && v.locate_positions));
}

// Whether launch_search runs the nucleotide wave kernel: the default there (launch_search_mode -> launch_search_pair);
// the refilling kernel with the same step (awry_set_search_variant(80), or a residency) and the state-machine one
// (81-84, count only) stay selectable.
static bool runs_wave_kernel(const IndexView& ix, SearchOut mode, const SearchVariant& v) {
  return !ix.wide && ix.alphabet == 0 && ix.pair_blocks != nullptr && (v.lanes == 0 || v.lanes == 8) &&
         finishes_in_text(ix, mode, v) && v.slots < 0 && slots_default() == 0 && v.blocks_per_sm == 0;
}

static cudaError_t reset_defer(uint64_t nq, uint32_t* d_defer, cudaStream_t s) {
  if (nq >= (1ull << 32) - (1u << 24)) return cudaErrorInvalidValue;  // 32-bit ticket counter
  cudaError_t e = cudaMemsetAsync(d_defer, 0, 4, s);                  // deferred-query count
  if (e != cudaSuccess) return e;
  return cudaMemsetAsync(d_defer + nq + 1, 0, 4, s);                  // ticket counter
}

template <int MODE>
static cudaError_t launch_search_pair(const IndexView& ix, const uint64_t* d_qwords, const uint64_t* d_qoff,
                                      uint64_t nq, void* d_out, uint32_t* d_defer, const SearchVariant& v,
                                      int sm_count, cudaStream_t s) {
  cudaError_t e = reset_defer(nq, d_defer, s);
  if (e != cudaSuccess) return e;
  const ByteRange br{v.b_lo, v.b_hi};
  const int slots = v.slots >= 0 ? v.slots : slots_default();
  const bool in_text = finishes_in_text(ix, SearchOut(MODE), v);
  if (runs_wave_kernel(ix, SearchOut(MODE), v)) {
    if (MODE == OUT_COUNT_U64) return launch_search_wave<OUT_COUNT_U64>(ix, d_qwords, d_qoff, nq, d_out, d_defer, sm_count, s, v.avg_len, br);
    if (MODE == OUT_SP_CNT_U32) return launch_search_wave<OUT_SP_CNT_U32>(ix, d_qwords, d_qoff, nq, d_out, d_defer, sm_count, s, v.avg_len, br);
  }
  if (MODE == OUT_SP_CNT_U32 && in_text)
    return launch_search_pair_b<OUT_SP_CNT_U32, 5, true>(ix, d_qwords, d_qoff, nq, d_out, d_defer, 0, sm_count, s, v.avg_len, br);
  // count mode with the text on the device: finish one-row intervals by comparing with the text (see the kernel)
  if (MODE == OUT_COUNT_U64 && in_text) {
    if (slots == 1) return launch_search_pairx_b<OUT_COUNT_U64, 8, 1, true>(ix, d_qwords, d_qoff, nq, d_out, d_defer, sm_count, s, v.avg_len, br);
    if (slots == 2) return launch_search_pairx_b<OUT_COUNT_U64, 5, 2, true>(ix, d_qwords, d_qoff, nq, d_out, d_defer, sm_count, s, v.avg_len, br);
    if (slots == 3) return launch_search_pairx_b<OUT_COUNT_U64, 6, 1, true>(ix, d_qwords, d_qoff, nq, d_out, d_defer, sm_count, s, v.avg_len, br);
    if (slots == 4) return launch_search_pairx_b<OUT_COUNT_U64, 4, 2, true>(ix, d_qwords, d_qoff, nq, d_out, d_defer, sm_count, s, v.avg_len, br);
    switch (v.blocks_per_sm) {
      case 4: return launch_search_pair_b<OUT_COUNT_U64, 4, true>(ix, d_qwords, d_qoff, nq, d_out, d_defer, 0, sm_count, s, v.avg_len, br);
      // 5 x 256 threads/SM: 48 registers hold the comparison without spills (at 6 x 256 = 40 registers two values
      // live in local memory and a launch takes 3.6 instead of 2.5 ms, profiles/r02_s8_text_finish_probe.log)
      case 6: return launch_search_pair_b<OUT_COUNT_U64, 6, true>(ix, d_qwords, d_qoff, nq, d_out, d_defer, 0, sm_count, s, v.avg_len, br);
      case 8: return launch_search_pair_b<OUT_COUNT_U64, 8, true>(ix, d_qwords, d_qoff, nq, d_out, d_defer, 0, sm_count, s, v.avg_len, br);
      default: return launch_search_pair_b<OUT_COUNT_U64, 5, true>(ix, d_qwords, d_qoff, nq, d_out, d_defer, 0, sm_count, s, v.avg_len, br);
    }
  }
  // the state-machine variant, kept selectable for A/B runs with its two best residencies (see the kernel)
  if (slots == 1 || slots == 3) return launch_search_pairx_b<MODE, 8, 1>(ix, d_qwords, d_qoff, nq, d_out, d_defer, sm_count, s, v.avg_len, br);
  if (slots == 2 || slots == 4) return launch_search_pairx_b<MODE, 5, 2>(ix, d_qwords, d_qoff, nq, d_out, d_defer, sm_count, s, v.avg_len, br);
  switch (v.blocks_per_sm) {
    case 4: return launch_search_pair_b<MODE, 4>(ix, d_qwords, d_qoff, nq, d_out, d_defer, 0, sm_count, s, v.avg_len, ByteRange{v.b_lo, v.b_hi});
    // 8 x 256 threads/SM (32 registers) is fastest for an isolated launch (16.2 vs 16.6-17.0 ms), 6 x 256
    // (40 registers) for launches back to back, where the part sits at its power cap (18.1 vs 18.7 ms,
    // profiles/r01_s31_sustained_ab.log): batches arrive back to back in production, so 6 is the default
    case 8: return launch_search_pair_b<MODE, 8>(ix, d_qwords, d_qoff, nq, d_out, d_defer, 0, sm_count, s, v.avg_len, ByteRange{v.b_lo, v.b_hi});
    case 0:
    case 6: return launch_search_pair_b<MODE, 6>(ix, d_qwords, d_qoff, nq, d_out, d_defer, 0, sm_count, s, v.avg_len, ByteRange{v.b_lo, v.b_hi});
    default: return launch_search_pair_b<MODE, 4>(ix, d_qwords, d_qoff, nq, d_out, d_defer, v.blocks_per_sm, sm_count, s, v.avg_len, ByteRange{v.b_lo, v.b_hi});
  }
}

// ---- amino kernel: 4 lanes per query, one 128-B block (4 x LDG.256) per symbol ----
// Same shape as the nucleotide pair kernel: the query (8-bit symbols) is staged in a 16-word
// shared-memory ring with one aligned read, groups refill in-loop, the warp leaves by vote and
// the rank reduction uses full-mask shuffles.  Slices 0/1 hold the planes of rows 0-31 / 32-63.
// VFY (count, and locate pass 1 for a gather pass 2; needs ix.full_sa and ix.rtext): as in the nucleotide kernels, a
// one-row interval with at least AMINO_VERIFY_MIN_LEFT symbols left is finished by reading SA[row] and comparing
// the rest of the query with the text (one byte per symbol) -- two dependent loads instead of `left`.
constexpr uint32_t AMINO_VERIFY_MIN_LEFT = 3;

// LIST: the peptides to run are the ones search_amino_wave_kernel handed on; `ticket` is then the counter behind
// their count (defer + nq + 3: the count sits one word in front of it, the numbers one word behind it).
template <int MODE, int TPB, int MINB, bool VFY = false, bool LIST = false>
__global__ void __launch_bounds__(TPB, MINB)
    search_amino_kernel(IndexView ix, const uint64_t* __restrict__ qwords,
                        const uint64_t* __restrict__ qoff, uint64_t nq, void* __restrict__ out,
                        uint32_t* __restrict__ ticket, uint32_t ticket_sz, ByteRange br) {
  constexpr int LANES = 4;
  constexpr uint32_t NONE = 0xffffffffu, FULL = 0xffffffffu;
  __shared__ uint64_t s_q[TPB / LANES][16];  // 128 symbols
  const uint32_t sub = threadIdx.x & 3;
  const uint32_t gbase = (threadIdx.x & 31) - sub;
  const uint32_t gmask = 0xfu << gbase;
  uint64_t* const ring = s_q[threadIdx.x / LANES];
  const uint32_t* const rest = LIST ? ticket - 1 : ticket;  // (LIST only)
  const uint32_t nq32 = LIST ? rest[0] : uint32_t(nq);
  uint32_t q = 0, q_end = 0;  // dynamic hand-out of ticket_sz queries at a time (see the pair kernel)
  bool more = true;
  uint32_t cur = NONE;
  uint32_t sp = 1, ep = 0, left = 0, len = 0;
  uint32_t ubase = 0, wlim = 8;

  for (;;) {
    if (left == 0 || sp > ep) {
      if (cur != NONE && sub == 0) store_result<MODE>(out, cur, sp, ep);
      cur = NONE;
      left = 0;
      if (q == q_end && more) {
        uint32_t t = 0;
        if (sub == 0) t = atomicAdd(ticket, ticket_sz);
        t = __shfl_sync(gmask, t, gbase);
        more = t < nq32;
        q = more ? t : 0u;
        q_end = more ? (nq32 - t < ticket_sz ? nq32 : t + ticket_sz) : 0u;
      }
      if (q < q_end) {
        cur = LIST ? rest[2 + q] : q;
        q++;
        uint64_t ov = qoff[cur + (sub & 1)];
        uint64_t o0 = __shfl_sync(gmask, ov, gbase), o1 = __shfl_sync(gmask, ov, gbase + 1);
        len = checked_len(o0, o1, br);
        sp = 1;
        ep = 0;
        if (len != 0) {
          ubase = 4 * (cur + uint32_t(o0 >> 5));
          const uint32_t nwords = (len + 7) >> 3;
          __syncwarp(gmask);
          if (4 * sub < nwords) {
            AWRY_CHK_QWORDS(ubase + 4 * sub, br, nq, 5);
            u32x8 t = ldg256(qwords + ubase + 4 * sub);
#pragma unroll
            for (int j = 0; j < 4; j++) ring[4 * sub + j] = uint64_t(t.v[2 * j]) | (uint64_t(t.v[2 * j + 1]) << 32);
          }
          __syncwarp(gmask);
          wlim = 8;
          const uint32_t k = ix.kmer_len;
          const uint64_t w = ring[0];
          bool seeded = false;
          if (k != 0 && len >= k) {  // k <= 8: inside word 0
            uint64_t idx = 0, mult = 1;
            bool ok = true;
#pragma unroll 1
            for (uint32_t j = 0; j < k; j++) {
              uint32_t c = uint32_t(w >> (8 * j)) & 0xffu;
              ok &= (c != uint32_t(AMINO_X)) & (c != uint32_t(AMINO_SENTINEL));
              idx += uint64_t(c == 21 ? 19 : c - 1) * mult;
              mult *= 20;
            }
            if (ok) {
              AWRY_CHK(idx < ix.n_table);
      uint2 r = __ldg(ix.table + idx);
              sp = r.x;
              ep = r.y;
              left = len - k;
              seeded = true;
            }
          }
          if (!seeded) {
            uint32_t c = uint32_t(w) & 0xffu;
            if (c != uint32_t(AMINO_SENTINEL)) {
              sp = ix.c_lo[c];
              ep = ix.c_hi[c];
              left = len - 1;
            }
          }
        }
      }
    }
    if (__all_sync(FULL, cur == NONE && q == q_end && !more)) break;

    bool active = left != 0 && sp <= ep;
    const uint32_t pos = len - left;
    if (active && (pos >> 3) >= wlim) {  // long query: bring in words [wlim+8, wlim+16)
      __syncwarp(gmask);
      if (sub < 2) {
        AWRY_CHK_QWORDS(ubase + wlim + 8 + 4 * sub, br, nq, 5);
        u32x8 t = ldg256(qwords + ubase + wlim + 8 + 4 * sub);
#pragma unroll
        for (int j = 0; j < 4; j++)
          ring[(wlim + 8 + 4 * sub + j) & 15] = uint64_t(t.v[2 * j]) | (uint64_t(t.v[2 * j + 1]) << 32);
      }
      __syncwarp(gmask);
      wlim += 8;
    }
    const uint32_t c = uint32_t(ring[(pos >> 3) & 15] >> (8 * (pos & 7))) & 0xffu;
    if (active && (c == uint32_t(AMINO_SENTINEL) || c > 21)) {  // rejected by the prepass; stay defined
      sp = 1;
      ep = 0;
      active = false;
    }
    const uint32_t pa = sp - 1, pb = ep;
    uint32_t ra = 0, rb = 0;
    if (active) {
      const uint32_t ba = pa >> 6, bb = pb >> 6;
      const int na = int(pa & 63) + 1 - int(32 * sub), nb = int(pb & 63) + 1 - int(32 * sub);
      AWRY_CHK(uint64_t(ba) * AMINO_BLOCK_UINT4 + 7 < ix.n_blocks_u4 && uint64_t(bb) * AMINO_BLOCK_UINT4 + 7 < ix.n_blocks_u4);
      u32x8 x = ldg256(ix.blocks + size_t(ba) * AMINO_BLOCK_UINT4 + 2 * sub);
      AminoSlice s = amino_slice(x, sub, c);
      ra = __popc(s.match & low_mask(na)) + s.count;
      if (bb != ba) {
        x = ldg256(ix.blocks + size_t(bb) * AMINO_BLOCK_UINT4 + 2 * sub);
        s = amino_slice(x, sub, c);
      }
      rb = __popc(s.match & low_mask(nb)) + s.count;
    }
    ra += __shfl_xor_sync(FULL, ra, 1);
    rb += __shfl_xor_sync(FULL, rb, 1);
    ra += __shfl_xor_sync(FULL, ra, 2);
    rb += __shfl_xor_sync(FULL, rb, 2);
    if (active) {
      const uint32_t base = ix.c_lo[c];
      sp = base + ra;
      ep = base + rb - 1;
      left--;
    }
    if (VFY) {
      // (the unconsumed symbols must all be in the ring: always, for queries of <= 128 symbols)
      if (active && sp == ep && left >= AMINO_VERIFY_MIN_LEFT && ((len + 7) >> 3) <= wlim + 8) {
        AWRY_CHK(sp < ix.n_full_sa);
        const uint32_t p = __ldg(ix.full_sa + sp);  // the matched suffix stands at text[p ..]
        bool ok = p >= left;                          // else the rest of the query would start before the text
        if (ok) {
          const uint32_t done = len - left;
          const uint32_t rb0 = ix.bwt_len - p - done;  // reversed-text index of search-order symbol 0
          const uint32_t s_first = (rb0 + done) >> 5, s_last = (rb0 + len - 1) >> 5;  // 32-B sectors = 32 symbols
          uint32_t bad = 0;
          for (uint32_t sec = s_first + sub; sec <= s_last; sec += 4) {
            AWRY_CHK(uint64_t(sec) * 32 + 31 < ix.n_rtext);
            const u32x8 t = ldg256(ix.rtext + size_t(sec) * 32);
            bad |= text_sector_mismatch8(t, ring, sec, rb0, done, len);
          }
          ok = !__any_sync(gmask, bad != 0u);
        }
        if (sub == 0) {
          if (MODE == OUT_COUNT_U64)
            reinterpret_cast<uint64_t*>(out)[cur] = ok ? 1ull : 0ull;
          else
            reinterpret_cast<uint2*>(out)[cur] = ok ? make_uint2(p - left, CNT_AT_TEXT_POS) : make_uint2(1u, 0u);
        }
        cur = NONE;
        left = 0;
      }
    }
  }
}

// ---- protein wave kernel: search_dna_wave_kernel's structure on the 64-row / 128-B protein blocks ----
// A warp takes 8 peptides at a time through the phases together: offsets, packed symbols (8 bits each: the
// 16-word ring holds 128), seed entry, one-symbol steps until every interval of the wave is one row wide (or
// empty, or used up), SA element, text (one byte per symbol).  Peptides longer than the ring, or still wide after
// AMINO_WAVE_MAX_STEPS steps, go to the `rest` list and are searched by search_amino_kernel<VFY, LIST>.
constexpr int AMINO_WAVE_MAX_STEPS = 8;

template <int MODE, int TPB, int MINB>
__global__ void __launch_bounds__(TPB, MINB)
    search_amino_wave_kernel(IndexView ix, const uint64_t* __restrict__ qwords, const uint64_t* __restrict__ qoff,
                             uint64_t nq, void* __restrict__ out, uint32_t* __restrict__ defer, uint32_t ticket_sz,
                             ByteRange br) {
  constexpr uint32_t FULL = 0xffffffffu;
  enum : uint32_t { W_NONE = 0, W_RUN = 1, W_EMPTY = 2 };
  __shared__ uint64_t s_q[TPB / 4][16];
  const uint32_t lane = threadIdx.x & 31, sub = lane & 3, gbase = lane - sub, gmask = 0xfu << gbase, grp = lane >> 2;
  uint64_t* const ring = s_q[threadIdx.x >> 2];
  const uint32_t nq32 = uint32_t(nq);
  uint32_t* const ticket = defer + nq + 1;
  uint32_t* const rest = defer + nq + 2;  // rest[0] = count, rest[2 ..] = query numbers
  uint32_t pn = 0, pe = 0;
  uint32_t ahead = 0;  // the warp's next ticket, drawn one ahead (lane 0)
  if (lane == 0) ahead = atomicAdd(ticket, ticket_sz);
  for (;;) {
    if (pn == pe) {  // warp-uniform
      uint32_t t = ahead;
      if (lane == 0 && t < nq32) ahead = atomicAdd(ticket, ticket_sz);
      t = __shfl_sync(FULL, t, 0);
      if (t >= nq32) break;
      pn = t;
      pe = t + (nq32 - t < ticket_sz ? nq32 - t : ticket_sz);
    }
    const uint32_t q = pn + grp;
    uint32_t st = q < pe ? W_RUN : W_NONE;
    pn = pe - pn > 8u ? pn + 8u : pe;

    // ---- offsets
    uint64_t ov = 0;
    if (st == W_RUN) ov = __ldg(qoff + q + (sub & 1));
    const uint64_t o0 = __shfl_sync(FULL, ov, gbase), o1 = __shfl_sync(FULL, ov, gbase + 1);
    const uint32_t len = st == W_RUN ? checked_len(o0, o1, br) : 0u;
    if (st == W_RUN && len == 0) st = W_EMPTY;
    const uint32_t nwords = (len + 7) >> 3;
    if (st == W_RUN && nwords > 16) {  // longer than the ring
      if (sub == 0) rest[2 + atomicAdd(rest, 1u)] = q;
      st = W_NONE;
    }
    // ---- packed symbols -> ring
    __syncwarp();  // the previous wave's ring reads are done
    if (st == W_RUN && 4 * sub < nwords) {
      const uint32_t ubase = 4 * (q + uint32_t(o0 >> 5));
      AWRY_CHK_QWORDS(ubase + 4 * sub, br, nq, 5);
      const u32x8 t = ldg256(qwords + ubase + 4 * sub);
#pragma unroll
      for (int j = 0; j < 4; j++) ring[4 * sub + j] = uint64_t(t.v[2 * j]) | (uint64_t(t.v[2 * j + 1]) << 32);
    }
    __syncwarp();
    // ---- seed
    uint32_t sp = 1, ep = 0, left = 0;
    if (st == W_RUN) {
      const uint32_t k = ix.kmer_len;
      const uint64_t w = ring[0];
      bool seeded = false;
      if (k != 0 && len >= k) {  // k <= 8: inside word 0
        uint64_t idx = 0, mult = 1;
        bool ok = true;
#pragma unroll 1
        for (uint32_t j = 0; j < k; j++) {
          const uint32_t c = uint32_t(w >> (8 * j)) & 0xffu;
          ok &= (c != uint32_t(AMINO_X)) & (c != uint32_t(AMINO_SENTINEL));
          idx += uint64_t(c == 21 ? 19 : c - 1) * mult;
          mult *= 20;
        }
        if (ok) {
          AWRY_CHK(idx < ix.n_table);
          const uint2 r = __ldg(ix.table + idx);
          sp = r.x;
          ep = r.y;
          left = len - k;
          seeded = true;
        }
      }
      if (!seeded) {
        const uint32_t c = uint32_t(w) & 0xffu;
        if (c != uint32_t(AMINO_SENTINEL) && c <= 21) {
          sp = ix.c_lo[c];
          ep = ix.c_hi[c];
          left = len - 1;
        }
      }
    }
    // ---- steps
#pragma unroll 1
    for (int it = 0; it <= AMINO_WAVE_MAX_STEPS; it++) {
      bool active = st == W_RUN && left != 0 && sp <= ep && !(sp == ep && left >= AMINO_VERIFY_MIN_LEFT);
      if (!__any_sync(FULL, active)) break;
      if (it == AMINO_WAVE_MAX_STEPS) {  // still wide: handed on
        if (active) {
          if (sub == 0) rest[2 + atomicAdd(rest, 1u)] = q;
          st = W_NONE;
        }
        break;
      }
      const uint32_t pos = len - left;
      const uint32_t c = uint32_t(ring[(pos >> 3) & 15] >> (8 * (pos & 7))) & 0xffu;
      if (active && (c == uint32_t(AMINO_SENTINEL) || c > 21)) {  // rejected by the prepass; stay defined
        sp = 1;
        ep = 0;
        active = false;
      }
      const uint32_t pa = sp - 1, pb = ep;
      uint32_t ra = 0, rb = 0;
      if (active) {
        const uint32_t ba = pa >> 6, bb = pb >> 6;
        AWRY_CHK(uint64_t(ba) * AMINO_BLOCK_UINT4 + 7 < ix.n_blocks_u4 && uint64_t(bb) * AMINO_BLOCK_UINT4 + 7 < ix.n_blocks_u4);
        const u32x8 x = ldg256(ix.blocks + size_t(ba) * AMINO_BLOCK_UINT4 + 2 * sub);
        u32x8 y = x;
        if (bb != ba) y = ldg256(ix.blocks + size_t(bb) * AMINO_BLOCK_UINT4 + 2 * sub);  // both reads before either use
        AminoSlice s = amino_slice(x, sub, c);
        ra = __popc(s.match & low_mask(int(pa & 63) + 1 - int(32 * sub))) + s.count;
        if (bb != ba) s = amino_slice(y, sub, c);
        rb = __popc(s.match & low_mask(int(pb & 63) + 1 - int(32 * sub))) + s.count;
      }
      ra += __shfl_xor_sync(FULL, ra, 1);
      rb += __shfl_xor_sync(FULL, rb, 1);
      ra += __shfl_xor_sync(FULL, ra, 2);
      rb += __shfl_xor_sync(FULL, rb, 2);
      if (active) {
        const uint32_t base = ix.c_lo[c];
        sp = base + ra;
        ep = base + rb - 1;
        left--;
      }
    }
    // ---- finish in the text
    const bool need = st == W_RUN && left != 0 && sp <= ep;  // (then sp == ep and left >= AMINO_VERIFY_MIN_LEFT)
    uint32_t p = 0;
    if (need) {
      AWRY_CHK(sp < ix.n_full_sa);
      p = __ldg(ix.full_sa + sp);
    }
    bool ok = need && p >= left;
    uint32_t bad = 0;
    if (ok) {
      const uint32_t done = len - left;
      const uint32_t rb0 = ix.bwt_len - p - done;
      const uint32_t s_first = (rb0 + done) >> 5, s_last = (rb0 + len - 1) >> 5;  // 32-B sectors = 32 symbols
      for (uint32_t sec = s_first + sub; sec <= s_last; sec += 4) {
        AWRY_CHK(uint64_t(sec) * 32 + 31 < ix.n_rtext);
        const u32x8 t = ldg256(ix.rtext + size_t(sec) * 32);
        bad |= text_sector_mismatch8(t, ring, sec, rb0, done, len);
      }
    }
    const uint32_t bad_groups = __ballot_sync(FULL, bad != 0);
    ok = ok && (bad_groups & gmask) == 0;
    // ---- results
    if (sub == 0) {
      if (st == W_EMPTY) {
        store_result<MODE>(out, q, 1u, 0u);
      } else if (st == W_RUN && !need) {
        store_result<MODE>(out, q, sp, ep);
      } else if (st == W_RUN) {
        if (MODE == OUT_COUNT_U64)
          reinterpret_cast<uint64_t*>(out)[q] = ok ? 1ull : 0ull;
        else
          reinterpret_cast<uint2*>(out)[q] = ok ? make_uint2(p - left, CNT_AT_TEXT_POS) : make_uint2(1u, 0u);
      }
    }
  }
}

template <int MODE>
static cudaError_t launch_search_amino(const IndexView& ix, const uint64_t* d_qwords, const uint64_t* d_qoff,
                                       uint64_t nq, void* d_out, uint32_t* d_ticket, const SearchVariant& v,
                                       int sm_count, cudaStream_t s) {
  if (nq >= (1ull << 32) - (1u << 24)) return cudaErrorInvalidValue;  // 32-bit ticket counter
  constexpr int TPB = 256;
  const bool in_text = v.finish_in_text && ix.rtext != nullptr && ix.full_sa != nullptr &&
                       (MODE == OUT_COUNT_U64 || (MODE == OUT_SP_CNT_U32 && v.locate_positions));
  auto kern = search_amino_kernel<MODE, TPB, 6>;
  if (in_text && MODE != OUT_RANGE_U64) kern = search_amino_kernel<MODE == OUT_RANGE_U64 ? OUT_COUNT_U64 : MODE, TPB, 6, true>;
  int per_sm = 0;
  cudaError_t e = cudaMemsetAsync(d_ticket, 0, 4, s);
  if (e != cudaSuccess) return e;
  if (in_text && MODE != OUT_RANGE_U64 && v.slots < 0 && v.blocks_per_sm == 0) {
    // default with the text on the device: the wave kernel, then the refilling kernel over what it handed on
    // (awry_set_search_variant(80) keeps the refilling kernel for everything)
    constexpr int M = MODE == OUT_RANGE_U64 ? OUT_COUNT_U64 : MODE;
    uint32_t* const d_defer = d_ticket;
    if ((e = cudaMemsetAsync(d_defer + nq + 1, 0, 12, s)) != cudaSuccess) return e;  // ticket, rest count, rest ticket
    auto wave = search_amino_wave_kernel<M, TPB, 6>;
    auto rest = search_amino_kernel<M, TPB, 6, true, true>;
    int per_w = 0, per_r = 0;
    if ((e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_w, wave, TPB, 0)) != cudaSuccess) return e;
    if ((e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_r, rest, TPB, 0)) != cudaSuccess) return e;
    const uint64_t need = (nq * 4 + TPB - 1) / TPB;
    const unsigned grid_w = unsigned(std::max<uint64_t>(1, std::min<uint64_t>(uint64_t(sm_count) * std::max(1, per_w), need)));
    const unsigned grid_r = unsigned(std::max<uint64_t>(1, std::min<uint64_t>(uint64_t(sm_count) * std::max(1, per_r), need)));
    const uint32_t wave_ticket = nq >= uint64_t(grid_w) * (TPB / 32) * 128 ? 32u : 8u;
    const ByteRange br{v.b_lo, v.b_hi};
    e = launch_with_table_window(wave, grid_w, TPB, s, ix, ix, d_qwords, d_qoff, nq, d_out, d_defer, wave_ticket, br);
    COUNT_LAUNCH();
    if (e != cudaSuccess) return e;
    e = launch_with_table_window(rest, grid_r, TPB, s, ix, ix, d_qwords, d_qoff, nq, d_out, d_defer + nq + 3,
                                 ticket_size(v.avg_len), br);
    COUNT_LAUNCH();
    return e;
  }
  e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, TPB, 0);
  if (e != cudaSuccess) return e;
  if (per_sm < 1) per_sm = 1;
  if (v.blocks_per_sm > 0 && v.blocks_per_sm < per_sm) per_sm = v.blocks_per_sm;
  uint64_t max_blocks = uint64_t(sm_count) * uint64_t(per_sm);
  uint64_t need_blocks = (nq * 4 + TPB - 1) / TPB;
  unsigned grid = unsigned(std::max<uint64_t>(1, std::min(max_blocks, need_blocks)));
  // (no batch-size cap here: the hand-out is per lane GROUP, and 12-residue peptides at 3.7 G/s with tickets
  // of 2 would be 1.8 G same-address atomics/s, far above what one counter retires)
  e = launch_with_table_window(kern, grid, TPB, s, ix, ix, d_qwords, d_qoff, nq, d_out, d_ticket, ticket_size(v.avg_len),
                               ByteRange{v.b_lo, v.b_hi});
  COUNT_LAUNCH();
  return e;
}

template <int MODE>
static cudaError_t launch_search_mode(const IndexView& ix, const uint64_t* d_qwords, const uint64_t* d_qoff,
                                      uint64_t nq, void* d_out, uint32_t* d_defer, const SearchVariant& v,
                                      int sm_count, cudaStream_t s) {
  if (ix.alphabet == 0 && v.lanes != -1) {
    if (ix.pair_blocks != nullptr && (v.lanes == 0 || v.lanes == 8))
      return launch_search_pair<MODE>(ix, d_qwords, d_qoff, nq, d_out, d_defer, v, sm_count, s);
    switch (v.lanes) {
      case 1: return launch_search_dna<1, MODE>(ix, d_qwords, d_qoff, nq, d_out, v, sm_count, s);
      case 4: return launch_search_dna<4, MODE>(ix, d_qwords, d_qoff, nq, d_out, v, sm_count, s);
      default: return launch_search_dna<2, MODE>(ix, d_qwords, d_qoff, nq, d_out, v, sm_count, s);
    }
  }
  if (ix.alphabet == 1 && v.lanes != -1)
    return launch_search_amino<MODE>(ix, d_qwords, d_qoff, nq, d_out, d_defer, v, sm_count, s);
  // lanes == -1: the scalar kernels, kept for cross-checking
  int per_sm = 8;
  uint64_t need_blocks = (nq + 255) / 256;
  unsigned grid = unsigned(std::max<uint64_t>(1, std::min<uint64_t>(uint64_t(sm_count) * per_sm, need_blocks)));
  if (ix.alphabet == 0)
    search_scalar_kernel<0, MODE, false><<<grid, 256, 0, s>>>(ix, d_qwords, d_qoff, nq, d_out, nullptr, ByteRange{v.b_lo, v.b_hi});
  else
    search_scalar_kernel<1, MODE, false><<<grid, 256, 0, s>>>(ix, d_qwords, d_qoff, nq, d_out, nullptr, ByteRange{v.b_lo, v.b_hi});
  COUNT_LAUNCH();
  return cudaGetLastError();
}

bool search_packs_ascii(const IndexView& ix, SearchOut mode, const SearchVariant& v) {
  const char* e = getenv("AWRY_B200_ASCII_WAVE");  // read per call: "0" keeps launch_pack + launch_search (A/B runs, tests)
  return !(e && e[0] == '0') && runs_wave_kernel(ix, mode, v);
}

bool search_strands_ascii(const IndexView& ix, SearchOut mode, const SearchVariant& v) {
  const char* e = getenv("AWRY_B200_STRAND_WAVE");  // read per call: "0" keeps the generic route (A/B runs, tests)
  return !(e && e[0] == '0') && search_packs_ascii(ix, mode, v);
}

cudaError_t launch_search_ascii(const IndexView& ix, const uint8_t* d_qbytes, const uint64_t* d_qoff, uint64_t nq,
                                uint64_t* d_qwords, unsigned long long* d_first_bad, SearchOut mode, void* d_out,
                                uint32_t* d_defer, const SearchVariant& v, int sm_count, cudaStream_t s, bool strands) {
  if (nq == 0) return cudaSuccess;
  if (!runs_wave_kernel(ix, mode, v) || (strands && (nq & 1))) return cudaErrorInvalidValue;
  cudaError_t e = reset_defer(nq, d_defer, s);
  if (e != cudaSuccess) return e;
  const ByteRange br{v.b_lo, v.b_hi};
  AsciiQueries a;
  a.qbytes = d_qbytes;
  a.qwords = d_qwords;
  a.first_bad = d_first_bad;
  if (strands) {
    if (mode == OUT_COUNT_U64)
      return launch_search_wave<OUT_COUNT_U64, true, true>(ix, d_qwords, d_qoff, nq, d_out, d_defer, sm_count, s, v.avg_len, br, a);
    return launch_search_wave<OUT_SP_CNT_U32, true, true>(ix, d_qwords, d_qoff, nq, d_out, d_defer, sm_count, s, v.avg_len, br, a);
  }
  if (mode == OUT_COUNT_U64)
    return launch_search_wave<OUT_COUNT_U64, true>(ix, d_qwords, d_qoff, nq, d_out, d_defer, sm_count, s, v.avg_len, br, a);
  return launch_search_wave<OUT_SP_CNT_U32, true>(ix, d_qwords, d_qoff, nq, d_out, d_defer, sm_count, s, v.avg_len, br, a);
}

cudaError_t launch_search(const IndexView& ix, const uint64_t* d_qwords, const uint64_t* d_qoff,
                          uint64_t nq, SearchOut mode, void* d_out, uint32_t* d_defer,
                          const SearchVariant& v, int sm_count, cudaStream_t s) {
  if (nq == 0) return cudaSuccess;
  if (ix.wide) return launch_search_wide(*ix.wide, d_qwords, d_qoff, nq, mode, d_out, d_defer, v, sm_count, s);
  switch (mode) {
    case OUT_COUNT_U64: return launch_search_mode<OUT_COUNT_U64>(ix, d_qwords, d_qoff, nq, d_out, d_defer, v, sm_count, s);
    case OUT_RANGE_U64: return launch_search_mode<OUT_RANGE_U64>(ix, d_qwords, d_qoff, nq, d_out, d_defer, v, sm_count, s);
    default: return launch_search_mode<OUT_SP_CNT_U32>(ix, d_qwords, d_qoff, nq, d_out, d_defer, v, sm_count, s);
  }
}

}  // namespace awry
