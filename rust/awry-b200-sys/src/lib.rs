//! Raw bindings: one `extern "C"` item per declaration of include/awry_b200.h.
#![allow(non_camel_case_types)]
use std::os::raw::{c_char, c_int, c_void};

#[repr(C)]
pub struct awry_index {
    _private: [u8; 0],
}

#[repr(C)]
#[derive(Clone, Copy, Debug, Default, PartialEq, Eq)]
pub struct awry_range {
    pub start_ptr: u64,
    pub end_ptr: u64,
}

#[repr(C)]
#[derive(Clone, Copy, Debug, Default, PartialEq, Eq, PartialOrd, Ord)]
pub struct awry_hit {
    pub seq_idx: u64,
    pub local_pos: u64,
}

pub const AWRY_METRIC_HAMMING: u32 = 0;
pub const AWRY_METRIC_EDIT: u32 = 1;

/// one edit operation of an alignment (include/awry_b200.h: awry_edit_op, 12 bytes)
#[repr(C)]
#[derive(Clone, Copy, Debug, Default, PartialEq, Eq)]
pub struct awry_edit_op {
    pub qpos: u32,
    pub tpos: u32,
    pub op: u8,
    pub query_sym: u8,
    pub text_sym: u8,
    pub pad: u8,
}

/// the alignment of one located hit (include/awry_b200.h: awry_alignment, 44 bytes)
#[repr(C)]
#[derive(Clone, Copy, Debug, Default, PartialEq, Eq)]
pub struct awry_alignment {
    pub text_len: u32,
    pub distance: u8,
    pub n_ops: u8,
    pub pad: [u8; 2],
    pub ops: [awry_edit_op; 3],
}

pub const AWRY_MAP_UNMAPPED: u8 = 1;
pub const AWRY_MAP_REFUSED: u8 = 2;

/// the best locus of one read (include/awry_b200.h: awry_mapping, 32 bytes); hit is (~0, ~0) when unmapped
#[repr(C)]
#[derive(Clone, Copy, Debug, Default, PartialEq, Eq)]
pub struct awry_mapping {
    pub hit: awry_hit,
    pub n_best: u32,
    pub n_second: u32,
    pub distance: u8,
    pub strand: u8,
    pub mapq: u8,
    pub flags: u8,
    pub pad: u32,
}

#[repr(C)]
#[derive(Clone, Copy)]
pub struct awry_info {
    pub version: u64,
    pub sa_ratio: u64,
    pub bwt_len: u64,
    pub alphabet: u32,
    pub kmer_len: u32,
    pub n_prefix_sums: u32,
    pub n_devices: u32,
    pub prefix_sums: [u64; 23],
    pub n_sequences: u64,
    pub device_bytes_blocks: u64,
    pub device_bytes_sa: u64,
    pub device_bytes_table: u64,
    pub device_bytes_pair: u64,
    pub device_bytes_full_sa: u64,
    pub device_bytes_lean_sa: u64,
    pub devices: [i32; 16],
    pub row_pointer_bits: u32,
    pub lean_sa_ratio: u32,
    pub device_bytes_text: u64,
}

#[repr(C)]
pub struct awry_parts {
    pub alphabet: u32,
    pub kmer_len: u32,
    pub sa_ratio: u64,
    pub bwt_len: u64,
    pub version: u64,
    pub blocks: *const u64,
    pub prefix_sums: *const u64,
    pub sa_words: *const u64,
    pub seq_starts: *const u64,
    pub headers: *const *const c_char,
    pub n_sequences: u64,
}

/// FmBuildArgs (fm_index.rs:78-96), the fields that mean something without libsufr
#[repr(C)]
pub struct awry_build_args {
    pub input_file_src: *const c_char,
    pub output_file_src: *const c_char,
    pub alphabet: u32,
    pub lookup_table_kmer_len: u32,
    pub suffix_array_compression_ratio: u64,
    pub device: i32,
}

/// awry_profile: per-kernel accounting kept by the library
#[repr(C)]
#[derive(Clone, Copy, Debug, Default)]
pub struct awry_profile {
    pub launches: u64,
    pub search_launches: u64,
    pub search_ms: f64,
    pub walk_launches: u64,
    pub walk_ms: f64,
    pub pack_launches: u64,
    pub pack_ms: f64,
    pub h2d_bytes: u64,
    pub d2h_bytes: u64,
}

pub const AWRY_OK: c_int = 0;
pub const AWRY_ERR_IO: c_int = -2;
pub const AWRY_ERR_INVALID_QUERY: c_int = -5;
pub const AWRY_LOCATE_BWT_ORDER: u32 = 0;
pub const AWRY_LOCATE_SORTED: u32 = 1;

extern "C" {
    pub fn awry_index_load(path: *const c_char, devices: *const c_int, n_dev: c_int, out: *mut *mut awry_index) -> c_int;
    pub fn awry_index_from_parts(parts: *const awry_parts, devices: *const c_int, n_dev: c_int, out: *mut *mut awry_index) -> c_int;
    pub fn awry_index_build(args: *const awry_build_args, devices: *const c_int, n_dev: c_int, out: *mut *mut awry_index) -> c_int;
    pub fn awry_build_index_file(args: *const awry_build_args) -> c_int;
    pub fn awry_build_parts(alphabet: u32, text: *const u8, n: u64, sa_ratio: u64, device: c_int, blocks: *mut u64,
                            prefix_sums: *mut u64, sa_words: *mut u64, phase_seconds: *mut f64) -> c_int;
    pub fn awry_parts_num_blocks(bwt_len: u64) -> u64;
    pub fn awry_parts_block_words(alphabet: u32) -> u64;
    pub fn awry_parts_sa_words(bwt_len: u64, sa_ratio: u64) -> u64;
    pub fn awry_index_free(index: *mut awry_index);
    pub fn awry_index_save(index: *const awry_index, path: *const c_char) -> c_int;
    pub fn awry_index_info(index: *const awry_index, info: *mut awry_info) -> c_int;
    pub fn awry_index_sequence_header(index: *const awry_index, seq_idx: u64, header: *mut *const c_char, header_len: *mut u64) -> c_int;
    pub fn awry_count_batch(index: *const awry_index, qbytes: *const u8, qoff: *const u64, nq: u64, counts: *mut u64) -> c_int;
    pub fn awry_search_batch(index: *const awry_index, qbytes: *const u8, qoff: *const u64, nq: u64, ranges: *mut awry_range) -> c_int;
    pub fn awry_locate_batch(index: *const awry_index, qbytes: *const u8, qoff: *const u64, nq: u64, flags: u32,
                             hit_off: *mut u64, hits: *mut *mut awry_hit, n_hits: *mut u64) -> c_int;
    pub fn awry_hits_free(hits: *mut awry_hit);
    pub fn awry_count_reads_file(index: *const awry_index, path: *const c_char, counts: *mut *mut u64, n_reads: *mut u64) -> c_int;
    pub fn awry_locate_reads_file(index: *const awry_index, path: *const c_char, flags: u32, hit_off: *mut *mut u64,
                                  hits: *mut *mut awry_hit, n_reads: *mut u64, n_hits: *mut u64) -> c_int;
    pub fn awry_buffer_free(p: *mut c_void);
    pub fn awry_set_host_pack(mode: c_int) -> c_int;
    pub fn awry_locate_batch_into(index: *const awry_index, qbytes: *const u8, qoff: *const u64, nq: u64, flags: u32,
                                  hit_off: *mut u64, hits: *mut awry_hit, capacity: u64, n_hits: *mut u64) -> c_int;
    pub fn awry_initial_range(index: *const awry_index, ascii_symbol: u8, out: *mut awry_range) -> c_int;
    pub fn awry_update_range(index: *const awry_index, range: awry_range, ascii_symbol: u8, out: *mut awry_range) -> c_int;
    pub fn awry_backstep(index: *const awry_index, bwt_row: u64, out: *mut u64) -> c_int;
    pub fn awry_count_device(index: *const awry_index, replica: c_int, d_qbytes: *const u8, d_qoff: *const u64, nq: u64,
                             d_counts: *mut u64, cuda_stream: *mut c_void) -> c_int;
    pub fn awry_locate_device(index: *const awry_index, replica: c_int, d_qbytes: *const u8, d_qoff: *const u64, nq: u64,
                              flags: u32, d_hit_off: *mut u64, d_hits: *mut *mut awry_hit, n_hits: *mut u64,
                              cuda_stream: *mut c_void) -> c_int;
    pub fn awry_device_free(index: *const awry_index, replica: c_int, d_ptr: *mut c_void) -> c_int;
    pub fn awry_device_check(index: *const awry_index, replica: c_int, cuda_stream: *mut c_void) -> c_int;
    pub fn awry_read_sequence_file(path: *const c_char, alphabet: u32, text: *mut *mut u8, n_text: *mut u64,
                                   starts: *mut *mut u64, n_records: *mut u64) -> c_int;
    pub fn awry_host_pack_dna(src: *const u8, n: u64, dst: *mut u8, exceptions: *mut u64, exc_cap: u64, n_exc: *mut u64) -> c_int;
    pub fn awry_count_batch_packed2(index: *const awry_index, crumbs: *const u8, qoff: *const u64, nq: u64,
                                    exceptions: *const u64, n_exc: u64, counts: *mut u64) -> c_int;
    pub fn awry_locate_batch_packed2(index: *const awry_index, crumbs: *const u8, qoff: *const u64, nq: u64,
                                     exceptions: *const u64, n_exc: u64, flags: u32, hit_off: *mut u64,
                                     hits: *mut awry_hit, capacity: u64, n_hits: *mut u64) -> c_int;
    pub fn awry_count_batch_hamming(index: *const awry_index, qbytes: *const u8, qoff: *const u64, nq: u64,
                                    max_mismatches: u32, counts: *mut u64) -> c_int;
    pub fn awry_locate_batch_hamming(index: *const awry_index, qbytes: *const u8, qoff: *const u64, nq: u64,
                                     max_mismatches: u32, hit_off: *mut u64, hits: *mut awry_hit, hit_mismatches: *mut u8,
                                     capacity: u64, n_hits: *mut u64) -> c_int;
    pub fn awry_count_device_hamming(index: *const awry_index, replica: c_int, d_qbytes: *const u8, d_qoff: *const u64,
                                     nq: u64, max_mismatches: u32, d_counts: *mut u64, cuda_stream: *mut c_void) -> c_int;
    pub fn awry_count_batch_strands(index: *const awry_index, qbytes: *const u8, qoff: *const u64, nq: u64,
                                    counts: *mut u64) -> c_int;
    pub fn awry_locate_batch_strands(index: *const awry_index, qbytes: *const u8, qoff: *const u64, nq: u64, flags: u32,
                                     hit_off: *mut u64, hits: *mut awry_hit, capacity: u64, n_hits: *mut u64) -> c_int;
    pub fn awry_count_device_strands(index: *const awry_index, replica: c_int, d_qbytes: *const u8, d_qoff: *const u64,
                                     nq: u64, d_counts: *mut u64, cuda_stream: *mut c_void) -> c_int;
    pub fn awry_locate_device_strands(index: *const awry_index, replica: c_int, d_qbytes: *const u8, d_qoff: *const u64,
                                      nq: u64, flags: u32, d_hit_off: *mut u64, d_hits: *mut *mut awry_hit,
                                      n_hits: *mut u64, cuda_stream: *mut c_void) -> c_int;
    pub fn awry_count_batch_hamming_strands(index: *const awry_index, qbytes: *const u8, qoff: *const u64, nq: u64,
                                            max_mismatches: u32, counts: *mut u64) -> c_int;
    pub fn awry_locate_batch_hamming_strands(index: *const awry_index, qbytes: *const u8, qoff: *const u64, nq: u64,
                                             max_mismatches: u32, hit_off: *mut u64, hits: *mut awry_hit,
                                             hit_mismatches: *mut u8, capacity: u64, n_hits: *mut u64) -> c_int;
    pub fn awry_count_device_hamming_strands(index: *const awry_index, replica: c_int, d_qbytes: *const u8,
                                             d_qoff: *const u64, nq: u64, max_mismatches: u32, d_counts: *mut u64,
                                             cuda_stream: *mut c_void) -> c_int;
    pub fn awry_count_batch_edit(index: *const awry_index, qbytes: *const u8, qoff: *const u64, nq: u64, max_edits: u32,
                                 counts: *mut u64) -> c_int;
    pub fn awry_locate_batch_edit(index: *const awry_index, qbytes: *const u8, qoff: *const u64, nq: u64, max_edits: u32,
                                  hit_off: *mut u64, hits: *mut awry_hit, hit_edits: *mut u8, capacity: u64,
                                  n_hits: *mut u64) -> c_int;
    pub fn awry_count_device_edit(index: *const awry_index, replica: c_int, d_qbytes: *const u8, d_qoff: *const u64,
                                  nq: u64, max_edits: u32, d_counts: *mut u64, cuda_stream: *mut c_void) -> c_int;
    pub fn awry_count_batch_edit_strands(index: *const awry_index, qbytes: *const u8, qoff: *const u64, nq: u64,
                                         max_edits: u32, counts: *mut u64) -> c_int;
    pub fn awry_locate_batch_edit_strands(index: *const awry_index, qbytes: *const u8, qoff: *const u64, nq: u64,
                                          max_edits: u32, hit_off: *mut u64, hits: *mut awry_hit, hit_edits: *mut u8,
                                          capacity: u64, n_hits: *mut u64) -> c_int;
    pub fn awry_count_device_edit_strands(index: *const awry_index, replica: c_int, d_qbytes: *const u8,
                                          d_qoff: *const u64, nq: u64, max_edits: u32, d_counts: *mut u64,
                                          cuda_stream: *mut c_void) -> c_int;
    pub fn awry_count_batch_edit_loci(index: *const awry_index, qbytes: *const u8, qoff: *const u64, nq: u64,
                                      strands: u32, max_edits: u32, counts: *mut u64) -> c_int;
    pub fn awry_locate_batch_edit_loci(index: *const awry_index, qbytes: *const u8, qoff: *const u64, nq: u64,
                                       strands: u32, max_edits: u32, hit_off: *mut u64, hits: *mut awry_hit,
                                       hit_edits: *mut u8, capacity: u64, n_hits: *mut u64) -> c_int;
    pub fn awry_count_device_edit_loci(index: *const awry_index, replica: c_int, d_qbytes: *const u8,
                                       d_qoff: *const u64, nq: u64, strands: u32, max_edits: u32, d_counts: *mut u64,
                                       cuda_stream: *mut c_void) -> c_int;
    pub fn awry_locate_device_edit_loci(index: *const awry_index, replica: c_int, d_qbytes: *const u8,
                                        d_qoff: *const u64, nq: u64, strands: u32, max_edits: u32,
                                        d_hit_off: *mut u64, d_hits: *mut *mut awry_hit, d_hit_edits: *mut *mut u8,
                                        n_hits: *mut u64, cuda_stream: *mut c_void) -> c_int;
    pub fn awry_locate_device_hamming(index: *const awry_index, replica: c_int, d_qbytes: *const u8, d_qoff: *const u64,
                                      nq: u64, max_mismatches: u32, d_hit_off: *mut u64, d_hits: *mut *mut awry_hit,
                                      d_hit_mismatches: *mut *mut u8, n_hits: *mut u64, cuda_stream: *mut c_void)
                                      -> c_int;
    pub fn awry_locate_device_hamming_strands(index: *const awry_index, replica: c_int, d_qbytes: *const u8,
                                              d_qoff: *const u64, nq: u64, max_mismatches: u32, d_hit_off: *mut u64,
                                              d_hits: *mut *mut awry_hit, d_hit_mismatches: *mut *mut u8,
                                              n_hits: *mut u64, cuda_stream: *mut c_void) -> c_int;
    pub fn awry_locate_device_edit(index: *const awry_index, replica: c_int, d_qbytes: *const u8, d_qoff: *const u64,
                                   nq: u64, max_edits: u32, d_hit_off: *mut u64, d_hits: *mut *mut awry_hit,
                                   d_hit_edits: *mut *mut u8, n_hits: *mut u64, cuda_stream: *mut c_void) -> c_int;
    pub fn awry_locate_device_edit_strands(index: *const awry_index, replica: c_int, d_qbytes: *const u8,
                                           d_qoff: *const u64, nq: u64, max_edits: u32, d_hit_off: *mut u64,
                                           d_hits: *mut *mut awry_hit, d_hit_edits: *mut *mut u8, n_hits: *mut u64,
                                           cuda_stream: *mut c_void) -> c_int;
    pub fn awry_align_batch(index: *const awry_index, qbytes: *const u8, qoff: *const u64, nq: u64, metric: u32,
                            strands: u32, k: u32, hit_off: *const u64, hits: *const awry_hit,
                            out: *mut awry_alignment) -> c_int;
    pub fn awry_align_device(index: *const awry_index, replica: c_int, d_qbytes: *const u8, d_qoff: *const u64, nq: u64,
                             metric: u32, strands: u32, k: u32, d_hit_off: *const u64, d_hits: *const awry_hit,
                             n_hits: u64, d_out: *mut awry_alignment, cuda_stream: *mut c_void) -> c_int;
    pub fn awry_alignment_cigar(a: *const awry_alignment, query_len: u32, buf: *mut c_char, cap: usize,
                                needed: *mut usize) -> c_int;
    pub fn awry_map_batch(index: *const awry_index, qbytes: *const u8, qoff: *const u64, nq: u64, metric: u32,
                          strands: u32, k: u32, out: *mut awry_mapping, aln: *mut awry_alignment) -> c_int;
    pub fn awry_map_device(index: *const awry_index, replica: c_int, d_qbytes: *const u8, d_qoff: *const u64, nq: u64,
                           metric: u32, strands: u32, k: u32, d_out: *mut awry_mapping, d_aln: *mut awry_alignment,
                           cuda_stream: *mut c_void) -> c_int;
    pub fn awry_set_host_threads(n: c_int) -> c_int;
    pub fn awry_host_threads() -> c_int;
    pub fn awry_profile_enable(on: c_int) -> c_int;
    pub fn awry_profile_reset() -> c_int;
    pub fn awry_profile_get(out: *mut awry_profile) -> c_int;
    pub fn awry_bench_random_gather(device: c_int, footprint_bytes: u64, granule: u32, lanes: u32, n_reads: u64, iters: c_int,
                                    reads_per_s: *mut f64, gb_per_s: *mut f64) -> c_int;
    pub fn awry_set_search_variant(lanes_per_query: c_int, threads_per_block: c_int, blocks_per_sm: c_int) -> c_int;
    pub fn awry_set_locate_variant(variant: c_int) -> c_int;
    pub fn awry_set_count_variant(variant: c_int) -> c_int;
    pub fn awry_last_error() -> *const c_char;
    pub fn awry_version() -> *const c_char;
}
