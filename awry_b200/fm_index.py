"""Host-side mirror of the reference's public search API over the C ABI (ctypes).

Names, argument meaning and error behaviour follow /root/reference/src:
  FmIndex.load / from_parts            fm_index_file.rs:132, fm_index.rs:271-289
  count_string / locate_string         fm_index.rs:499-501, :516-544
  parallel_count / parallel_locate     fm_index.rs:455-487
  update_range_with_symbol / backstep  fm_index.rs:559-593
  initial_search_range                 fm_index.rs:383
  SearchRange                          search.rs:25-81
  LocalizedSequencePosition            sequence_index.rs:32-78
Where the reference panics (empty query, sentinel in a query) this raises AwryError.
"""
import ctypes as C
import enum
import os
from typing import Iterable, List, NamedTuple, Optional, Sequence, Tuple

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None


def library_path() -> str:
    # AWRY_B200_LIB: another build of the same library (kernel experiments); default = the in-tree one
    return os.environ.get("AWRY_B200_LIB") or os.path.join(_HERE, "libawry_b200.so")


class AwryError(RuntimeError):
    def __init__(self, code: int, message: str):
        super().__init__(f"[awry_b200 {code}] {message}")
        self.code = code


class SymbolAlphabet(enum.IntEnum):  # alphabet.rs:28-31
    Nucleotide = 0
    Amino = 1


class Symbol(NamedTuple):  # alphabet.rs:76-79 (ASCII-encoded symbols only)
    alphabet: SymbolAlphabet
    ascii: str

    @classmethod
    def new_ascii(cls, alphabet: SymbolAlphabet, ch: str) -> "Symbol":
        return cls(alphabet, ch.upper())


class SearchRange(NamedTuple):  # search.rs:25-28
    start_ptr: int
    end_ptr: int

    @classmethod
    def zero(cls) -> "SearchRange":
        return cls(1, 0)

    def is_empty(self) -> bool:
        return self.start_ptr > self.end_ptr

    def len(self) -> int:
        return 0 if self.is_empty() else self.end_ptr - self.start_ptr + 1

    def range_iter(self) -> range:
        return range(0, 0) if self.is_empty() else range(self.start_ptr, self.end_ptr + 1)


class LocalizedSequencePosition(NamedTuple):  # sequence_index.rs:33-36
    sequence_idx: int
    local_position: int


class _Range(C.Structure):
    _fields_ = [("start_ptr", C.c_uint64), ("end_ptr", C.c_uint64)]


class _Info(C.Structure):
    _fields_ = [("version", C.c_uint64), ("sa_ratio", C.c_uint64), ("bwt_len", C.c_uint64),
                ("alphabet", C.c_uint32), ("kmer_len", C.c_uint32), ("n_prefix_sums", C.c_uint32),
                ("n_devices", C.c_uint32), ("prefix_sums", C.c_uint64 * 23),
                ("n_sequences", C.c_uint64), ("device_bytes_blocks", C.c_uint64),
                ("device_bytes_sa", C.c_uint64), ("device_bytes_table", C.c_uint64),
                ("device_bytes_pair", C.c_uint64), ("device_bytes_full_sa", C.c_uint64),
                ("device_bytes_lean_sa", C.c_uint64),
                ("devices", C.c_int32 * 16), ("row_pointer_bits", C.c_uint32), ("lean_sa_ratio", C.c_uint32),
                ("device_bytes_text", C.c_uint64)]


class _Parts(C.Structure):
    _fields_ = [("alphabet", C.c_uint32), ("kmer_len", C.c_uint32), ("sa_ratio", C.c_uint64),
                ("bwt_len", C.c_uint64), ("version", C.c_uint64), ("blocks", C.c_void_p),
                ("prefix_sums", C.c_void_p), ("sa_words", C.c_void_p), ("seq_starts", C.c_void_p),
                ("headers", C.c_void_p), ("n_sequences", C.c_uint64)]


class BuildArgs(C.Structure):  # awry_build_args <- FmBuildArgs (fm_index.rs:78-96)
    _fields_ = [("input_file_src", C.c_char_p), ("output_file_src", C.c_char_p), ("alphabet", C.c_uint32),
                ("lookup_table_kmer_len", C.c_uint32), ("suffix_array_compression_ratio", C.c_uint64),
                ("device", C.c_int32)]


class FmBuildArgs(NamedTuple):  # fm_index.rs:78-96
    input_file_src: str
    suffix_array_output_src: Optional[str] = None      # libsufr's intermediate file: unused here
    suffix_array_compression_ratio: Optional[int] = None
    lookup_table_kmer_len: Optional[int] = None
    alphabet: "SymbolAlphabet" = 0
    max_query_len: Optional[int] = None                # a libsufr sort bound: unused here
    remove_intermediate_suffix_array_file: bool = True


class Profile(C.Structure):
    _fields_ = [("launches", C.c_uint64), ("search_launches", C.c_uint64), ("search_ms", C.c_double),
                ("walk_launches", C.c_uint64), ("walk_ms", C.c_double), ("pack_launches", C.c_uint64),
                ("pack_ms", C.c_double), ("h2d_bytes", C.c_uint64), ("d2h_bytes", C.c_uint64)]

    def as_dict(self):
        return {n: getattr(self, n) for n, _ in self._fields_}


# every symbol include/awry_b200.h declares (checked by tests/test_abi.py)
EXPORTS = ["awry_read_sequence_file", "awry_index_build", "awry_build_index_file", "awry_build_parts", "awry_parts_num_blocks", "awry_parts_block_words",
           "awry_parts_sa_words", "awry_index_load", "awry_index_from_parts", "awry_index_free", "awry_index_save", "awry_index_info",
           "awry_index_sequence_header", "awry_count_batch", "awry_search_batch",
           "awry_locate_batch", "awry_locate_batch_into", "awry_hits_free", "awry_count_reads_file",
           "awry_locate_reads_file", "awry_buffer_free", "awry_initial_range", "awry_update_range",
           "awry_backstep", "awry_count_device", "awry_locate_device", "awry_device_free",
           "awry_device_check", "awry_profile_enable", "awry_profile_reset", "awry_profile_get",
           "awry_bench_random_gather", "awry_set_search_variant", "awry_set_locate_variant", "awry_set_count_variant", "awry_set_host_pack",
           "awry_host_pack_dna", "awry_last_error", "awry_version", "awry_count_batch_packed2",
           "awry_locate_batch_packed2", "awry_set_host_threads", "awry_host_threads", "awry_count_batch_hamming",
           "awry_locate_batch_hamming", "awry_count_device_hamming", "awry_count_batch_strands",
           "awry_locate_batch_strands", "awry_count_device_strands", "awry_locate_device_strands",
           "awry_count_batch_hamming_strands", "awry_locate_batch_hamming_strands", "awry_count_device_hamming_strands",
           "awry_count_batch_edit", "awry_locate_batch_edit", "awry_count_device_edit", "awry_count_batch_edit_strands",
           "awry_locate_batch_edit_strands", "awry_count_device_edit_strands", "awry_locate_device_hamming",
           "awry_locate_device_hamming_strands", "awry_locate_device_edit", "awry_locate_device_edit_strands",
           "awry_align_batch", "awry_align_device", "awry_alignment_cigar", "awry_count_batch_edit_loci",
           "awry_locate_batch_edit_loci", "awry_count_device_edit_loci", "awry_locate_device_edit_loci",
           "awry_map_batch", "awry_map_device"]


def native():
    """The loaded C-ABI library.  Raises (never falls back) when it has not been built."""
    global _LIB
    if _LIB is not None:
        return _LIB
    path = library_path()
    if not os.path.exists(path):
        raise ImportError(
            f"{path} is missing: build it with `make -C awry_b200/csrc` (or "
            "`python -c 'import __graft_entry__ as g; g.build()'`). awry_b200 has no CPU fallback.")
    L = C.CDLL(path)
    vp, u64, i32 = C.c_void_p, C.c_uint64, C.c_int
    L.awry_last_error.restype = C.c_char_p
    L.awry_version.restype = C.c_char_p
    L.awry_read_sequence_file.argtypes = [C.c_char_p, C.c_uint32, C.POINTER(vp), C.POINTER(u64), C.POINTER(vp),
                                          C.POINTER(u64)]
    L.awry_index_build.argtypes = [C.POINTER(BuildArgs), vp, i32, C.POINTER(vp)]
    L.awry_build_index_file.argtypes = [C.POINTER(BuildArgs)]
    L.awry_build_parts.argtypes = [C.c_uint32, vp, u64, u64, i32, vp, vp, vp, vp]
    L.awry_parts_num_blocks.argtypes = [u64]
    L.awry_parts_num_blocks.restype = u64
    L.awry_parts_block_words.argtypes = [C.c_uint32]
    L.awry_parts_block_words.restype = u64
    L.awry_parts_sa_words.argtypes = [u64, u64]
    L.awry_parts_sa_words.restype = u64
    L.awry_index_load.argtypes = [C.c_char_p, vp, i32, C.POINTER(vp)]
    L.awry_index_from_parts.argtypes = [C.POINTER(_Parts), vp, i32, C.POINTER(vp)]
    L.awry_index_free.argtypes = [vp]
    L.awry_index_save.argtypes = [vp, C.c_char_p]
    L.awry_index_free.restype = None
    L.awry_index_info.argtypes = [vp, C.POINTER(_Info)]
    L.awry_index_sequence_header.argtypes = [vp, u64, C.POINTER(C.c_char_p), C.POINTER(u64)]
    L.awry_count_batch.argtypes = [vp, vp, vp, u64, vp]
    L.awry_search_batch.argtypes = [vp, vp, vp, u64, vp]
    L.awry_locate_batch.argtypes = [vp, vp, vp, u64, C.c_uint32, vp, C.POINTER(vp), C.POINTER(u64)]
    L.awry_locate_batch_into.argtypes = [vp, vp, vp, u64, C.c_uint32, vp, vp, u64, C.POINTER(u64)]
    L.awry_hits_free.argtypes = [vp]
    L.awry_hits_free.restype = None
    L.awry_initial_range.argtypes = [vp, C.c_uint8, C.POINTER(_Range)]
    L.awry_update_range.argtypes = [vp, _Range, C.c_uint8, C.POINTER(_Range)]
    L.awry_backstep.argtypes = [vp, u64, C.POINTER(u64)]
    L.awry_count_device.argtypes = [vp, i32, vp, vp, u64, vp, vp]
    L.awry_locate_device.argtypes = [vp, i32, vp, vp, u64, C.c_uint32, vp, C.POINTER(vp),
                                     C.POINTER(u64), vp]
    L.awry_device_free.argtypes = [vp, i32, vp]
    L.awry_device_check.argtypes = [vp, i32, vp]
    L.awry_profile_enable.argtypes = [i32]
    L.awry_profile_get.argtypes = [C.POINTER(Profile)]
    L.awry_bench_random_gather.argtypes = [i32, u64, C.c_uint32, C.c_uint32, u64, i32,
                                           C.POINTER(C.c_double), C.POINTER(C.c_double)]
    L.awry_count_reads_file.argtypes = [vp, C.c_char_p, C.POINTER(vp), C.POINTER(u64)]
    L.awry_locate_reads_file.argtypes = [vp, C.c_char_p, C.c_uint32, C.POINTER(vp), C.POINTER(vp), C.POINTER(u64),
                                         C.POINTER(u64)]
    L.awry_buffer_free.argtypes = [vp]
    L.awry_buffer_free.restype = None
    L.awry_set_search_variant.argtypes = [i32, i32, i32]
    L.awry_set_locate_variant.argtypes = [i32]
    L.awry_set_count_variant.argtypes = [i32]
    L.awry_set_host_pack.argtypes = [i32]
    L.awry_host_pack_dna.argtypes = [vp, u64, vp, vp, u64, C.POINTER(u64)]
    L.awry_count_batch_packed2.argtypes = [vp, vp, vp, u64, vp, u64, vp]
    L.awry_locate_batch_packed2.argtypes = [vp, vp, vp, u64, vp, u64, C.c_uint32, vp, vp, u64, C.POINTER(u64)]
    L.awry_set_host_threads.argtypes = [i32]
    L.awry_count_batch_hamming.argtypes = [vp, vp, vp, u64, C.c_uint32, vp]
    L.awry_locate_batch_hamming.argtypes = [vp, vp, vp, u64, C.c_uint32, vp, vp, vp, u64, C.POINTER(u64)]
    L.awry_count_device_hamming.argtypes = [vp, i32, vp, vp, u64, C.c_uint32, vp, vp]
    L.awry_count_batch_strands.argtypes = [vp, vp, vp, u64, vp]
    L.awry_locate_batch_strands.argtypes = [vp, vp, vp, u64, C.c_uint32, vp, vp, u64, C.POINTER(u64)]
    L.awry_count_device_strands.argtypes = [vp, i32, vp, vp, u64, vp, vp]
    L.awry_locate_device_strands.argtypes = [vp, i32, vp, vp, u64, C.c_uint32, vp, C.POINTER(vp), C.POINTER(u64), vp]
    L.awry_count_batch_hamming_strands.argtypes = [vp, vp, vp, u64, C.c_uint32, vp]
    L.awry_locate_batch_hamming_strands.argtypes = [vp, vp, vp, u64, C.c_uint32, vp, vp, vp, u64, C.POINTER(u64)]
    L.awry_count_device_hamming_strands.argtypes = [vp, i32, vp, vp, u64, C.c_uint32, vp, vp]
    for strands in ("", "_strands"):
        getattr(L, "awry_count_batch_edit" + strands).argtypes = [vp, vp, vp, u64, C.c_uint32, vp]
        getattr(L, "awry_locate_batch_edit" + strands).argtypes = [vp, vp, vp, u64, C.c_uint32, vp, vp, vp, u64,
                                                                   C.POINTER(u64)]
        getattr(L, "awry_count_device_edit" + strands).argtypes = [vp, i32, vp, vp, u64, C.c_uint32, vp, vp]
        for metric in ("hamming", "edit"):
            getattr(L, "awry_locate_device_" + metric + strands).argtypes = [vp, i32, vp, vp, u64, C.c_uint32, vp,
                                                                             C.POINTER(vp), C.POINTER(vp),
                                                                             C.POINTER(u64), vp]
    L.awry_count_batch_edit_loci.argtypes = [vp, vp, vp, u64, C.c_uint32, C.c_uint32, vp]
    L.awry_locate_batch_edit_loci.argtypes = [vp, vp, vp, u64, C.c_uint32, C.c_uint32, vp, vp, vp, u64, C.POINTER(u64)]
    L.awry_count_device_edit_loci.argtypes = [vp, i32, vp, vp, u64, C.c_uint32, C.c_uint32, vp, vp]
    L.awry_locate_device_edit_loci.argtypes = [vp, i32, vp, vp, u64, C.c_uint32, C.c_uint32, vp, C.POINTER(vp),
                                               C.POINTER(vp), C.POINTER(u64), vp]
    L.awry_align_batch.argtypes = [vp, vp, vp, u64, C.c_uint32, C.c_uint32, C.c_uint32, vp, vp, vp]
    L.awry_align_device.argtypes = [vp, i32, vp, vp, u64, C.c_uint32, C.c_uint32, C.c_uint32, vp, vp, u64, vp, vp]
    L.awry_alignment_cigar.argtypes = [vp, C.c_uint32, C.c_char_p, C.c_size_t, C.POINTER(C.c_size_t)]
    L.awry_map_batch.argtypes = [vp, vp, vp, u64, C.c_uint32, C.c_uint32, C.c_uint32, vp, vp]
    L.awry_map_device.argtypes = [vp, i32, vp, vp, u64, C.c_uint32, C.c_uint32, C.c_uint32, vp, vp, vp]
    _LIB = L
    return L


def _check(rc: int):
    if rc != 0:
        raise AwryError(rc, native().awry_last_error().decode(errors="replace"))


def pack_queries(queries: Iterable) -> Tuple[np.ndarray, np.ndarray]:
    """Collects an iterable of str/bytes queries into the C ABI's (qbytes, qoff) form, order
    preserved -- what the Rust facade does with its `impl ParallelIterator<Item=&str>`."""
    qs = [q.encode() if isinstance(q, str) else bytes(q) for q in queries]
    off = np.zeros(len(qs) + 1, dtype=np.uint64)
    if qs:
        off[1:] = np.cumsum([len(q) for q in qs], dtype=np.uint64)
    data = np.frombuffer(b"".join(qs), dtype=np.uint8).copy() if qs else np.zeros(0, np.uint8)
    return data, off


LOCATE_BWT_ORDER, LOCATE_SORTED = 0, 1
METRIC_HAMMING, METRIC_EDIT = 0, 1
_METRICS = {"hamming": METRIC_HAMMING, "edit": METRIC_EDIT, METRIC_HAMMING: METRIC_HAMMING, METRIC_EDIT: METRIC_EDIT}

# awry_alignment / awry_edit_op (include/awry_b200.h): 44 bytes, ops[t] = (qpos, tpos, op, query_sym, text_sym, pad)
EDIT_OP_DTYPE = np.dtype([("qpos", "<u4"), ("tpos", "<u4"), ("op", "u1"), ("query_sym", "u1"), ("text_sym", "u1"),
                          ("pad", "u1")])
ALIGNMENT_DTYPE = np.dtype([("text_len", "<u4"), ("distance", "u1"), ("n_ops", "u1"), ("pad", "u1", (2,)),
                            ("ops", EDIT_OP_DTYPE, (3,))])
assert ALIGNMENT_DTYPE.itemsize == 44

# awry_mapping (include/awry_b200.h): 32 bytes; seq_idx / local_pos are ~0 when the read is unmapped
MAP_UNMAPPED, MAP_REFUSED = 1, 2
MAPPING_DTYPE = np.dtype([("seq_idx", "<u8"), ("local_pos", "<u8"), ("n_best", "<u4"), ("n_second", "<u4"),
                          ("distance", "u1"), ("strand", "u1"), ("mapq", "u1"), ("flags", "u1"), ("pad", "<u4")])
assert MAPPING_DTYPE.itemsize == 32


def cigar(alignment, query_len: int) -> str:
    """awry_alignment_cigar: the extended CIGAR (=, X, I, D) of one alignment (a record of ALIGNMENT_DTYPE) of a query of
    length query_len; no device needed"""
    rec = np.ascontiguousarray(np.asarray(alignment, dtype=ALIGNMENT_DTYPE).reshape(1))
    need = C.c_size_t()
    native().awry_alignment_cigar(rec.ctypes.data, int(query_len), None, 0, C.byref(need))
    buf = C.create_string_buffer(max(1, need.value))
    _check(native().awry_alignment_cigar(rec.ctypes.data, int(query_len), buf, len(buf), C.byref(need)))
    return buf.value.decode()


class FmIndex:
    """Device-resident replica of an awry FM-index (query side)."""

    def __init__(self, handle: int):
        self._h = C.c_void_p(handle)
        info = _Info()
        _check(native().awry_index_info(self._h, C.byref(info)))
        self._info = info

    # ---- construction -------------------------------------------------------------------
    @classmethod
    def load(cls, path, devices: Sequence[int] = None) -> "FmIndex":
        """FmIndex::load (fm_index_file.rs:132-160)."""
        h = C.c_void_p()
        dev = (C.c_int * len(devices))(*devices) if devices else None
        _check(native().awry_index_load(os.fsencode(path), dev, len(devices) if devices else 0,
                                        C.byref(h)))
        return cls(h.value)

    @classmethod
    def new(cls, args: "FmBuildArgs", devices: Sequence[int] = None, save_to=None) -> "FmIndex":
        """FmIndex::new (fm_index.rs:142-268) on the GPU: FASTA/FASTQ -> searchable index; with
        `save_to` also FmIndex::save (fm_index_file.rs:42) of the same index."""
        a = BuildArgs(os.fsencode(args.input_file_src), os.fsencode(save_to) if save_to else None,
                      int(args.alphabet), int(args.lookup_table_kmer_len or 0),
                      int(args.suffix_array_compression_ratio or 0), int(devices[0]) if devices else 0)
        h = C.c_void_p()
        dev = (C.c_int * len(devices))(*devices) if devices else None
        _check(native().awry_index_build(C.byref(a), dev, len(devices) if devices else 0, C.byref(h)))
        return cls(h.value)

    @classmethod
    def from_parts(cls, alphabet, sa_ratio, bwt_len, kmer_len, blocks, prefix_sums, sa_words,
                   seq_starts=None, headers=None, devices: Sequence[int] = None) -> "FmIndex":
        """Device replica of the arrays the reference's FmIndex::new produced
        (fm_index.rs:242-251), all in the reference layout."""
        blocks = np.ascontiguousarray(blocks, dtype=np.uint64)
        prefix_sums = np.ascontiguousarray(prefix_sums, dtype=np.uint64)
        sa_words = np.ascontiguousarray(sa_words, dtype=np.uint64)
        if seq_starts is None:
            seq_starts = np.zeros(1, dtype=np.uint64)
        seq_starts = np.ascontiguousarray(seq_starts, dtype=np.uint64)
        hdr_arr = None
        if headers is not None:
            hdr_arr = (C.c_char_p * len(headers))(*[h.encode() for h in headers])
        p = _Parts(int(alphabet), int(kmer_len), int(sa_ratio), int(bwt_len), 1, blocks.ctypes.data,
                   prefix_sums.ctypes.data, sa_words.ctypes.data, seq_starts.ctypes.data,
                   C.cast(hdr_arr, C.c_void_p) if hdr_arr is not None else None, len(seq_starts))
        h = C.c_void_p()
        dev = (C.c_int * len(devices))(*devices) if devices else None
        _check(native().awry_index_from_parts(C.byref(p), dev, len(devices) if devices else 0,
                                              C.byref(h)))
        return cls(h.value)

    def save(self, path) -> None:
        """FmIndex::save (fm_index_file.rs:42-106): `.awry` v1 file from this handle's device layout."""
        _check(native().awry_index_save(self._h, os.fsencode(path)))

    def close(self):
        if getattr(self, "_h", None):
            native().awry_index_free(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    # ---- getters (fm_index.rs:302-368) ----------------------------------------------------
    @property
    def handle(self):
        return self._h

    def alphabet(self) -> SymbolAlphabet:
        return SymbolAlphabet(self._info.alphabet)

    def suffix_array_compression_ratio(self) -> int:
        return int(self._info.sa_ratio)

    def bwt_len(self) -> int:
        return int(self._info.bwt_len)

    def version_number(self) -> int:
        return int(self._info.version)

    def prefix_sums(self) -> List[int]:
        return [int(self._info.prefix_sums[i]) for i in range(self._info.n_prefix_sums)]

    def kmer_len(self) -> int:
        return int(self._info.kmer_len)

    def row_pointer_bits(self) -> int:
        """32 while bwt_len < 2^32 - 256 (cooperative kernels), else 64 (kernels_wide.cu)"""
        return int(self._info.row_pointer_bits)

    def lean_sa_ratio(self) -> int:
        """sampling distance of the derived position-sampled suffix array (bounded locate), 0 if not built"""
        return int(self._info.lean_sa_ratio)

    def n_devices(self) -> int:
        return int(self._info.n_devices)

    def device_bytes(self) -> dict:
        return {"blocks": int(self._info.device_bytes_blocks), "sa": int(self._info.device_bytes_sa),
                "table": int(self._info.device_bytes_table), "pair": int(self._info.device_bytes_pair),
                "full_sa": int(self._info.device_bytes_full_sa), "lean_sa": int(self._info.device_bytes_lean_sa), "text": int(self._info.device_bytes_text)}

    def sequence_header(self, seq_idx: int) -> str:
        p, n = C.c_char_p(), C.c_uint64()
        _check(native().awry_index_sequence_header(self._h, seq_idx, C.byref(p), C.byref(n)))
        return C.string_at(p, n.value).decode(errors="replace")

    # ---- single steps ---------------------------------------------------------------------
    @staticmethod
    def _ascii(sym) -> int:
        if isinstance(sym, Symbol):
            sym = sym.ascii
        if isinstance(sym, str):
            return ord(sym)
        if isinstance(sym, bytes):
            return sym[0]
        return int(sym)

    def initial_search_range(self, sym) -> SearchRange:
        r = _Range()
        _check(native().awry_initial_range(self._h, self._ascii(sym), C.byref(r)))
        return SearchRange(r.start_ptr, r.end_ptr)

    def update_range_with_symbol(self, search_range: SearchRange, sym) -> SearchRange:
        r = _Range()
        _check(native().awry_update_range(self._h, _Range(search_range[0], search_range[1]),
                                          self._ascii(sym), C.byref(r)))
        return SearchRange(r.start_ptr, r.end_ptr)

    def backstep(self, search_pointer: int) -> int:
        out = C.c_uint64()
        _check(native().awry_backstep(self._h, search_pointer, C.byref(out)))
        return out.value

    # ---- batched search -------------------------------------------------------------------
    def count_packed(self, qbytes: np.ndarray, qoff: np.ndarray, out: np.ndarray = None) -> np.ndarray:
        qbytes = np.ascontiguousarray(qbytes, dtype=np.uint8)
        qoff = np.ascontiguousarray(qoff, dtype=np.uint64)
        nq = len(qoff) - 1
        counts = out if out is not None else np.empty(nq, dtype=np.uint64)
        _check(native().awry_count_batch(self._h, qbytes.ctypes.data, qoff.ctypes.data, nq,
                                         counts.ctypes.data))
        return counts

    def search_packed(self, qbytes: np.ndarray, qoff: np.ndarray) -> np.ndarray:
        qbytes = np.ascontiguousarray(qbytes, dtype=np.uint8)
        qoff = np.ascontiguousarray(qoff, dtype=np.uint64)
        nq = len(qoff) - 1
        ranges = np.empty((nq, 2), dtype=np.uint64)
        _check(native().awry_search_batch(self._h, qbytes.ctypes.data, qoff.ctypes.data, nq,
                                          ranges.ctypes.data))
        return ranges

    def locate_packed(self, qbytes: np.ndarray, qoff: np.ndarray, sorted_hits: bool = False):
        """-> (hit_off uint64[nq+1], hits uint64[n_hits, 2] = (seq_idx, local_pos))"""
        qbytes = np.ascontiguousarray(qbytes, dtype=np.uint8)
        qoff = np.ascontiguousarray(qoff, dtype=np.uint64)
        nq = len(qoff) - 1
        hit_off = np.zeros(nq + 1, dtype=np.uint64)
        hits, n = C.c_void_p(), C.c_uint64()
        _check(native().awry_locate_batch(self._h, qbytes.ctypes.data, qoff.ctypes.data, nq,
                                          LOCATE_SORTED if sorted_hits else LOCATE_BWT_ORDER,
                                          hit_off.ctypes.data, C.byref(hits), C.byref(n)))
        arr = np.empty((n.value, 2), dtype=np.uint64)
        if n.value:
            C.memmove(arr.ctypes.data, hits, n.value * 16)
        native().awry_hits_free(hits)
        return hit_off, arr

    def locate_packed_into(self, qbytes: np.ndarray, qoff: np.ndarray, hit_off: np.ndarray, hits: np.ndarray,
                           sorted_hits: bool = False) -> int:
        """locate into caller-owned arrays (hit_off uint64[nq+1], hits uint64[capacity, 2], e.g. pinned);
        returns the number of hits; raises AwryError(-8) with `.needed` set when hits is too small."""
        qbytes = np.ascontiguousarray(qbytes, dtype=np.uint8)
        qoff = np.ascontiguousarray(qoff, dtype=np.uint64)
        n = C.c_uint64()
        rc = native().awry_locate_batch_into(self._h, qbytes.ctypes.data, qoff.ctypes.data, len(qoff) - 1,
                                             LOCATE_SORTED if sorted_hits else LOCATE_BWT_ORDER,
                                             hit_off.ctypes.data, hits.ctypes.data, len(hits), C.byref(n))
        if rc != 0:
            err = AwryError(rc, native().awry_last_error().decode(errors="replace"))
            err.needed = n.value
            raise err
        return n.value

    # ---- pre-packed nucleotide reads (2 bits per base; see include/awry_b200.h) --------------
    def count_prepacked(self, crumbs: np.ndarray, qoff: np.ndarray, exceptions: np.ndarray = None,
                        out: np.ndarray = None) -> np.ndarray:
        """parallel_count on reads the caller holds as 2-bit codes (the output of host_pack_dna)."""
        crumbs = np.ascontiguousarray(crumbs, dtype=np.uint8)
        qoff = np.ascontiguousarray(qoff, dtype=np.uint64)
        exc = np.zeros(0, np.uint64) if exceptions is None else np.ascontiguousarray(exceptions, dtype=np.uint64)
        nq = len(qoff) - 1
        counts = out if out is not None else np.empty(nq, dtype=np.uint64)
        _check(native().awry_count_batch_packed2(self._h, crumbs.ctypes.data, qoff.ctypes.data, nq,
                                                 exc.ctypes.data if len(exc) else None, len(exc), counts.ctypes.data))
        return counts

    def locate_prepacked_into(self, crumbs: np.ndarray, qoff: np.ndarray, exceptions: np.ndarray, hit_off: np.ndarray,
                              hits: np.ndarray, sorted_hits: bool = False) -> int:
        """parallel_locate on 2-bit packed reads into caller-owned arrays (see locate_packed_into)."""
        crumbs = np.ascontiguousarray(crumbs, dtype=np.uint8)
        qoff = np.ascontiguousarray(qoff, dtype=np.uint64)
        exc = np.zeros(0, np.uint64) if exceptions is None else np.ascontiguousarray(exceptions, dtype=np.uint64)
        n = C.c_uint64()
        rc = native().awry_locate_batch_packed2(self._h, crumbs.ctypes.data, qoff.ctypes.data, len(qoff) - 1,
                                                exc.ctypes.data if len(exc) else None, len(exc),
                                                LOCATE_SORTED if sorted_hits else LOCATE_BWT_ORDER,
                                                hit_off.ctypes.data, hits.ctypes.data, len(hits), C.byref(n))
        if rc != 0:
            err = AwryError(rc, native().awry_last_error().decode(errors="replace"))
            err.needed = n.value
            raise err
        return n.value

    # ---- Hamming search: windows within max_mismatches <= 3 substitutions (include/awry_b200.h) --
    def count_hamming_packed(self, qbytes: np.ndarray, qoff: np.ndarray, max_mismatches: int) -> np.ndarray:
        """-> uint64[nq, max_mismatches + 1]: [q, d] = windows of the text at Hamming distance exactly d"""
        qbytes = np.ascontiguousarray(qbytes, dtype=np.uint8)
        qoff = np.ascontiguousarray(qoff, dtype=np.uint64)
        nq = len(qoff) - 1
        counts = np.zeros((nq, int(max_mismatches) + 1), dtype=np.uint64)
        _check(native().awry_count_batch_hamming(self._h, qbytes.ctypes.data, qoff.ctypes.data, nq, int(max_mismatches),
                                                 counts.ctypes.data))
        return counts

    def locate_hamming_packed(self, qbytes: np.ndarray, qoff: np.ndarray, max_mismatches: int, capacity: int = None):
        """-> (hit_off uint64[nq+1], hits uint64[n_hits, 2] = (seq_idx, local_pos) of the window start, mismatches
        uint8[n_hits]); per query ascending by text position.  A first guess of `capacity` hits (default: one per
        query) that proves too small is retried once with the total the library reports."""
        qbytes = np.ascontiguousarray(qbytes, dtype=np.uint8)
        qoff = np.ascontiguousarray(qoff, dtype=np.uint64)
        nq = len(qoff) - 1
        hit_off = np.zeros(nq + 1, dtype=np.uint64)
        cap = max(1, nq if capacity is None else int(capacity))
        n = C.c_uint64()
        for _ in range(2):
            hits = np.zeros((cap, 2), dtype=np.uint64)
            mm = np.zeros(cap, dtype=np.uint8)
            rc = native().awry_locate_batch_hamming(self._h, qbytes.ctypes.data, qoff.ctypes.data, nq, int(max_mismatches),
                                                    hit_off.ctypes.data, hits.ctypes.data, mm.ctypes.data, cap, C.byref(n))
            if rc != -8:
                break
            cap = max(1, n.value)
        if rc != 0:
            err = AwryError(rc, native().awry_last_error().decode(errors="replace"))
            err.needed = n.value
            raise err
        return hit_off, hits[: n.value], mm[: n.value]

    def count_hamming_device(self, d_qbytes: int, d_qoff: int, nq: int, max_mismatches: int, d_counts: int,
                             stream: int = 0, replica: int = 0):
        """count_hamming_packed on device pointers (d_counts: nq * (max_mismatches + 1) u64); see device_check"""
        _check(native().awry_count_device_hamming(self._h, replica, d_qbytes, d_qoff, nq, int(max_mismatches), d_counts,
                                                  stream))

    def _locate_approx_device(self, fn, d_qbytes, d_qoff, nq, k, d_hit_off, distances, stream, replica):
        hits, dist, n = C.c_void_p(), C.c_void_p(), C.c_uint64()
        _check(fn(self._h, replica, d_qbytes, d_qoff, nq, int(k), d_hit_off, C.byref(hits),
                  C.byref(dist) if distances else None, C.byref(n), stream))
        return hits.value, dist.value, n.value

    def locate_hamming_device(self, d_qbytes: int, d_qoff: int, nq: int, max_mismatches: int, d_hit_off: int,
                              distances: bool = True, stream: int = 0, replica: int = 0):
        """locate_hamming_packed on device pointers (d_hit_off: nq + 1 u64) -> (device pointer to n_hits x {u64
        seq_idx, u64 local_pos}, device pointer to n_hits u8 mismatches (None without `distances`), n_hits); both
        pointers are None when there are no hits.  Free each with device_free; see device_check"""
        return self._locate_approx_device(native().awry_locate_device_hamming, d_qbytes, d_qoff, nq, max_mismatches,
                                          d_hit_off, distances, stream, replica)

    # ---- both strands: every query and its reverse complement (include/awry_b200.h) ----------
    def count_strands_packed(self, qbytes: np.ndarray, qoff: np.ndarray) -> np.ndarray:
        """-> uint64[nq, 2]: [q, 0] = count of q, [q, 1] = count of its reverse complement"""
        qbytes = np.ascontiguousarray(qbytes, dtype=np.uint8)
        qoff = np.ascontiguousarray(qoff, dtype=np.uint64)
        nq = len(qoff) - 1
        counts = np.empty((nq, 2), dtype=np.uint64)
        _check(native().awry_count_batch_strands(self._h, qbytes.ctypes.data, qoff.ctypes.data, nq, counts.ctypes.data))
        return counts

    def locate_strands_packed(self, qbytes: np.ndarray, qoff: np.ndarray, sorted_hits: bool = False,
                              capacity: int = None):
        """-> (hit_off uint64[2 nq + 1], hits uint64[n_hits, 2] = (seq_idx, local_pos)): query q's forward hits are
        hits[hit_off[2q]:hit_off[2q+1]], its reverse-strand hits hits[hit_off[2q+1]:hit_off[2q+2]].  A first guess of
        `capacity` hits (default: two per query) that proves too small is retried once with the reported total."""
        qbytes = np.ascontiguousarray(qbytes, dtype=np.uint8)
        qoff = np.ascontiguousarray(qoff, dtype=np.uint64)
        nq = len(qoff) - 1
        hit_off = np.zeros(2 * nq + 1, dtype=np.uint64)
        cap = max(1, 2 * nq if capacity is None else int(capacity))
        n = C.c_uint64()
        for _ in range(2):
            hits = np.zeros((cap, 2), dtype=np.uint64)
            rc = native().awry_locate_batch_strands(self._h, qbytes.ctypes.data, qoff.ctypes.data, nq,
                                                    LOCATE_SORTED if sorted_hits else LOCATE_BWT_ORDER,
                                                    hit_off.ctypes.data, hits.ctypes.data, cap, C.byref(n))
            if rc != -8:
                break
            cap = max(1, n.value)
        if rc != 0:
            err = AwryError(rc, native().awry_last_error().decode(errors="replace"))
            err.needed = n.value
            raise err
        return hit_off, hits[: n.value]

    def count_strands_device(self, d_qbytes: int, d_qoff: int, nq: int, d_counts: int, stream: int = 0,
                             replica: int = 0):
        """count_strands_packed on device pointers (d_counts: 2 nq u64, [2q] forward, [2q+1] reverse); see device_check"""
        _check(native().awry_count_device_strands(self._h, replica, d_qbytes, d_qoff, nq, d_counts, stream))

    def locate_strands_device(self, d_qbytes: int, d_qoff: int, nq: int, d_hit_off: int, sorted_hits=False,
                              stream: int = 0, replica: int = 0):
        """locate_strands_packed on device pointers (d_hit_off: 2 nq + 1 u64) -> (device pointer to n_hits x
        {u64 seq_idx, u64 local_pos}, n_hits); free with device_free"""
        hits, n = C.c_void_p(), C.c_uint64()
        _check(native().awry_locate_device_strands(self._h, replica, d_qbytes, d_qoff, nq,
                                                   LOCATE_SORTED if sorted_hits else LOCATE_BWT_ORDER,
                                                   d_hit_off, C.byref(hits), C.byref(n), stream))
        return hits.value, n.value

    # ---- Hamming search on both strands (include/awry_b200.h) ----------------------------------
    def count_hamming_strands_packed(self, qbytes: np.ndarray, qoff: np.ndarray, max_mismatches: int) -> np.ndarray:
        """-> uint64[nq, 2, max_mismatches + 1]: [q, s, d] = windows at Hamming distance exactly d from q (s = 0) or
        from its reverse complement (s = 1)"""
        qbytes = np.ascontiguousarray(qbytes, dtype=np.uint8)
        qoff = np.ascontiguousarray(qoff, dtype=np.uint64)
        nq = len(qoff) - 1
        counts = np.zeros((nq, 2, int(max_mismatches) + 1), dtype=np.uint64)
        _check(native().awry_count_batch_hamming_strands(self._h, qbytes.ctypes.data, qoff.ctypes.data, nq,
                                                         int(max_mismatches), counts.ctypes.data))
        return counts

    def locate_hamming_strands_packed(self, qbytes: np.ndarray, qoff: np.ndarray, max_mismatches: int,
                                      capacity: int = None):
        """-> (hit_off uint64[2 nq + 1], hits uint64[n_hits, 2], mismatches uint8[n_hits]): query q's forward hits are
        hits[hit_off[2q]:hit_off[2q+1]], its reverse-strand hits hits[hit_off[2q+1]:hit_off[2q+2]], each ascending by
        text position.  A first guess of `capacity` hits (default: two per query) that proves too small is retried
        once with the total the library reports."""
        qbytes = np.ascontiguousarray(qbytes, dtype=np.uint8)
        qoff = np.ascontiguousarray(qoff, dtype=np.uint64)
        nq = len(qoff) - 1
        hit_off = np.zeros(2 * nq + 1, dtype=np.uint64)
        cap = max(1, 2 * nq if capacity is None else int(capacity))
        n = C.c_uint64()
        for _ in range(2):
            hits = np.zeros((cap, 2), dtype=np.uint64)
            mm = np.zeros(cap, dtype=np.uint8)
            rc = native().awry_locate_batch_hamming_strands(self._h, qbytes.ctypes.data, qoff.ctypes.data, nq,
                                                            int(max_mismatches), hit_off.ctypes.data, hits.ctypes.data,
                                                            mm.ctypes.data, cap, C.byref(n))
            if rc != -8:
                break
            cap = max(1, n.value)
        if rc != 0:
            err = AwryError(rc, native().awry_last_error().decode(errors="replace"))
            err.needed = n.value
            raise err
        return hit_off, hits[: n.value], mm[: n.value]

    def count_hamming_strands_device(self, d_qbytes: int, d_qoff: int, nq: int, max_mismatches: int, d_counts: int,
                                     stream: int = 0, replica: int = 0):
        """count_hamming_strands_packed on device pointers (d_counts: 2 nq (max_mismatches + 1) u64, [(2q + s)(k+1) +
        d]); see device_check"""
        _check(native().awry_count_device_hamming_strands(self._h, replica, d_qbytes, d_qoff, nq, int(max_mismatches),
                                                          d_counts, stream))

    def locate_hamming_strands_device(self, d_qbytes: int, d_qoff: int, nq: int, max_mismatches: int, d_hit_off: int,
                                      distances: bool = True, stream: int = 0, replica: int = 0):
        """locate_hamming_strands_packed on device pointers (d_hit_off: 2 nq + 1 u64) -> (hits pointer, mismatches
        pointer or None, n_hits), as locate_hamming_device; free each with device_free"""
        return self._locate_approx_device(native().awry_locate_device_hamming_strands, d_qbytes, d_qoff, nq,
                                          max_mismatches, d_hit_off, distances, stream, replica)

    # ---- edit-distance search: starts within max_edits <= 3 substitutions, insertions, deletions -------------
    def _count_edit(self, fn, qbytes, qoff, max_edits, per):
        qbytes = np.ascontiguousarray(qbytes, dtype=np.uint8)
        qoff = np.ascontiguousarray(qoff, dtype=np.uint64)
        nq = len(qoff) - 1
        counts = np.zeros((nq,) + per + (int(max_edits) + 1,), dtype=np.uint64)
        _check(fn(self._h, qbytes.ctypes.data, qoff.ctypes.data, nq, int(max_edits), counts.ctypes.data))
        return counts

    def _locate_edit(self, fn, qbytes, qoff, max_edits, per, capacity):
        qbytes = np.ascontiguousarray(qbytes, dtype=np.uint8)
        qoff = np.ascontiguousarray(qoff, dtype=np.uint64)
        nq = len(qoff) - 1
        hit_off = np.zeros(per * nq + 1, dtype=np.uint64)
        cap = max(1, per * nq if capacity is None else int(capacity))
        n = C.c_uint64()
        for _ in range(2):
            hits = np.zeros((cap, 2), dtype=np.uint64)
            ed = np.zeros(cap, dtype=np.uint8)
            rc = fn(self._h, qbytes.ctypes.data, qoff.ctypes.data, nq, int(max_edits), hit_off.ctypes.data,
                    hits.ctypes.data, ed.ctypes.data, cap, C.byref(n))
            if rc != -8:
                break
            cap = max(1, n.value)
        if rc != 0:
            err = AwryError(rc, native().awry_last_error().decode(errors="replace"))
            err.needed = n.value
            raise err
        return hit_off, hits[: n.value], ed[: n.value]

    def count_edit_packed(self, qbytes: np.ndarray, qoff: np.ndarray, max_edits: int) -> np.ndarray:
        """-> uint64[nq, max_edits + 1]: [q, d] = text starts s whose edit distance d(s) to q is exactly d"""
        return self._count_edit(native().awry_count_batch_edit, qbytes, qoff, max_edits, ())

    def locate_edit_packed(self, qbytes: np.ndarray, qoff: np.ndarray, max_edits: int, capacity: int = None):
        """-> (hit_off uint64[nq+1], hits uint64[n_hits, 2] = (seq_idx, local_pos) of the start, edits uint8[n_hits]);
        per query ascending by text position.  Neighbouring starts of one locus are all reported.  A first guess of
        `capacity` hits (default: one per query) that proves too small is retried once with the reported total."""
        return self._locate_edit(native().awry_locate_batch_edit, qbytes, qoff, max_edits, 1, capacity)

    def count_edit_device(self, d_qbytes: int, d_qoff: int, nq: int, max_edits: int, d_counts: int, stream: int = 0,
                          replica: int = 0):
        """count_edit_packed on device pointers (d_counts: nq * (max_edits + 1) u64); see device_check"""
        _check(native().awry_count_device_edit(self._h, replica, d_qbytes, d_qoff, nq, int(max_edits), d_counts, stream))

    def locate_edit_device(self, d_qbytes: int, d_qoff: int, nq: int, max_edits: int, d_hit_off: int,
                           distances: bool = True, stream: int = 0, replica: int = 0):
        """locate_edit_packed on device pointers (d_hit_off: nq + 1 u64) -> (device pointer to n_hits x {u64 seq_idx,
        u64 local_pos}, device pointer to n_hits u8 edits (None without `distances`), n_hits); both pointers are None
        when there are no hits.  Free each with device_free; see device_check"""
        return self._locate_approx_device(native().awry_locate_device_edit, d_qbytes, d_qoff, nq, max_edits, d_hit_off,
                                          distances, stream, replica)

    def count_edit_strands_packed(self, qbytes: np.ndarray, qoff: np.ndarray, max_edits: int) -> np.ndarray:
        """-> uint64[nq, 2, max_edits + 1]: [q, s, d] = starts at edit distance exactly d from q (s = 0) or from its
        reverse complement (s = 1)"""
        return self._count_edit(native().awry_count_batch_edit_strands, qbytes, qoff, max_edits, (2,))

    def locate_edit_strands_packed(self, qbytes: np.ndarray, qoff: np.ndarray, max_edits: int, capacity: int = None):
        """-> (hit_off uint64[2 nq + 1], hits uint64[n_hits, 2], edits uint8[n_hits]): query q's forward hits are
        hits[hit_off[2q]:hit_off[2q+1]], its reverse-strand hits hits[hit_off[2q+1]:hit_off[2q+2]], each ascending by
        text position (default capacity: two per query, retried once as locate_edit_packed)"""
        return self._locate_edit(native().awry_locate_batch_edit_strands, qbytes, qoff, max_edits, 2, capacity)

    def count_edit_strands_device(self, d_qbytes: int, d_qoff: int, nq: int, max_edits: int, d_counts: int,
                                  stream: int = 0, replica: int = 0):
        """count_edit_strands_packed on device pointers (d_counts: 2 nq (max_edits + 1) u64, [(2q + s)(k+1) + d]);
        see device_check"""
        _check(native().awry_count_device_edit_strands(self._h, replica, d_qbytes, d_qoff, nq, int(max_edits), d_counts,
                                                       stream))

    def locate_edit_strands_device(self, d_qbytes: int, d_qoff: int, nq: int, max_edits: int, d_hit_off: int,
                                   distances: bool = True, stream: int = 0, replica: int = 0):
        """locate_edit_strands_packed on device pointers (d_hit_off: 2 nq + 1 u64) -> (hits pointer, edits pointer or
        None, n_hits), as locate_edit_device; free each with device_free"""
        return self._locate_approx_device(native().awry_locate_device_edit_strands, d_qbytes, d_qoff, nq, max_edits,
                                          d_hit_off, distances, stream, replica)

    # ---- edit-distance loci: one hit per occurrence, not every neighbouring start (include/awry_b200.h) ----------
    def count_edit_loci_packed(self, qbytes: np.ndarray, qoff: np.ndarray, max_edits: int,
                               strands: bool = False) -> np.ndarray:
        """-> uint64[nq, max_edits + 1] (strands: [nq, 2, max_edits + 1]): [q, (s,) d] = loci of q (s = 0) or of its
        reverse complement (s = 1) at edit distance exactly d"""
        fn = native().awry_count_batch_edit_loci
        return self._count_edit(lambda h, qb, qo, nq, k, c: fn(h, qb, qo, nq, int(bool(strands)), k, c), qbytes, qoff,
                                max_edits, (2,) if strands else ())

    def locate_edit_loci_packed(self, qbytes: np.ndarray, qoff: np.ndarray, max_edits: int, strands: bool = False,
                                capacity: int = None):
        """-> (hit_off, hits, edits) as locate_edit_packed (strands: as locate_edit_strands_packed), holding only the
        loci: the hits no hit within max_edits beats and that do not continue a run of adjacent equal-distance starts"""
        fn = native().awry_locate_batch_edit_loci
        return self._locate_edit(lambda h, qb, qo, nq, k, *rest: fn(h, qb, qo, nq, int(bool(strands)), k, *rest), qbytes,
                                 qoff, max_edits, 2 if strands else 1, capacity)

    def count_edit_loci_device(self, d_qbytes: int, d_qoff: int, nq: int, max_edits: int, d_counts: int,
                               strands: bool = False, stream: int = 0, replica: int = 0):
        """count_edit_loci_packed on device pointers (d_counts: (nq << strands) (max_edits + 1) u64); costs about a
        device locate (two synchronisations); see device_check"""
        _check(native().awry_count_device_edit_loci(self._h, replica, d_qbytes, d_qoff, nq, int(bool(strands)),
                                                    int(max_edits), d_counts, stream))

    def locate_edit_loci_device(self, d_qbytes: int, d_qoff: int, nq: int, max_edits: int, d_hit_off: int,
                                strands: bool = False, distances: bool = True, stream: int = 0, replica: int = 0):
        """locate_edit_loci_packed on device pointers (d_hit_off: (nq << strands) + 1 u64) -> (hits pointer, edits
        pointer or None, n_hits), as locate_edit_device; free each with device_free"""
        fn = native().awry_locate_device_edit_loci
        return self._locate_approx_device(
            lambda h, rep, qb, qo, nq, k, *rest: fn(h, rep, qb, qo, nq, int(bool(strands)), k, *rest), d_qbytes, d_qoff,
            nq, max_edits, d_hit_off, distances, stream, replica)

    # ---- alignment of located Hamming / edit-distance hits (include/awry_b200.h) -------------
    def align_hits_packed(self, qbytes: np.ndarray, qoff: np.ndarray, metric, max_dist: int, hit_off: np.ndarray,
                          hits: np.ndarray, strands: bool = False) -> np.ndarray:
        """-> ALIGNMENT_DTYPE[n_hits]: each hit of a locate_{hamming,edit}[_strands]_packed call (its hit_off and hits,
        with that call's reads, metric "hamming" / "edit" and k) aligned: text_len, distance, the ops (a CIGAR: see
        cigar()).  Reverse-strand hits are aligned as rc(q)."""
        qbytes = np.ascontiguousarray(qbytes, dtype=np.uint8)
        qoff = np.ascontiguousarray(qoff, dtype=np.uint64)
        hit_off = np.ascontiguousarray(hit_off, dtype=np.uint64)
        hits = np.ascontiguousarray(hits, dtype=np.uint64).reshape(-1, 2)
        out = np.zeros(max(1, len(hits)), dtype=ALIGNMENT_DTYPE)
        _check(native().awry_align_batch(self._h, qbytes.ctypes.data, qoff.ctypes.data, len(qoff) - 1, _METRICS[metric],
                                         int(bool(strands)), int(max_dist), hit_off.ctypes.data, hits.ctypes.data,
                                         out.ctypes.data))
        return out[:len(hits)]

    def align_hits_device(self, d_qbytes: int, d_qoff: int, nq: int, metric, max_dist: int, d_hit_off: int, d_hits: int,
                          n_hits: int, d_out: int, strands: bool = False, stream: int = 0, replica: int = 0):
        """align_hits_packed on device pointers: the reads and the hits of a locate_*_device call, d_out = n_hits x 44
        bytes (ALIGNMENT_DTYPE) on the device.  Returns without waiting; see device_check"""
        _check(native().awry_align_device(self._h, replica, d_qbytes, d_qoff, nq, _METRICS[metric], int(bool(strands)),
                                          int(max_dist), d_hit_off, d_hits, n_hits, d_out, stream))

    # ---- read mapping: the best locus per read (include/awry_b200.h) -------------------------
    def map_packed(self, qbytes: np.ndarray, qoff: np.ndarray, metric, max_dist: int, strands: bool = True,
                   align: bool = True):
        """-> (MAPPING_DTYPE[nq], ALIGNMENT_DTYPE[nq] or None): each read's best locus under metric "hamming" / "edit"
        within max_dist, over both strands (strands=True) or the read as given: distance, the number of distinct starts
        at it and one worse, the primary hit (chosen among the best by a hash of the read), its strand, mapping
        quality, and (align) its alignment"""
        qbytes = np.ascontiguousarray(qbytes, dtype=np.uint8)
        qoff = np.ascontiguousarray(qoff, dtype=np.uint64)
        nq = len(qoff) - 1
        out = np.zeros(max(1, nq), dtype=MAPPING_DTYPE)
        aln = np.zeros(max(1, nq), dtype=ALIGNMENT_DTYPE) if align else None
        _check(native().awry_map_batch(self._h, qbytes.ctypes.data, qoff.ctypes.data, nq, _METRICS[metric],
                                       int(bool(strands)), int(max_dist), out.ctypes.data,
                                       aln.ctypes.data if align else None))
        return out[:nq], (aln[:nq] if align else None)

    def map_device(self, d_qbytes: int, d_qoff: int, nq: int, metric, max_dist: int, d_out: int, d_aln: int = None,
                   strands: bool = True, stream: int = 0, replica: int = 0):
        """map_packed on device pointers: d_out = nq x 32 bytes (MAPPING_DTYPE), d_aln = None or nq x 44 bytes
        (ALIGNMENT_DTYPE), both on the device.  Returns without waiting; see device_check"""
        _check(native().awry_map_device(self._h, replica, d_qbytes, d_qoff, nq, _METRICS[metric], int(bool(strands)),
                                        int(max_dist), d_out, d_aln, stream))

    # ---- streaming reads-file front-end (FASTQ / FASTA parsed on the device) ---------------
    def count_reads_file(self, path) -> np.ndarray:
        """parallel_count over every record of a FASTQ / FASTA file; read i of the file is entry i."""
        ptr, n = C.c_void_p(), C.c_uint64()
        _check(native().awry_count_reads_file(self._h, os.fsencode(path), C.byref(ptr), C.byref(n)))
        out = np.empty(n.value, dtype=np.uint64)
        if n.value:
            C.memmove(out.ctypes.data, ptr, n.value * 8)
        native().awry_buffer_free(ptr)
        return out

    def locate_reads_file(self, path, sorted_hits: bool = False):
        """parallel_locate over a FASTQ / FASTA file -> (hit_off uint64[n_reads+1], hits uint64[n_hits, 2])"""
        off_p, hits_p, n, nh = C.c_void_p(), C.c_void_p(), C.c_uint64(), C.c_uint64()
        _check(native().awry_locate_reads_file(self._h, os.fsencode(path),
                                               LOCATE_SORTED if sorted_hits else LOCATE_BWT_ORDER,
                                               C.byref(off_p), C.byref(hits_p), C.byref(n), C.byref(nh)))
        off = np.empty(n.value + 1, dtype=np.uint64)
        C.memmove(off.ctypes.data, off_p, (n.value + 1) * 8)
        hits = np.empty((nh.value, 2), dtype=np.uint64)
        if nh.value:
            C.memmove(hits.ctypes.data, hits_p, nh.value * 16)
        native().awry_buffer_free(off_p)
        native().awry_hits_free(hits_p)
        return off, hits

    def get_search_range_for_string(self, query) -> SearchRange:
        qb, qo = pack_queries([query])
        r = self.search_packed(qb, qo)[0]
        return SearchRange(int(r[0]), int(r[1]))

    def count_string(self, query) -> int:
        """FmIndex::count_string (fm_index.rs:499-501): a batch of one."""
        qb, qo = pack_queries([query])
        return int(self.count_packed(qb, qo)[0])

    def locate_string(self, query) -> List[LocalizedSequencePosition]:
        """FmIndex::locate_string (fm_index.rs:516-544): hits in BWT-row order."""
        qb, qo = pack_queries([query])
        _, hits = self.locate_packed(qb, qo)
        return [LocalizedSequencePosition(int(a), int(b)) for a, b in hits]

    def parallel_count(self, queries: Iterable) -> List[int]:
        """FmIndex::parallel_count (fm_index.rs:455-460); input order preserved."""
        qb, qo = pack_queries(queries)
        return [int(c) for c in self.count_packed(qb, qo)]

    def parallel_locate(self, queries: Iterable) -> List[List[LocalizedSequencePosition]]:
        """FmIndex::parallel_locate (fm_index.rs:479-487)."""
        qb, qo = pack_queries(queries)
        off, hits = self.locate_packed(qb, qo)
        out = []
        for i in range(len(qo) - 1):
            seg = hits[int(off[i]):int(off[i + 1])]
            out.append([LocalizedSequencePosition(int(a), int(b)) for a, b in seg])
        return out

    # ---- device-resident (raw device pointers, e.g. torch tensors' data_ptr()) -------------
    def count_device(self, d_qbytes: int, d_qoff: int, nq: int, d_counts: int, stream: int = 0,
                     replica: int = 0):
        _check(native().awry_count_device(self._h, replica, d_qbytes, d_qoff, nq, d_counts, stream))

    def locate_device(self, d_qbytes: int, d_qoff: int, nq: int, d_hit_off: int, sorted_hits=False,
                      stream: int = 0, replica: int = 0):
        """-> (device pointer to n_hits x {u64 seq_idx, u64 local_pos}, n_hits); free with device_free"""
        hits, n = C.c_void_p(), C.c_uint64()
        _check(native().awry_locate_device(self._h, replica, d_qbytes, d_qoff, nq,
                                           LOCATE_SORTED if sorted_hits else LOCATE_BWT_ORDER,
                                           d_hit_off, C.byref(hits), C.byref(n), stream))
        return hits.value, n.value

    def device_free(self, ptr: int, replica: int = 0):
        _check(native().awry_device_free(self._h, replica, ptr))

    def device_check(self, stream: int = 0, replica: int = 0):
        _check(native().awry_device_check(self._h, replica, stream))


def build_index_file(input_file_src, output_file_src, alphabet=SymbolAlphabet.Nucleotide,
                     suffix_array_compression_ratio: int = 0, lookup_table_kmer_len: int = 0, device: int = 0):
    """FmIndex::new + save on the GPU: FASTA/FASTQ -> `.awry` v1 file (load it with FmIndex.load)."""
    a = BuildArgs(os.fsencode(input_file_src), os.fsencode(output_file_src), int(alphabet),
                  int(lookup_table_kmer_len), int(suffix_array_compression_ratio), int(device))
    _check(native().awry_build_index_file(C.byref(a)))
    return output_file_src


def build_parts(alphabet: int, text, n: int = None, sa_ratio: int = 8, device: int = 0):
    """The construction pass of fm_index.rs:202-240 on the GPU.  `text`: uint8 numpy array (host) or an
    int device pointer (then `n` is required).  -> (blocks, prefix_sums, sa_words, phase seconds)"""
    L = native()
    if isinstance(text, int):
        ptr = text
    else:
        text = np.ascontiguousarray(text, dtype=np.uint8)
        ptr, n = text.ctypes.data, len(text)
    bwt_len = n + 1
    blocks = np.empty(L.awry_parts_num_blocks(bwt_len) * L.awry_parts_block_words(int(alphabet)), dtype=np.uint64)
    prefix = np.zeros(7 if int(alphabet) == 0 else 23, dtype=np.uint64)
    sa_words = np.empty(L.awry_parts_sa_words(bwt_len, sa_ratio), dtype=np.uint64)
    phases = np.zeros(8, dtype=np.float64)
    _check(L.awry_build_parts(int(alphabet), ptr, n, sa_ratio, device, blocks.ctypes.data, prefix.ctypes.data,
                              sa_words.ctypes.data, phases.ctypes.data))
    names = ["ingest", "keys", "sort", "ties", "bwt", "milestones", "sa_pack_copy", "total"]
    return blocks, prefix, sa_words, dict(zip(names, [float(x) for x in phases]))


def profile_enable(on: bool):
    _check(native().awry_profile_enable(1 if on else 0))


def profile_reset():
    _check(native().awry_profile_reset())


def profile_get() -> dict:
    p = Profile()
    _check(native().awry_profile_get(C.byref(p)))
    return p.as_dict()


def bench_random_gather(device: int, footprint_bytes: int, granule: int, lanes: int, n_reads: int,
                        iters: int = 3):
    r, g = C.c_double(), C.c_double()
    _check(native().awry_bench_random_gather(device, footprint_bytes, granule, lanes, n_reads, iters,
                                             C.byref(r), C.byref(g)))
    return r.value, g.value


def set_search_variant(lanes: int = 0, tpb: int = 0, blocks_per_sm: int = 0):
    _check(native().awry_set_search_variant(lanes, tpb, blocks_per_sm))


def set_count_variant(variant: int = 0):
    """0 = nucleotide counts finish one-row intervals by comparing with the text (when the index holds the
    unsampled suffix array and the text); 1 = backward search to the last symbol.  Same counts either way."""
    _check(native().awry_set_count_variant(variant))


def set_locate_variant(variant: int = 0):
    """0 = the best pass 2 the index holds (unsampled-SA gather, else the bounded walk on the position-sampled
    array, else the LF-walk); 1 = always LF-walk to the file's row samples; 2 = the bounded walk if present."""
    _check(native().awry_set_locate_variant(variant))


def set_host_pack(mode: int = -1):
    """-1 = auto, 0 = send ASCII queries over PCIe, 1 = pack nucleotide queries to 2 bits on the host first."""
    _check(native().awry_set_host_pack(mode))


def set_host_threads(n: int = 0):
    """threads of the host-side packer pool (0 = default: min(16, cores / LOCAL_WORLD_SIZE))"""
    _check(native().awry_set_host_threads(int(n)))


def host_threads() -> int:
    return int(native().awry_host_threads())


def host_pack_dna(src: np.ndarray):
    """the host packer alone (tests): -> (crumb bytes uint8[ceil(n/4)], exceptions uint64[] = (i << 8) | byte)"""
    src = np.ascontiguousarray(src, dtype=np.uint8)
    dst = np.zeros((len(src) + 3) // 4 + 64, dtype=np.uint8)
    exc = np.zeros(min(len(src), 1 << 20) + 1, dtype=np.uint64)
    n = C.c_uint64()
    _check(native().awry_host_pack_dna(src.ctypes.data, len(src), dst.ctypes.data, exc.ctypes.data, len(exc), C.byref(n)))
    if n.value > len(exc):          # more exceptions than the first guess: once more with room for all
        exc = np.zeros(n.value, dtype=np.uint64)
        _check(native().awry_host_pack_dna(src.ctypes.data, len(src), dst.ctypes.data, exc.ctypes.data, len(exc), C.byref(n)))
    return dst[: (len(src) + 3) // 4], exc[: n.value]


def read_sequence_file(path, alphabet: int = 0):
    """libsufr's read_sequence_file as the builder sees it: -> (text uint8[], record starts uint64[])"""
    tp, sp, n, nr = C.c_void_p(), C.c_void_p(), C.c_uint64(), C.c_uint64()
    _check(native().awry_read_sequence_file(os.fsencode(path), int(alphabet), C.byref(tp), C.byref(n), C.byref(sp),
                                            C.byref(nr)))
    text = np.empty(n.value, dtype=np.uint8)
    starts = np.empty(nr.value, dtype=np.uint64)
    if n.value:
        C.memmove(text.ctypes.data, tp, n.value)
    if nr.value:
        C.memmove(starts.ctypes.data, sp, nr.value * 8)
    native().awry_buffer_free(tp)
    native().awry_buffer_free(sp)
    return text, starts
