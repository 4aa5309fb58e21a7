"""CPU tests of the both-strand Hamming-search boundary (awry_*_hamming_strands): argument errors are reported before
any device is touched, and the C++ mirror's methods compile cleanly.  The searches themselves run in
tests/test_gpu_hamming_strands.py."""
import ctypes as C
import os
import subprocess

import numpy as np

from conftest import ROOT


def test_bad_arguments_need_no_device():
    from awry_b200 import fm_index as f
    lib = f.native()
    qb = np.frombuffer(b"ACGTACGT", np.uint8).copy()
    qo = np.array([0, 8], np.uint64)
    counts = np.zeros(16, np.uint64)
    off = np.zeros(3, np.uint64)
    hits = np.zeros((4, 2), np.uint64)
    mm = np.zeros(4, np.uint8)
    n = C.c_uint64()
    assert lib.awry_count_batch_hamming_strands(None, qb.ctypes.data, qo.ctypes.data, 1, 1, counts.ctypes.data) == -1
    assert lib.awry_locate_batch_hamming_strands(None, qb.ctypes.data, qo.ctypes.data, 1, 1, off.ctypes.data,
                                                 hits.ctypes.data, mm.ctypes.data, 4, C.byref(n)) == -1
    assert lib.awry_count_device_hamming_strands(None, 0, qb.ctypes.data, qo.ctypes.data, 1, 1, counts.ctypes.data,
                                                 None) == -1
    # null buffers
    assert lib.awry_count_batch_hamming_strands(None, None, None, 1, 1, None) == -1
    assert lib.awry_locate_batch_hamming_strands(None, None, None, 1, 1, None, None, None, 0, None) == -1
    assert lib.awry_count_device_hamming_strands(None, 0, None, None, 1, 1, None, None) == -1
    assert b"null" in lib.awry_last_error()
    # k > AWRY_HAMMING_MAX
    for k in (4, 7, 1 << 31):
        assert lib.awry_count_batch_hamming_strands(None, qb.ctypes.data, qo.ctypes.data, 1, k, counts.ctypes.data) == -1
        assert lib.awry_locate_batch_hamming_strands(None, qb.ctypes.data, qo.ctypes.data, 1, k, off.ctypes.data,
                                                     hits.ctypes.data, mm.ctypes.data, 4, C.byref(n)) == -1
        assert lib.awry_count_device_hamming_strands(None, 0, qb.ctypes.data, qo.ctypes.data, 1, k,
                                                     counts.ctypes.data, None) == -1
    # an empty batch still needs an index
    assert lib.awry_count_batch_hamming_strands(None, None, None, 0, 1, None) == -1
    assert lib.awry_locate_batch_hamming_strands(None, None, None, 0, 1, off.ctypes.data, None, None, 0,
                                                 C.byref(n)) == -1
    assert lib.awry_count_device_hamming_strands(None, 0, None, None, 0, 1, None, None) == -1


def test_cxx_mirror_hamming_strand_methods_compile(tmp_path):
    src = tmp_path / "hs.cpp"
    src.write_text("""#include "awry_b200.hpp"
#include <cstdio>
int main() {
  try {
    awry::FmIndex ix = awry::FmIndex::load("x.awry");
    auto counts = ix.parallel_count_hamming_strands({"ACGTACGTAC", "GATTACA"}, 2);
    auto hits = ix.parallel_locate_hamming_strands({"ACGTACGTAC"}, AWRY_HAMMING_MAX);
    for (int strand = 0; strand < 2; strand++)
      for (auto& h : hits[0][strand])
        std::printf("%d %llu %llu %u\\n", strand, (unsigned long long)h.first.sequence_idx(),
                    (unsigned long long)h.first.local_position(), h.second);
    return int(counts[0][0].size() + counts[0][1].size());
  } catch (const awry::Error& e) {
    return e.code;
  }
}
""")
    subprocess.check_call(["g++", "-std=c++17", "-Wall", "-Wextra", "-Werror", "-fsyntax-only", "-I",
                           os.path.join(ROOT, "include"), str(src)])
