"""CPU tests of the both-strand boundary (awry_*_strands): argument errors are reported before any device is touched,
and the C++ mirror's methods compile cleanly.  The searches themselves run in tests/test_gpu_strands.py."""
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
    counts = np.zeros(2, np.uint64)
    off = np.zeros(3, np.uint64)
    hits = np.zeros((4, 2), np.uint64)
    hp = C.c_void_p()
    n = C.c_uint64()
    assert lib.awry_count_batch_strands(None, qb.ctypes.data, qo.ctypes.data, 1, counts.ctypes.data) == -1
    assert lib.awry_locate_batch_strands(None, qb.ctypes.data, qo.ctypes.data, 1, 0, off.ctypes.data, hits.ctypes.data, 4,
                                         C.byref(n)) == -1
    assert lib.awry_count_device_strands(None, 0, qb.ctypes.data, qo.ctypes.data, 1, counts.ctypes.data, None) == -1
    assert lib.awry_locate_device_strands(None, 0, qb.ctypes.data, qo.ctypes.data, 1, 0, off.ctypes.data, C.byref(hp),
                                          C.byref(n), None) == -1
    # null buffers
    assert lib.awry_count_batch_strands(None, None, None, 1, None) == -1
    assert lib.awry_locate_batch_strands(None, None, None, 1, 0, None, None, 0, None) == -1
    assert lib.awry_count_device_strands(None, 0, None, None, 1, None, None) == -1
    assert lib.awry_locate_device_strands(None, 0, None, None, 1, 0, None, None, None, None) == -1
    assert b"null" in lib.awry_last_error()


def test_cxx_mirror_strand_methods_compile(tmp_path):
    src = tmp_path / "s.cpp"
    src.write_text("""#include "awry_b200.hpp"
#include <cstdio>
int main() {
  try {
    awry::FmIndex ix = awry::FmIndex::load("x.awry");
    auto counts = ix.parallel_count_strands({"ACGTACGTAC", "GATTACA"});
    auto hits = ix.parallel_locate_strands({"ACGTACGTAC"}, true);
    for (int strand = 0; strand < 2; strand++)
      for (auto& h : hits[0][strand])
        std::printf("%d %llu %llu\\n", strand, (unsigned long long)h.sequence_idx(), (unsigned long long)h.local_position());
    return int(counts[0][0] + counts[0][1]);
  } catch (const awry::Error& e) {
    return e.code;
  }
}
""")
    subprocess.check_call(["g++", "-std=c++17", "-Wall", "-Wextra", "-Werror", "-fsyntax-only", "-I",
                           os.path.join(ROOT, "include"), str(src)])
