"""CPU tests of the edit-distance search boundary (awry_*_edit[_strands]): argument errors are reported before any
device is touched, the C++ mirror's methods compile cleanly, and the brute-force reference the GPU tests compare with
(tests/edit_brute.c) agrees with a plain Levenshtein DP.  The searches themselves run in tests/test_gpu_edit.py."""
import ctypes as C
import os
import subprocess

import numpy as np

from conftest import ROOT

SINGLE = ("awry_count_batch_edit", "awry_locate_batch_edit", "awry_count_device_edit")
BOTH = ("awry_count_batch_edit_strands", "awry_locate_batch_edit_strands", "awry_count_device_edit_strands")


def test_bad_arguments_need_no_device():
    from awry_b200 import fm_index as f
    lib = f.native()
    qb = np.frombuffer(b"ACGTACGT", np.uint8).copy()
    qo = np.array([0, 8], np.uint64)
    counts = np.zeros(16, np.uint64)
    off = np.zeros(3, np.uint64)
    hits = np.zeros((4, 2), np.uint64)
    ed = np.zeros(4, np.uint8)
    n = C.c_uint64()
    for count, locate, device in (SINGLE, BOTH):
        count, locate, device = getattr(lib, count), getattr(lib, locate), getattr(lib, device)
        # null index
        assert count(None, qb.ctypes.data, qo.ctypes.data, 1, 1, counts.ctypes.data) == -1
        assert locate(None, qb.ctypes.data, qo.ctypes.data, 1, 1, off.ctypes.data, hits.ctypes.data, ed.ctypes.data, 4,
                      C.byref(n)) == -1
        assert device(None, 0, qb.ctypes.data, qo.ctypes.data, 1, 1, counts.ctypes.data, None) == -1
        # null buffers
        assert count(None, None, None, 1, 1, None) == -1
        assert locate(None, None, None, 1, 1, None, None, None, 0, None) == -1
        assert device(None, 0, None, None, 1, 1, None, None) == -1
        assert b"null" in lib.awry_last_error()
        # k > AWRY_EDIT_MAX
        for k in (4, 7, 1 << 31):
            assert count(None, qb.ctypes.data, qo.ctypes.data, 1, k, counts.ctypes.data) == -1
            assert locate(None, qb.ctypes.data, qo.ctypes.data, 1, k, off.ctypes.data, hits.ctypes.data,
                          ed.ctypes.data, 4, C.byref(n)) == -1
            assert device(None, 0, qb.ctypes.data, qo.ctypes.data, 1, k, counts.ctypes.data, None) == -1
        # an empty batch still needs an index
        assert count(None, None, None, 0, 1, None) == -1
        assert locate(None, None, None, 0, 1, off.ctypes.data, None, None, 0, C.byref(n)) == -1
        assert device(None, 0, None, None, 0, 1, None, None) == -1


def test_cxx_mirror_edit_methods_compile(tmp_path):
    src = tmp_path / "ed.cpp"
    src.write_text("""#include "awry_b200.hpp"
#include <cstdio>
int main() {
  try {
    awry::FmIndex ix = awry::FmIndex::load("x.awry");
    auto counts = ix.parallel_count_edit({"ACGTACGTAC", "GATTACA"}, 2);
    auto hits = ix.parallel_locate_edit({"ACGTACGTAC"}, AWRY_EDIT_MAX);
    for (auto& h : hits[0])
      std::printf("%llu %llu %u\\n", (unsigned long long)h.first.sequence_idx(),
                  (unsigned long long)h.first.local_position(), h.second);
    auto both = ix.parallel_count_edit_strands({"ACGTACGTAC"}, 1);
    auto both_hits = ix.parallel_locate_edit_strands({"ACGTACGTAC"}, 3);
    for (int strand = 0; strand < 2; strand++)
      for (auto& h : both_hits[0][strand]) std::printf("%d %u\\n", strand, h.second);
    return int(counts[0].size() + both[0][1].size());
  } catch (const awry::Error& e) {
    return e.code;
  }
}
""")
    subprocess.check_call(["g++", "-std=c++17", "-Wall", "-Wextra", "-Werror", "-fsyntax-only", "-I",
                           os.path.join(ROOT, "include"), str(src)])


def levenshtein_start(text, s, q):
    """d(s) = min over l of ed(q, text[s .. s+l)), plain full DP"""
    n, L = len(text), len(q)
    prev = list(range(n - s + 1))               # row 0: D[0][j] = j
    for i in range(1, L + 1):
        cur = [i] + [0] * (n - s)
        for j in range(1, n - s + 1):
            cur[j] = min(prev[j - 1] + (q[i - 1] != text[s + j - 1]), prev[j] + 1, cur[j - 1] + 1)
        prev = cur
    return min(prev)


def test_brute_force_reference_equals_plain_dp(tmp_path, po):
    so = str(tmp_path / "libedit_brute.so")
    subprocess.check_call(["gcc", "-O2", "-fopenmp", "-shared", "-fPIC", "-o", so, os.path.join(ROOT, "tests", "edit_brute.c")])
    L = C.CDLL(so)
    L.edit_brute.restype = C.c_int64
    L.edit_brute.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint32,
                             C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    lut = np.array([po.lib().awo_ascii_to_index(0, c) for c in range(256)], dtype=np.uint8)
    r = np.random.default_rng(3)
    for trial in range(24):
        n = int(r.integers(1, 70))
        text = bytes(r.choice(np.frombuffer(b"ACGTN" if trial % 3 == 0 else b"ACGT", np.uint8), n))
        if trial % 4 == 1:
            text = b"A" * (n // 2) + text[n // 2:]       # a homopolymer run
        k = trial % 4
        qs = []
        for _ in range(12):
            ln = int(r.integers(k + 1, 14))
            if r.random() < 0.6 and n > ln:           # a window of the text with random edits
                p = int(r.integers(0, n - ln))
                q = bytearray(text[p:p + ln])
                for _ in range(int(r.integers(0, k + 2))):
                    at, op = int(r.integers(0, len(q))), int(r.integers(0, 3))
                    if op == 0:
                        q[at] = ord("ACGT"[int(r.integers(0, 4))])
                    elif op == 1:
                        q.insert(at, ord("ACGT"[int(r.integers(0, 4))]))
                    elif len(q) > k + 1:
                        del q[at]
                qs.append(bytes(q))
            else:
                qs.append(bytes(r.choice(np.frombuffer(b"ACGTn", np.uint8), ln)))
        qb = np.frombuffer(b"".join(qs), np.uint8).copy()
        qo = np.zeros(len(qs) + 1, np.uint64)
        qo[1:] = np.cumsum([len(q) for q in qs])
        tb = np.frombuffer(text, np.uint8).copy()
        counts = np.zeros((len(qs), k + 1), np.uint64)
        off = np.zeros(len(qs) + 1, np.uint64)
        args = (lut.ctypes.data, tb.ctypes.data, n, qb.ctypes.data, qo.ctypes.data, len(qs), k, counts.ctypes.data,
                off.ctypes.data)
        total = L.edit_brute(*args, None, None)
        pos = np.zeros(max(1, total), np.uint64)
        dist = np.zeros(max(1, total), np.uint8)
        L.edit_brute(*args, pos.ctypes.data, dist.ctypes.data)
        tsym = [int(lut[b]) for b in text]
        for qi, q in enumerate(qs):
            qsym = [int(lut[b]) for b in q]
            want = [(s, d) for s in range(n) for d in [levenshtein_start(tsym, s, qsym)] if d <= k]
            got = [(int(pos[i]), int(dist[i])) for i in range(int(off[qi]), int(off[qi + 1]))]
            assert got == want, (trial, text, q, k)
            assert [sum(1 for _, d in want if d == e) for e in range(k + 1)] == counts[qi].tolist()
