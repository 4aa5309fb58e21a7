"""CPU tests of the alignment boundary (awry_align_batch, awry_align_device, awry_alignment_cigar): argument errors are
reported before any device is touched, the numpy record matches the C layout, the CIGAR of hand-built alignments, the
C++ mirror compiles, and the brute-force reference the GPU tests compare with (tests/align_brute.c) agrees with an
exhaustive enumeration of every alignment of tiny strings.  The alignments themselves run in tests/test_gpu_align.py."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from conftest import ROOT


def lib():
    from awry_b200 import fm_index as f
    return f.native()


def last_error():
    return lib().awry_last_error().decode()


def test_bad_arguments_need_no_device():
    L = lib()
    qb = np.frombuffer(b"ACGTACGT", np.uint8).copy()
    qo = np.array([0, 8], np.uint64)
    off = np.array([0, 1, 1], np.uint64)
    hits = np.zeros((1, 2), np.uint64)
    out = np.zeros(44, np.uint8)
    fake = C.c_void_p(1)                                    # never dereferenced: the arguments fail first

    def batch(ix=None, qbp=qb.ctypes.data, qop=qo.ctypes.data, nq=1, metric=0, strands=0, k=1, offp=off.ctypes.data,
              hp=hits.ctypes.data, op=out.ctypes.data):
        return L.awry_align_batch(ix, qbp, qop, nq, metric, strands, k, offp, hp, op)

    def device(ix=None, replica=0, qbp=qb.ctypes.data, qop=qo.ctypes.data, nq=1, metric=0, strands=0, k=1,
               offp=off.ctypes.data, hp=hits.ctypes.data, n=1, op=out.ctypes.data):
        return L.awry_align_device(ix, replica, qbp, qop, nq, metric, strands, k, offp, hp, n, op, None)

    for call in (batch, device):
        assert call() == -1 and "null" in last_error()                       # null index
        for k in (4, 7, 1 << 31):
            assert call(ix=fake, k=k) == -1 and "0 .. 3" in last_error(), k
        assert call(ix=fake, metric=1, k=5) == -1 and "max_edits" in last_error()
        for m in (2, 99):
            assert call(ix=fake, metric=m) == -1 and "metric" in last_error(), m
        assert call(ix=fake, strands=2) == -1 and "strands" in last_error()
        assert call(ix=fake, offp=None) == -1 and "null" in last_error()
        assert call(ix=fake, qbp=None) == -1 and "null" in last_error()
        assert call(ix=fake, hp=None) == -1 and "null" in last_error()
        assert call(ix=fake, op=None) == -1 and "null" in last_error()
        assert call(nq=0) == -1                                              # an empty batch still needs an index
    # the host call checks its hit offsets
    qo2 = np.array([0, 4, 8], np.uint64)
    bad = np.array([0, 2, 1], np.uint64)
    assert batch(ix=fake, qop=qo2.ctypes.data, nq=2, offp=bad.ctypes.data) == -1 and "monotone" in last_error()
    bad = np.array([1, 1, 1], np.uint64)
    assert batch(ix=fake, offp=bad.ctypes.data) == -1 and "hit_off[0]" in last_error()
    two = np.array([0, 1, 1, 1, 1], np.uint64)                               # both strands: 2 nq + 1 offsets
    bad = np.array([0, 1, 0, 1, 1], np.uint64)
    assert batch(ix=fake, strands=1, offp=bad.ctypes.data) == -1 and "monotone" in last_error()
    assert batch(strands=1, offp=two.ctypes.data) == -1 and "null" in last_error()


def test_alignment_record_matches_the_header(tmp_path):
    from awry_b200 import fm_index as f
    src = tmp_path / "al.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "awry_b200.h"\nint main(void){'
                   'printf("%zu %zu %zu %zu %zu %zu %zu %zu %zu %zu\\n", sizeof(awry_alignment), sizeof(awry_edit_op), '
                   'offsetof(awry_alignment, distance), offsetof(awry_alignment, n_ops), offsetof(awry_alignment, ops), '
                   'offsetof(awry_edit_op, tpos), offsetof(awry_edit_op, op), offsetof(awry_edit_op, query_sym), '
                   'offsetof(awry_edit_op, text_sym), (size_t)AWRY_METRIC_EDIT);return 0;}\n')
    exe = tmp_path / "al"
    subprocess.check_call(["gcc", "-std=c99", "-Wall", "-Werror", "-pedantic", "-I", os.path.join(ROOT, "include"),
                           str(src), "-o", str(exe)])
    got = [int(x) for x in subprocess.check_output([str(exe)]).split()]
    d, o = f.ALIGNMENT_DTYPE, f.EDIT_OP_DTYPE
    assert got == [d.itemsize, o.itemsize, d.fields["distance"][1], d.fields["n_ops"][1], d.fields["ops"][1],
                   o.fields["tpos"][1], o.fields["op"][1], o.fields["query_sym"][1], o.fields["text_sym"][1],
                   f.METRIC_EDIT]


def record(ops, text_len=0):
    from awry_b200 import fm_index as f
    a = np.zeros((), f.ALIGNMENT_DTYPE)
    a["text_len"] = text_len
    a["distance"] = a["n_ops"] = len(ops)
    for t, (q, tp, op) in enumerate(ops):
        a["ops"][t] = (q, tp, ord(op), 0 if op == "D" else ord("A"), 0 if op == "I" else ord("C"), 0)
    return a


def test_cigar_of_hand_built_alignments():
    from awry_b200 import AwryError
    from awry_b200 import fm_index as f
    assert f.cigar(record([]), 150) == "150="
    assert f.cigar(record([(47, 47, "X")]), 150) == "47=1X102="
    assert f.cigar(record([(0, 0, "X"), (9, 9, "X")]), 10) == "1X8=1X"               # ops at both ends
    assert f.cigar(record([(0, 0, "I"), (9, 8, "I")]), 10) == "1I8=1I"
    assert f.cigar(record([(0, 0, "D"), (9, 10, "D")]), 10) == "1D9=1D1="             # D in front of the first / last
    assert f.cigar(record([(3, 3, "X"), (4, 4, "X"), (5, 5, "X")]), 10) == "3=3X4="    # adjacent ops merge
    assert f.cigar(record([(3, 3, "I"), (4, 3, "I")]), 10) == "3=2I5="
    assert f.cigar(record([(3, 3, "D"), (3, 4, "D")]), 10) == "3=2D7="
    assert f.cigar(record([(3, 3, "I"), (4, 3, "D")]), 10) == "3=1I1D6="               # I then D
    assert f.cigar(record([(3, 3, "D"), (3, 4, "X")]), 10) == "3=1D1X6="
    assert f.cigar(record([(2, 2, "X"), (5, 5, "I"), (7, 6, "D")]), 8) == "2=1X2=1I1=1D1="
    # capacity: AWRY_ERR_CAPACITY with the full size in *needed
    a = record([(47, 47, "X")])
    need = C.c_size_t()
    for cap in (0, 1, 9):
        buf = C.create_string_buffer(max(cap, 1))
        assert lib().awry_alignment_cigar(a.ctypes.data, 150, buf, cap, C.byref(need)) == -8
        assert need.value == len("47=1X102=") + 1
    buf = C.create_string_buffer(10)
    assert lib().awry_alignment_cigar(a.ctypes.data, 150, buf, 10, C.byref(need)) == 0 and buf.value == b"47=1X102="
    assert lib().awry_alignment_cigar(a.ctypes.data, 150, buf, 10, None) == 0
    # not alignments
    none = np.zeros((), f.ALIGNMENT_DTYPE)
    none["distance"] = 3                                                            # "no alignment within k = 2"
    for bad, ln in ((none, 10), (record([(5, 5, "X"), (3, 3, "X")]), 10), (record([(10, 10, "X")]), 10),
                    (record([(1, 1, "Q")]), 10)):
        with pytest.raises(AwryError) as e:
            f.cigar(bad, ln)
        assert e.value.code == -1
    assert lib().awry_alignment_cigar(None, 10, buf, 10, None) == -1


def test_cxx_mirror_align_methods_compile(tmp_path):
    src = tmp_path / "al.cpp"
    src.write_text("""#include "awry_b200.hpp"
#include <cstdio>
int main() {
  try {
    awry::FmIndex ix = awry::FmIndex::load("x.awry");
    std::vector<uint64_t> off{0, 1};
    std::vector<awry_hit> hits{awry_hit{0, 5}};
    auto al = ix.align_hits({"ACGTACGTAC"}, AWRY_METRIC_EDIT, 2, off, hits);
    std::printf("%s %u\\n", awry::FmIndex::cigar(al[0], 10).c_str(), al[0].text_len);
    return 0;
  } catch (const awry::Error& e) {
    return e.code;
  }
}
""")
    subprocess.check_call(["g++", "-std=c++17", "-Wall", "-Wextra", "-Werror", "-fsyntax-only", "-I",
                           os.path.join(ROOT, "include"), str(src)])


# ---- the reference against exhaustive enumeration -------------------------------------------------------------------

ORDER = {"=": 0, "X": 1, "I": 2, "D": 3}


def all_alignments(q, t):
    """every alignment of q (all of it) against a prefix of t: (ops string, [(op, i, j)])"""
    out = []

    def go(i, j, ops, at):
        if i == len(q):
            out.append(("".join(ops), list(at)))
        if i < len(q) and j < len(t):
            op = "=" if q[i] == t[j] else "X"
            go(i + 1, j + 1, ops + [op], at + ([] if op == "=" else [("X", i, j)]))
        if i < len(q):
            go(i + 1, j, ops + ["I"], at + [("I", i, j)])
        if j < len(t):
            go(i, j + 1, ops + ["D"], at + [("D", i, j)])
    go(0, 0, [], [])
    return out


def want_edit(q, t, k):
    best = None
    for ops, at in all_alignments(q, t):
        cost = len(at)
        key = (cost, [ORDER[c] for c in ops])
        if cost <= k and (best is None or key < best[0]):
            best = (key, ops, at)
    return best


def test_brute_force_reference_equals_exhaustive_enumeration(tmp_path, po):
    so = str(tmp_path / "libalign_brute.so")
    subprocess.check_call(["gcc", "-O2", "-fopenmp", "-shared", "-fPIC", "-o", so, os.path.join(ROOT, "tests", "align_brute.c")])
    B = C.CDLL(so)
    B.align_brute_one.restype = C.c_uint32
    B.align_brute_one.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint64, C.c_void_p, C.c_uint64, C.c_uint32,
                                  C.c_uint32, C.c_void_p]
    lut = np.array([po.lib().awo_ascii_to_index(0, c) for c in range(256)], dtype=np.uint8)
    letters = "$ACGNT"
    r = np.random.default_rng(17)
    out = np.zeros(44, np.uint8)
    checked = {0: 0, 1: 0}
    for trial in range(1500):
        alpha = b"ACGN" if trial % 5 == 0 else (b"AC" if trial % 3 == 0 else b"ACGT")
        n = int(r.integers(1, 10))
        text = bytes(r.choice(np.frombuffer(alpha, np.uint8), n))
        L = int(r.integers(1, 7))
        k = int(r.integers(0, 4))
        s = int(r.integers(0, n))
        q = bytearray(text[s:s + L]) if r.random() < 0.6 else bytearray()
        while len(q) < L:
            q.append(int(r.choice(np.frombuffer(alpha, np.uint8))))
        for _ in range(int(r.integers(0, 3))):
            q[int(r.integers(0, L))] = int(r.choice(np.frombuffer(alpha, np.uint8)))
        q = bytes(q[:L])
        tb, qb = np.frombuffer(text, np.uint8).copy(), np.frombuffer(q, np.uint8).copy()
        tsym, qsym = [int(lut[c]) for c in text], [int(lut[c]) for c in q]
        for metric in (0, 1):
            d = B.align_brute_one(lut.ctypes.data, tb.ctypes.data, n, s, qb.ctypes.data, L, metric, k, out.ctypes.data)
            rec = out.copy()
            text_len = int(rec[:4].view(np.uint32)[0])
            ops = [(chr(rec[16 + 12 * t]), int(rec[8 + 12 * t:12 + 12 * t].view(np.uint32)[0]),
                    int(rec[12 + 12 * t:16 + 12 * t].view(np.uint32)[0]), rec[17 + 12 * t], rec[18 + 12 * t])
                   for t in range(int(rec[5]))]
            what = (trial, text, s, q, k, metric)
            if L <= k:                                                      # refused
                assert d == k + 1 and not rec[5] and text_len == 0, what
                continue
            if metric == 0:
                win = tsym[s:s + L]
                mm = [i for i in range(L) if len(win) == L and qsym[i] != win[i]]
                if len(win) < L or len(mm) > k:
                    assert d == k + 1 and rec[4] == k + 1 and not rec[5:].any() and text_len == 0, what
                else:
                    assert d == len(mm) == rec[4] == rec[5] and text_len == L, what
                    assert [(o, i, j) for o, i, j, _, _ in ops] == [("X", i, i) for i in mm], what
                    checked[0] += 1
            else:
                best = want_edit(qsym, tsym[s:], k)
                if best is None:
                    assert d == k + 1 and rec[4] == k + 1 and not rec[5:].any() and text_len == 0, what
                else:
                    (cost, _), opstr, at = best
                    assert d == cost == rec[4] == rec[5], (what, opstr, d)
                    assert [(o, i, j) for o, i, j, _, _ in ops] == at, (what, opstr, ops)
                    assert text_len == sum(1 for c in opstr if c != "I"), (what, opstr)
                    for o, i, j, qs, ts in ops:
                        assert qs == (0 if o == "D" else ord(letters[qsym[i]])), what
                        assert ts == (0 if o == "I" else ord(letters[tsym[s + j]])), what
                checked[metric] += best is not None
            assert not rec[6:8].any() and all(not rec[19 + 12 * t] for t in range(3)), what   # pad bytes
            assert not rec[8 + 12 * int(rec[5]):].any(), what                                   # unused ops
    assert min(checked.values()) > 150, checked


def test_exhaustive_enumeration_itself():
    """the enumeration the reference is checked against: a few cases worked by hand"""
    sym = {"A": 1, "C": 2, "G": 3, "T": 5}
    enc = lambda x: [sym[c] for c in x]                                     # noqa: E731
    assert want_edit(enc("ACGT"), enc("ACGT"), 0)[1] == "===="
    assert want_edit(enc("ACGT"), enc("AGT"), 1)[1] == "=I=="               # C inserted in the query
    assert want_edit(enc("AGT"), enc("ACGT"), 1)[1] == "=D=="               # C deleted from the query
    assert want_edit(enc("AAC"), enc("ACC"), 1)[1] == "=X="                 # X sorts before I / D
    assert want_edit(enc("ACGT"), enc("TTTT"), 1) is None
    assert sorted(a for a, _ in all_alignments([1], [1])) == sorted(["=", "I", "ID", "DI"])
