"""CPU tests of edit-distance search by locus (awry_*_edit_loci): argument errors are reported before any device is
touched, the C++ mirror's methods compile cleanly, and the reference filter `loci` that tests/test_gpu_edit_loci.py
applies to the brute-force hits agrees with a literal restatement of the header's rules (a) and (b) on random hit
lists and on hand-built cases.  The searches themselves run in tests/test_gpu_edit_loci.py."""
import ctypes as C
import os
import subprocess

import numpy as np

from conftest import ROOT


def loci(hit_off, pos, dist, k):
    """the locus filter of include/awry_b200.h on hits sorted per query: hit_off (nv + 1), global starts `pos`
    (ascending within a query) and distances `dist` -> (hit_off, keep) with keep a bool mask over the hits.  A hit is
    a locus unless (a) a hit of its query within k has a smaller distance, or (b) its distance is >= 1 and the start
    just before it is a hit at the same distance."""
    hit_off = np.asarray(hit_off, np.int64)
    pos = np.asarray(pos, np.int64)
    dist = np.asarray(dist, np.int64)
    keep = np.ones(len(pos), bool)
    for v in range(len(hit_off) - 1):
        a, b = int(hit_off[v]), int(hit_off[v + 1])
        p, d = pos[a:b], dist[a:b]
        for j in range(1, k + 1):                      # the neighbour j places to the left / right
            if b - a <= j:
                break
            near = p[j:] - p[:-j] <= k                 # pairs (i - j, i) within k
            keep[a + j:b] &= ~(near & (d[:-j] < d[j:]))
            keep[a:b - j] &= ~(near & (d[j:] < d[:-j]))
            if j == 1:
                keep[a + 1:b] &= ~((p[1:] - p[:-1] == 1) & (d[1:] == d[:-1]) & (d[1:] > 0))
    off = np.zeros(len(hit_off), np.uint64)
    off[1:] = np.cumsum([keep[int(hit_off[v]):int(hit_off[v + 1])].sum() for v in range(len(hit_off) - 1)])
    return off, keep


def literal(hits, k):
    """rules (a) and (b) read literally, O(n^2), over one query's hits {start: distance}"""
    return sorted(s for s, d in hits.items()
                  if not any(0 < abs(t - s) <= k and e < d for t, e in hits.items())
                  and not (d >= 1 and hits.get(s - 1) == d))


def run(groups, k):
    """groups: one {start: distance} per query -> the loci of each query through `loci`"""
    off = np.zeros(len(groups) + 1, np.uint64)
    off[1:] = np.cumsum([len(g) for g in groups])
    pos = np.array([s for g in groups for s in sorted(g)], np.int64)
    dist = np.array([g[s] for g in groups for s in sorted(g)], np.int64)
    new_off, keep = loci(off, pos, dist, k)
    kept = pos[keep]
    return [kept[int(new_off[v]):int(new_off[v + 1])].tolist() for v in range(len(groups))]


def test_reference_equals_the_literal_rules_on_random_hits():
    r = np.random.default_rng(17)
    for trial in range(400):
        k = trial % 4
        groups = []
        for _ in range(int(r.integers(1, 5))):
            span = int(r.integers(1, 40))
            starts = r.choice(span, int(r.integers(0, span + 1)), replace=False)
            groups.append({int(s): int(r.integers(0, k + 1)) for s in starts})
        assert run(groups, k) == [literal(g, k) for g in groups], (trial, k, groups)


def test_hand_built_cases():
    # a plateau: one locus, at its leftmost start; a strictly better start within k removes it
    assert run([{10: 1, 11: 1, 12: 1, 13: 1}], 2) == [[10]]
    assert run([{10: 2, 11: 2, 12: 1, 13: 2}], 1) == [[10, 12]]
    # a homopolymer of exact hits: all stay, and their shifted copies go
    assert run([{s: 0 for s in range(20, 26)} | {19: 1, 26: 1}], 1) == [list(range(20, 26))]
    # two exact hits exactly k and k + 1 apart, with the shifted starts between them
    for k in (1, 2, 3):
        assert run([{0: 0, k: 0}], k) == [[0, k]]
        assert run([{0: 0, k + 1: 0}], k) == [[0, k + 1]]
        between = {s: 1 for s in range(1, k + 1)} | {0: 0, k + 1: 0}
        assert run([between], k) == [[0, k + 1]]
    # a chain d = 2, 1, 0 spaced k apart: each is within k of a better one
    for k in (1, 2, 3):
        assert run([{0: 2, k: 1, 2 * k: 0}], k) == [[2 * k]]
        assert run([{0: 2, k + 1: 1, 2 * k + 2: 0}], k) == [[0, k + 1, 2 * k + 2]]
    # adjacent queries never interact: the same starts are judged per query
    assert run([{5: 0}, {6: 1}, {7: 1}, {}], 3) == [[5], [6], [7], []]
    # k = 0: every hit is a locus
    assert run([{3: 0, 4: 0, 9: 0}], 0) == [[3, 4, 9]]


SINGLE = ("awry_count_batch_edit_loci", "awry_locate_batch_edit_loci", "awry_count_device_edit_loci",
          "awry_locate_device_edit_loci")


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
    dh, dd = C.c_void_p(), C.c_void_p()
    count, locate, dcount, dlocate = (getattr(lib, s) for s in SINGLE)

    def all_four(ix=None, qbp=qb.ctypes.data, qop=qo.ctypes.data, nq=1, strands=0, k=1, replica=0, outs=True):
        return (count(ix, qbp, qop, nq, strands, k, counts.ctypes.data if outs else None),
                locate(ix, qbp, qop, nq, strands, k, off.ctypes.data if outs else None, hits.ctypes.data if outs else None,
                       ed.ctypes.data, 4, C.byref(n) if outs else None),
                dcount(ix, replica, qbp, qop, nq, strands, k, counts.ctypes.data if outs else None, None),
                dlocate(ix, replica, qbp, qop, nq, strands, k, off.ctypes.data if outs else None,
                        C.byref(dh) if outs else None, C.byref(dd), C.byref(n) if outs else None, None))

    for strands in (2, 3, 1 << 31):                      # strands is 0 or 1, checked first
        assert all_four(strands=strands) == (-1,) * 4, strands
        assert b"strands" in lib.awry_last_error()
    for strands in (0, 1):
        assert all_four(strands=strands) == (-1,) * 4     # null index
        for k in (4, 7, 1 << 31):                        # k > AWRY_EDIT_MAX
            assert all_four(strands=strands, k=k) == (-1,) * 4, k
        assert all_four(strands=strands, qbp=None, qop=None, outs=False) == (-1,) * 4
        assert all_four(strands=strands, nq=0, qbp=None, qop=None) == (-1,) * 4   # an empty batch still needs an index
        assert all_four(strands=strands, replica=-1) == (-1,) * 4


def test_cxx_mirror_loci_methods_compile(tmp_path):
    src = tmp_path / "loci.cpp"
    src.write_text("""#include "awry_b200.hpp"
#include <cstdio>
int main() {
  try {
    awry::FmIndex ix = awry::FmIndex::load("x.awry");
    auto counts = ix.parallel_count_edit_loci({"ACGTACGTAC", "GATTACA"}, 2);
    auto hits = ix.parallel_locate_edit_loci({"ACGTACGTAC"}, AWRY_EDIT_MAX);
    for (auto& h : hits[0])
      std::printf("%llu %llu %u\\n", (unsigned long long)h.first.sequence_idx(),
                  (unsigned long long)h.first.local_position(), h.second);
    auto both = ix.parallel_count_edit_loci_strands({"ACGTACGTAC"}, 1);
    auto both_hits = ix.parallel_locate_edit_loci_strands({"ACGTACGTAC"}, 3);
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
