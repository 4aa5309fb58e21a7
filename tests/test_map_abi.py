"""CPU tests of read mapping (awry_map_batch, awry_map_device): argument errors are reported before any device is
touched, the record is 32 bytes and MAPPING_DTYPE matches it, the header's mapping-quality table equals its formula,
the read hash maps bytes as the header says, and the Python reference `ref_map` that tests/test_gpu_map.py applies to
brute-force and library hit lists agrees with a literal per-read statement of the rules.  The mapping itself runs in
tests/test_gpu_map.py."""
import ctypes as C
import math
import os
import re
import subprocess

import numpy as np

from conftest import ROOT

M64 = (1 << 64) - 1
CODE = bytes(0 if c in b"Aa" else 1 if c in b"Cc" else 2 if c in b"Gg" else 3 if c in b"TtUu" else 4
             for c in range(256))


def read_hash(q: bytes) -> int:
    """fmix64(FNV-1a-64 over the codes of the read's bytes), as include/awry_b200.h states it"""
    h = 0xcbf29ce484222325
    for b in q:
        h = ((h ^ CODE[b]) * 0x100000001b3) & M64
    h ^= h >> 33
    h = (h * 0xff51afd7ed558ccd) & M64
    h ^= h >> 33
    h = (h * 0xc4ceb9fe1a85ec53) & M64
    return h ^ (h >> 33)


def mapq(n_best, n_second, best, k):
    if n_best != 1:
        return 0
    if best == k:
        return 25
    if n_second == 0:
        return 37
    return max(0, 23 - math.floor(4.343 * math.log(min(n_second, 255)) + 0.5))


def refused(q: bytes, k: int) -> bool:
    return len(q) <= k or b"$" in q or b"#" in q


REF_DTYPE = np.dtype([("start", "<u8"), ("n_best", "<u4"), ("n_second", "<u4"), ("distance", "u1"), ("strand", "u1"),
                      ("mapq", "u1"), ("flags", "u1")])


def ref_map(hit_off, starts, dists, reads, k, strands):
    """the records of include/awry_b200.h from each virtual query's hit set: hit_off ((nq << strands) + 1), global
    starts and distances of the hits (H_v: Hamming windows, or edit loci), the reads as given -> REF_DTYPE[nq], with the
    primary's global start (~0 when unmapped) in place of (seq_idx, local_pos)"""
    per = 2 if strands else 1
    hit_off = np.asarray(hit_off, np.int64)
    starts = np.asarray(starts, np.uint64)
    dists = np.asarray(dists, np.int64)
    out = np.zeros(len(reads), REF_DTYPE)
    for q, read in enumerate(reads):
        r = out[q]
        a, b = int(hit_off[per * q]), int(hit_off[per * q + per])
        if refused(read, k) or a == b:
            r["start"], r["distance"] = M64, k + 1
            r["flags"] = 1 | (2 if refused(read, k) else 0)
            continue
        s = starts[a:b]
        strand = np.zeros(b - a, np.int64)
        if strands:
            strand[int(hit_off[2 * q + 1]) - a:] = 1
        key = dists[a:b] * 2 + strand
        order = np.lexsort((key, s))
        s, key = s[order], key[order]
        first = np.ones(len(s), bool)
        first[1:] = s[1:] != s[:-1]
        s, d, st = s[first], key[first] >> 1, key[first] & 1
        best = int(d.min())
        at_best = np.nonzero(d == best)[0]
        n_second = int((d == best + 1).sum()) if best < k else 0
        i = at_best[read_hash(read) % len(at_best)]
        r["start"], r["distance"], r["strand"] = s[i], best, st[i]
        r["n_best"], r["n_second"] = len(at_best), n_second
        r["mapq"] = mapq(len(at_best), n_second, best, k)
    return out


def literal(groups, read, k):
    """the rules read literally over one read: groups = one {start: distance} per searched strand"""
    if refused(read, k):
        return (M64, 0, 0, k + 1, 0, 0, 3)
    D = {}
    for strand, g in enumerate(groups):
        for s, d in g.items():
            if s not in D or (d, strand) < D[s]:
                D[s] = (d, strand)
    if not D:
        return (M64, 0, 0, k + 1, 0, 0, 1)
    best = min(d for d, _ in D.values())
    B = sorted(s for s, (d, _) in D.items() if d == best)
    n_second = len([s for s, (d, _) in D.items() if d == best + 1]) if best < k else 0
    p = B[read_hash(read) % len(B)]
    return (p, len(B), n_second, best, D[p][1], mapq(len(B), n_second, best, k), 0)


def run(reads, per_read_groups, k, strands):
    """per_read_groups: per read, one {start: distance} per strand -> ref_map's records as tuples"""
    off, starts, dists = [0], [], []
    for groups in per_read_groups:
        for g in groups:
            for s in r_shuffle(g):
                starts.append(s)
                dists.append(g[s])
            off.append(len(starts))
    got = ref_map(off, np.array(starts, np.uint64), np.array(dists, np.int64), reads, k, strands)
    return [tuple(int(x) for x in r) for r in got]


def r_shuffle(g):
    """the hits of one query in ascending start, as the locate calls return them"""
    return sorted(g)


def test_reference_equals_the_literal_rules_on_random_hits():
    r = np.random.default_rng(23)
    for trial in range(500):
        k = trial % 4
        strands = bool(trial & 4)
        reads, groups = [], []
        for _ in range(int(r.integers(1, 6))):
            ln = int(r.integers(0, 12))
            reads.append(bytes(np.frombuffer(b"ACGTNacgtuRY$", np.uint8)[r.integers(0, 12 if trial % 5 else 13, ln)]))
            span = int(r.integers(1, 30))
            gs = []
            for _ in range(2 if strands else 1):
                st = r.choice(span, int(r.integers(0, min(span, 8) + 1)), replace=False)
                gs.append({int(s): int(r.integers(0, k + 1)) for s in st})
            groups.append(gs)
        assert run(reads, groups, k, strands) == [literal(g, q, k) for g, q in zip(groups, reads)], (trial, groups)


def test_hand_built_cases():
    q = b"ACGTACGTAC"
    # a palindromic start on both strands at one distance counts once, on strand 0
    assert run([q], [[{5: 1}, {5: 1}]], 2, True)[0] == (5, 1, 0, 1, 0, 37, 0)
    # ... and the better strand wins when the distances differ
    assert run([q], [[{5: 2}, {5: 1}]], 2, True)[0] == (5, 1, 0, 1, 1, 37, 0)
    # equal distance on both strands at different starts: two best starts, mapq 0, the hash picks
    rec = run([q], [[{3: 1}, {9: 1}]], 2, True)[0]
    assert rec[1:4] == (2, 0, 1) and rec[5] == 0 and rec[0] == [3, 9][read_hash(q) % 2]
    assert rec[4] == (0 if rec[0] == 3 else 1)
    # best = k: n_second is 0 (that stratum was not searched) and mapq 25
    assert run([q], [[{4: 2}]], 2, False)[0] == (4, 1, 0, 2, 0, 25, 0)
    # one worse start gives 23, a few give less
    assert run([q], [[{4: 0, 40: 1}]], 2, False)[0] == (4, 1, 1, 0, 0, 23, 0)
    assert run([q], [[{4: 0, 40: 1, 50: 1, 60: 1}]], 2, False)[0][5] == 18
    # no hits: unmapped; a refused read: unmapped and refused, whatever its hits
    assert run([q], [[{}, {}]], 1, True)[0] == (M64, 0, 0, 2, 0, 0, 1)
    assert run([b"AC$GT"], [[{4: 0}]], 1, False)[0] == (M64, 0, 0, 2, 0, 0, 3)
    assert run([b"A"], [[{4: 0}]], 1, False)[0] == (M64, 0, 0, 2, 0, 0, 3)
    assert run([b""], [[{}]], 0, False)[0] == (M64, 0, 0, 1, 0, 0, 3)
    # n_second > 255 is capped in the table: mapq 0
    many = {s: 1 for s in range(100, 100 + 300)}
    assert run([q], [[{7: 0} | many]], 3, False)[0] == (7, 1, 300, 0, 0, 0, 0)
    # the primary is B[h mod n_best] in ascending start, whatever the strand
    B = list(range(10, 80, 7))
    rec = run([q], [[{s: 1 for s in B[::2]}, {s: 1 for s in B[1::2]}]], 3, True)[0]
    assert rec[0] == B[read_hash(q) % len(B)] and rec[1] == len(B)


def test_hash_maps_bytes_as_specified():
    base = read_hash(b"ACGTACGTTN")
    for same in (b"acgtacgttn", b"ACGUACGUUN", b"acguACGTtR", b"ACGTACGTTY", b"ACGTACGTT*", b"AcGtAcGuUk"):
        assert read_hash(same) == base, same
    assert read_hash(b"ACGTACGTTA") != base and read_hash(b"ACGTACGTT") != base
    assert read_hash(b"AC") != read_hash(b"CA")                  # the order matters: it is the read as given
    # an independent statement: the header's rule compiled as C
    words = [b"", b"A", b"ACGTACGTTN", b"acguRYKMnn$", b"TTTTTTTTTTTTTTTTTTTTTTTTTTTTTTTTTTTTTTTTTTTTTTTTTTTTTTTTT"]
    assert c_hashes(words) == [read_hash(w) for w in words]


C_HASH = r"""#include <stdio.h>
#include <stdint.h>
#include <string.h>
static unsigned code(unsigned char c) {
  switch (c) {
    case 'A': case 'a': return 0;
    case 'C': case 'c': return 1;
    case 'G': case 'g': return 2;
    case 'T': case 't': case 'U': case 'u': return 3;
    default: return 4;
  }
}
int main(int argc, char** argv) {
  for (int i = 1; i < argc; i++) {
    uint64_t x = 0xcbf29ce484222325ull;
    for (size_t j = 0; j < strlen(argv[i]); j++) x = (x ^ code((unsigned char)argv[i][j])) * 0x100000001b3ull;
    x ^= x >> 33; x *= 0xff51afd7ed558ccdull; x ^= x >> 33; x *= 0xc4ceb9fe1a85ec53ull; x ^= x >> 33;
    printf("%llu\n", (unsigned long long)x);
  }
  return 0;
}
"""


def c_hashes(words):
    import tempfile
    with tempfile.TemporaryDirectory() as d:
        src, exe = os.path.join(d, "h.c"), os.path.join(d, "h")
        with open(src, "w") as f:
            f.write(C_HASH)
        subprocess.check_call(["gcc", "-O1", "-o", exe, src])
        return [int(x) for x in subprocess.check_output([exe] + [w.decode() for w in words]).split()]


def test_mapq_table_equals_the_formula():
    text = open(os.path.join(ROOT, "include", "awry_b200.h")).read()
    body = re.search(r"#define AWRY_MAPQ_SECOND\s*\\\s*\{([^}]*)\}", text).group(1)
    table = [int(x) for x in body.replace("\\", "").split(",")]
    assert len(table) == 256
    assert table[0] == 37
    for n in range(1, 256):
        g = math.floor(4.343 * math.log(n) + 0.5)
        assert abs(4.343 * math.log(n) + 0.5 - round(4.343 * math.log(n) + 0.5)) > 0.002   # no rounding tie
        assert table[n] == max(0, 23 - g), n
        assert mapq(1, n, 0, 3) == table[n]


def test_record_layout():
    from awry_b200 import fm_index as f

    class Hit(C.Structure):
        _fields_ = [("seq_idx", C.c_uint64), ("local_pos", C.c_uint64)]

    class Mapping(C.Structure):
        _fields_ = [("hit", Hit), ("n_best", C.c_uint32), ("n_second", C.c_uint32), ("distance", C.c_uint8),
                    ("strand", C.c_uint8), ("mapq", C.c_uint8), ("flags", C.c_uint8), ("pad", C.c_uint32)]

    assert C.sizeof(Mapping) == 32 == f.MAPPING_DTYPE.itemsize
    for name in ("n_best", "n_second", "distance", "strand", "mapq", "flags", "pad"):
        assert getattr(Mapping, name).offset == f.MAPPING_DTYPE.fields[name][1], name
    assert f.MAPPING_DTYPE.fields["seq_idx"][1] == 0 and f.MAPPING_DTYPE.fields["local_pos"][1] == 8
    assert (f.MAP_UNMAPPED, f.MAP_REFUSED) == (1, 2)


def test_bad_arguments_need_no_device():
    from awry_b200 import fm_index as f
    lib = f.native()
    qb = np.frombuffer(b"ACGTACGT", np.uint8).copy()
    qo = np.array([0, 8], np.uint64)
    out = np.zeros(2, f.MAPPING_DTYPE)
    aln = np.zeros(2, f.ALIGNMENT_DTYPE)

    def both(ix=None, qbp=qb.ctypes.data, qop=qo.ctypes.data, nq=1, metric=0, strands=0, k=1, replica=0, outs=True):
        o = out.ctypes.data if outs else None
        return (lib.awry_map_batch(ix, qbp, qop, nq, metric, strands, k, o, aln.ctypes.data),
                lib.awry_map_device(ix, replica, qbp, qop, nq, metric, strands, k, o, None, None))

    for metric in (2, 7, 1 << 31):                           # metric, strands and k are checked first
        assert both(metric=metric) == (-1, -1), metric
        assert b"metric" in lib.awry_last_error()
    for strands in (2, 1 << 31):
        assert both(strands=strands) == (-1, -1), strands
        assert b"strands" in lib.awry_last_error()
    for metric in (0, 1):
        for k in (4, 9, 1 << 31):
            assert both(metric=metric, k=k) == (-1, -1), (metric, k)
        for strands in (0, 1):
            assert both(metric=metric, strands=strands) == (-1, -1)                          # null index
            assert both(metric=metric, strands=strands, qbp=None, qop=None, outs=False) == (-1, -1)
            assert both(metric=metric, strands=strands, nq=0, qbp=None, qop=None) == (-1, -1)  # still needs an index
            assert both(metric=metric, strands=strands, replica=-1) == (-1, -1)


def test_cxx_mirror_map_compiles(tmp_path):
    src = tmp_path / "map.cpp"
    src.write_text("""#include "awry_b200.hpp"
#include <cstdio>
int main() {
  try {
    awry::FmIndex ix = awry::FmIndex::load("x.awry");
    auto [recs, alns] = ix.parallel_map({"ACGTACGTAC", "GATTACA"}, AWRY_METRIC_EDIT, 2);
    for (size_t q = 0; q < recs.size(); q++) {
      const awry_mapping& m = recs[q];
      if (m.flags & AWRY_MAP_UNMAPPED) continue;
      std::printf("%llu %llu %u %u %u %s\\n", (unsigned long long)m.hit.seq_idx, (unsigned long long)m.hit.local_pos,
                  m.distance, m.strand, m.mapq, awry::FmIndex::cigar(alns[q], 10).c_str());
    }
    auto fwd = ix.parallel_map({"ACGTACGTAC"}, AWRY_METRIC_HAMMING, 1, false, false);
    return int(fwd.first.size() + fwd.second.size());
  } catch (const awry::Error& e) {
    return e.code;
  }
}
""")
    subprocess.check_call(["g++", "-std=c++17", "-Wall", "-Wextra", "-Werror", "-fsyntax-only", "-I",
                           os.path.join(ROOT, "include"), str(src)])
    # the C header alone, as C
    csrc = tmp_path / "map.c"
    csrc.write_text('#include "awry_b200.h"\nstatic const unsigned char t[256] = AWRY_MAPQ_SECOND;\n'
                    'int main(void) { awry_mapping m = {0}; return (int)sizeof m + t[0] - 69; }\n')
    subprocess.check_call(["gcc", "-std=c99", "-Wall", "-Wextra", "-Werror", "-fsyntax-only", "-I",
                           os.path.join(ROOT, "include"), str(csrc)])
