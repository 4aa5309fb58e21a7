"""Hamming search on both strands (awry_*_hamming_strands): query q stands for the virtual queries 2q (q) and 2q + 1
(its reverse complement, as include/awry_b200.h defines it).  Strand 0 must equal the single-strand Hamming calls on q
and strand 1 those calls on rc(q), and both must equal a brute-force scan over every window of the text
(tests/hamming_brute.c): counts per distance, hit lists in text order and each hit's distance, k = 1, 2, 3.  Reads of
every length k+1 .. 300 and up to 600 cross every alignment of the piece boundaries against the 16-symbol word and the
64-byte unit, which is where the piece words are cut from the reads' words; reads are drawn from both strands with
planted substitutions, with lowercase / U / N / IUPAC bytes, and as palindromes.  k = 0 equals exact search on both
strands; the device entry point equals the batch call; refused batches name the caller's query as the single-strand
calls do."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT, device_from_parts, mixed_queries
from test_gpu_hamming import brute, brute_lib, hamming_queries, multi, multi_dev, repeats, substitute  # noqa: F401
from test_gpu_strands import rc

pytestmark = pytest.mark.gpu


def pack(qs):
    from awry_b200 import fm_index as f
    return f.pack_queries(qs)


def unpack(qb, qo):
    return [bytes(qb[int(qo[i]):int(qo[i + 1])]) for i in range(len(qo) - 1)]


def interleave(fwd, rev):
    """two single-strand results (counts, hit_off, hits, mismatches) -> the both-strand layout"""
    cf, of, hf, df = fwd
    cr, orr, hr, dr = rev
    nq = len(of) - 1
    counts = np.stack([cf, cr], axis=1)
    lens = np.stack([np.diff(of.astype(np.int64)), np.diff(orr.astype(np.int64))], axis=1).ravel()
    off = np.zeros(2 * nq + 1, np.uint64)
    off[1:] = np.cumsum(lens).astype(np.uint64)
    hits, dist = [], []
    for q in range(nq):
        hits += [hf[int(of[q]):int(of[q + 1])], hr[int(orr[q]):int(orr[q + 1])]]
        dist += [df[int(of[q]):int(of[q + 1])], dr[int(orr[q]):int(orr[q + 1])]]
    hits = np.concatenate(hits).reshape(-1, 2) if hits else np.zeros((0, 2), np.uint64)
    dist = np.concatenate(dist) if dist else np.zeros(0, np.uint8)
    return counts, off, hits.astype(np.uint64), dist.astype(np.uint8)


def assert_both_strands(dev, parts, qs, k, brute_lib, single=True):  # noqa: F811
    """the both-strand calls against brute force on q and rc(q) (and, with `single`, against the single-strand calls)"""
    qb, qo = pack(qs)
    rb, ro = pack([rc(q) for q in qs])
    want = interleave(brute(brute_lib, parts, qb, qo, k), brute(brute_lib, parts, rb, ro, k))
    if single:
        one = interleave((dev.count_hamming_packed(qb, qo, k),) + dev.locate_hamming_packed(qb, qo, k),
                         (dev.count_hamming_packed(rb, ro, k),) + dev.locate_hamming_packed(rb, ro, k))
        for a, b in zip(one, want):
            assert np.array_equal(a, b), k
    got = dev.count_hamming_strands_packed(qb, qo, k)
    bad = np.nonzero((got != want[0]).any(axis=(1, 2)))[0]
    assert len(bad) == 0, (k, bad[:5], got[bad[:5]], want[0][bad[:5]])
    goff, ghits, gd = dev.locate_hamming_strands_packed(qb, qo, k)
    assert np.array_equal(goff, want[1]), k
    assert np.array_equal(ghits, want[2]) and np.array_equal(gd, want[3]), k
    return want


def reverse_strand_reads(parts, k, seed, n=600):
    """rc(window with m = 0 .. k+1 planted substitutions) -> (reads, m)"""
    r = np.random.default_rng(seed)
    t = bytes(parts.text)
    qs, ms = [], []
    for i in range(n):
        ln = int(r.integers(k + 1, 300)) if i % 4 else int(r.integers(k + 1, 40))
        p = int(r.integers(0, len(t) - ln))
        q = bytearray(t[p:p + ln])
        m = i % (k + 2)
        cuts = [j * ln // (k + 1) for j in range(k + 2)]
        kind = (i // (k + 2)) % 4
        if kind == 0:
            at = r.choice(ln, size=min(m, ln), replace=False)
        elif kind == 1:                                  # one in each of the first m pieces
            at = [int(r.integers(cuts[j], cuts[j + 1])) for j in range(min(m, k + 1))]
        elif kind == 2:                                  # at piece boundaries
            at = sorted(set(min(ln - 1, c) for c in cuts[1:]))[:m]
        else:                                            # first and last symbol
            at = [0, ln - 1][:m]
        for a in at:
            substitute(q, int(a), r)
        qs.append(rc(bytes(q)))
        ms.append(len(set(int(a) for a in at)))
    return qs, np.array(ms)


def length_sweep(parts, k, seed):
    """one read of every length k+1 .. 300 at a random start (with a substitution in every other one), and a few up
    to 600; every third is reverse-complemented"""
    r = np.random.default_rng(seed)
    t = bytes(parts.text)
    qs = []
    for i, ln in enumerate(list(range(k + 1, 301)) + [301, 319, 320, 321, 383, 384, 385, 447, 511, 512, 513, 599, 600]):
        p = int(r.integers(0, len(t) - ln))
        q = bytearray(t[p:p + ln])
        if i % 2:
            substitute(q, int(r.integers(0, ln)), r)
        qs.append(rc(bytes(q)) if i % 3 == 0 else bytes(q))
    return qs


@pytest.mark.parametrize("k", [1, 2, 3])
def test_both_strands_equal_single_strand_and_brute_force(k, multi, multi_dev, brute_lib):  # noqa: F811
    qs = unpack(*hamming_queries(multi, k, seed=200 + k, n_random=900))
    qs = [rc(q) if i % 2 else q for i, q in enumerate(qs)]   # true hits on both strands
    qs += length_sweep(multi, k, seed=300 + k)
    rev, ms = reverse_strand_reads(multi, k, seed=400 + k)
    qs += rev
    counts = assert_both_strands(multi_dev, multi, qs, k, brute_lib)[0]
    assert all((counts[:, s, d] > 0).sum() > 30 for s in (0, 1) for d in range(k + 1)), k
    # a read from the reverse strand with m <= k substitutions is found there at distance <= m
    rc_counts = counts[len(qs) - len(rev):, 1]
    for i, m in enumerate(ms):
        if m <= k:
            assert rc_counts[i, :m + 1].sum() >= 1, (k, i, m)


def test_k0_equals_exact_search_on_both_strands(fx):
    text = fx.gen_text(0, 200_000, 31)
    parts = fx.build_parts(text, 0, ratio=8, kmer_len=8)
    qb, qo = mixed_queries(fx, parts.text, 4000, 24, seed=2)
    qs = unpack(qb, qo)
    qb, qo = pack([rc(q) if i % 2 else q for i, q in enumerate(qs)])
    with device_from_parts(parts) as ix:
        counts = ix.count_hamming_strands_packed(qb, qo, 0)
        assert np.array_equal(counts[:, :, 0], ix.count_strands_packed(qb, qo))
        off, hits = ix.locate_strands_packed(qb, qo, sorted_hits=True)
        hoff, hhits, hd = ix.locate_hamming_strands_packed(qb, qo, 0)
        assert np.array_equal(hoff, off) and np.array_equal(hhits, hits) and not hd.any()


def test_bytes_and_palindromes(fx, brute_lib):  # noqa: F811
    r = np.random.default_rng(8)
    base = bytearray(fx.gen_text(0, 150_000, 56).tobytes())
    pals = []
    for i in range(200):
        s = bytes(r.choice(list(b"ACGT"), size=int(r.integers(4, 90))).astype(np.uint8))
        p = s + rc(s)
        pals.append(p)
        at = int(r.integers(0, len(base) - len(p)))
        base[at:at + len(p)] = p
    parts = fx.build_parts(bytes(base), 0, ratio=8, kmer_len=9)
    qs = list(pals)
    for i in range(300):                                 # lowercase, U, N and IUPAC bytes anywhere, ends included
        ln = int(r.integers(10, 260))
        p = int(r.integers(0, len(base) - ln))
        q = bytearray(base[p:p + ln])
        for _ in range(i % 3):
            q[int(r.choice([0, ln - 1, int(r.integers(0, ln))]))] = ord("NRYnykU"[int(r.integers(0, 7))])
        if i % 4 == 1:
            q = bytearray(bytes(q).lower())
        if i % 5 == 2:
            q = bytearray(bytes(q).replace(b"T", b"U").replace(b"t", b"u"))
        qs.append(rc(bytes(q)) if i % 2 else bytes(q))
    with device_from_parts(parts) as ix:
        for k in (1, 2):
            assert_both_strands(ix, parts, qs, k, brute_lib)
            off, hits, dist = ix.locate_hamming_strands_packed(*pack(pals), k)
            for q in range(len(pals)):                   # nothing deduplicated: the same windows on both strands
                fwd = slice(int(off[2 * q]), int(off[2 * q + 1]))
                rev = slice(int(off[2 * q + 1]), int(off[2 * q + 2]))
                assert np.array_equal(hits[fwd], hits[rev]) and np.array_equal(dist[fwd], dist[rev]), (k, q)


def test_repeat_rich_text_and_tiny_slices(repeats, brute_lib, monkeypatch):  # noqa: F811
    parts, ix, qb, qo = repeats
    qs = unpack(qb, qo)
    qs = [rc(q) if i % 2 else q for i, q in enumerate(qs)]
    want = assert_both_strands(ix, parts, qs, 2, brute_lib, single=False)
    assert np.diff(want[1].astype(np.int64)).max() >= 200
    monkeypatch.setenv("AWRY_B200_HAMMING_SLICE", "16")
    got = ix.count_hamming_strands_packed(*pack(qs), 2)
    assert np.array_equal(got, want[0])
    goff, ghits, gd = ix.locate_hamming_strands_packed(*pack(qs), 2)
    assert np.array_equal(goff, want[1]) and np.array_equal(ghits, want[2]) and np.array_equal(gd, want[3])


def err(call):
    from awry_b200 import AwryError
    with pytest.raises(AwryError) as e:
        call()
    return e.value.code, str(e.value)


def test_errors_name_the_callers_query(fx, multi, multi_dev, monkeypatch):  # noqa: F811
    from awry_b200 import fm_index as f
    t = bytes(multi.text)
    reads = [t[100 + 7 * i:160 + 7 * i] for i in range(8)]
    cases = [(k, 5, t[:k]) for k in (1, 2, 3)] + [(2, 5, b""), (1, 5, b"AC$GT"), (2, 5, b"#"), (3, 0, b"ACGTACGT$"),
                                                  (1, 7, b"")]
    for k, at, bad in cases:
        qs = list(reads)
        qs[at] = bad
        qb, qo = pack(qs)
        single = err(lambda: multi_dev.count_hamming_packed(qb, qo, k))
        assert single[0] == -5 and "query %d" % at in single[1], single
        assert err(lambda: multi_dev.count_hamming_strands_packed(qb, qo, k)) == single, (k, at, bad)
        assert err(lambda: multi_dev.locate_hamming_strands_packed(qb, qo, k)) == \
            err(lambda: multi_dev.locate_hamming_packed(qb, qo, k)), (k, at, bad)
    qb, qo = pack(reads)
    for at, val in ((3, 10**6), (6, 0)):                 # offsets that are not monotone
        o = qo.copy()
        o[at] = val
        single = err(lambda: multi_dev.count_hamming_packed(qb, o, 1))
        assert err(lambda: multi_dev.count_hamming_strands_packed(qb, o, 1)) == single
        assert err(lambda: multi_dev.locate_hamming_strands_packed(qb, o, 1))[0] == single[0]
    assert err(lambda: multi_dev.count_hamming_strands_packed(qb, qo, 4))[0] == -1
    assert err(lambda: multi_dev.locate_hamming_strands_packed(qb, qo, 4))[0] == -1
    # too small a buffer: the offsets are complete, and the retry gives the same hits
    qs = unpack(*hamming_queries(multi, 1, seed=3, n_random=300))
    qs = [rc(q) if i % 2 else q for i, q in enumerate(qs)]
    qb, qo = pack(qs)
    nq = len(qo) - 1
    hoff, hits, dist = multi_dev.locate_hamming_strands_packed(qb, qo, 1, capacity=nq * 200)
    off = np.zeros(2 * nq + 1, np.uint64)
    small = np.zeros((5, 2), np.uint64)
    mm = np.zeros(5, np.uint8)
    n = C.c_uint64()
    rc_ = f.native().awry_locate_batch_hamming_strands(multi_dev.handle, qb.ctypes.data, qo.ctypes.data, nq, 1,
                                                       off.ctypes.data, small.ctypes.data, mm.ctypes.data, 5, C.byref(n))
    assert rc_ == -8 and n.value == len(hits) and np.array_equal(off, hoff)
    assert np.array_equal(small, hits[:5]) and np.array_equal(mm, dist[:5])
    assert np.array_equal(multi_dev.locate_hamming_strands_packed(qb, qo, 1, capacity=3)[1], hits)
    assert np.array_equal(multi_dev.count_hamming_strands_packed(qb, qo, 1)[:, 0],
                          multi_dev.count_hamming_packed(qb, qo, 1))   # no sticky error
    # indexes the search does not exist for
    import torch
    prot = fx.build_parts(fx.gen_text(1, 20_000, 3), 1, ratio=8, kmer_len=3)
    with device_from_parts(prot) as ix:
        pq = pack([b"ACDEFG"])
        assert err(lambda: ix.count_hamming_strands_packed(*pq, 1))[0] == -6
        assert err(lambda: ix.locate_hamming_strands_packed(*pq, 1))[0] == -6
        d = torch.zeros(16, dtype=torch.int64, device="cuda")
        assert err(lambda: ix.count_hamming_strands_device(d.data_ptr(), d.data_ptr(), 1, 1, d.data_ptr()))[0] == -6
    dna = fx.gen_text(0, 30_000, 3)
    parts = fx.build_parts(dna, 0, ratio=8, kmer_len=8)
    monkeypatch.setenv("AWRY_B200_TEXT", "0")
    with device_from_parts(parts) as ix:
        dq = pack([bytes(dna[:40])])
        assert err(lambda: ix.count_hamming_strands_packed(*dq, 1))[0] == -6
        assert err(lambda: ix.locate_hamming_strands_packed(*dq, 1))[0] == -6


def test_device_entry_point(multi, multi_dev):  # noqa: F811
    import torch
    qs = unpack(*hamming_queries(multi, 3, seed=12, n_random=800))
    qs = [rc(q) if i % 2 else q for i, q in enumerate(qs)]
    qb, qo = pack(qs)
    nq = len(qo) - 1
    want = multi_dev.count_hamming_strands_packed(qb, qo, 3)
    d_qb = torch.from_numpy(np.concatenate([np.zeros(3, np.uint8), qb])).cuda()
    d_qo = torch.from_numpy(qo.view(np.int64)).cuda()
    st = torch.cuda.current_stream().cuda_stream
    d_counts = torch.full((nq, 2, 4), 7, dtype=torch.int64, device="cuda")
    multi_dev.count_hamming_strands_device(d_qb.data_ptr() + 3, d_qo.data_ptr(), nq, 3, d_counts.data_ptr(), st)
    multi_dev.device_check(st)
    assert np.array_equal(d_counts.cpu().numpy().view(np.uint64), want)
    # a refused read is latched under the caller's index, as the single-strand call latches it; its counts are 0
    t = bytes(multi.text)
    for bad in (b"ACG", b"", b"AC$GTACGT"):
        qb2, qo2 = pack([t[500:600], t[700:760], t[800:850], t[900:940], t[1000:1100], bad, t[1200:1260]])
        d_qb, d_qo = torch.from_numpy(qb2 if len(qb2) else np.zeros(1, np.uint8)).cuda(), \
            torch.from_numpy(qo2.view(np.int64)).cuda()
        d_counts = torch.full((7, 2, 4), 9, dtype=torch.int64, device="cuda")
        multi_dev.count_hamming_strands_device(d_qb.data_ptr(), d_qo.data_ptr(), 7, 3, d_counts.data_ptr(), st)
        both = err(lambda: multi_dev.device_check(st))
        d_one = torch.zeros((7, 4), dtype=torch.int64, device="cuda")
        multi_dev.count_hamming_device(d_qb.data_ptr(), d_qo.data_ptr(), 7, 3, d_one.data_ptr(), st)
        one = err(lambda: multi_dev.device_check(st))
        assert both == one and both[0] == -5 and "query 5" in both[1], (bad, both, one)
        got = d_counts.cpu().numpy()
        assert np.array_equal(got[:, 0], d_one.cpu().numpy()), bad
        assert got[0, 0, 0] >= 1 and got[6, 0, 0] >= 1, bad
        if len(bad) <= 3:                                # no pieces to search: nothing is counted
            assert not got[5].any(), bad
        multi_dev.device_check(st)


def test_several_replicas_equal_one(multi, multi_dev):  # noqa: F811
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    qs = unpack(*hamming_queries(multi, 2, seed=21, n_random=800))
    qs = [rc(q) if i % 2 else q for i, q in enumerate(qs)]
    qb, qo = pack(qs)
    want_c = multi_dev.count_hamming_strands_packed(qb, qo, 2)
    want_l = multi_dev.locate_hamming_strands_packed(qb, qo, 2)
    ix = device_from_parts(multi, devices=[0, 1])
    try:
        assert np.array_equal(ix.count_hamming_strands_packed(qb, qo, 2), want_c)
        for a, b in zip(ix.locate_hamming_strands_packed(qb, qo, 2), want_l):
            assert np.array_equal(a, b)
    finally:
        ix.close()


def test_on_the_bounds_checked_build():
    """this file against libawry_b200_checked.so (every data-dependent load bounds-checked, layout.cuh): no assert"""
    checked = os.path.join(ROOT, "awry_b200", "libawry_b200_checked.so")
    if os.environ.get("AWRY_B200_LIB"):
        pytest.skip("already running against another build")
    if not os.path.exists(checked):
        subprocess.check_call(["make", "-s", "-C", os.path.join(ROOT, "awry_b200", "csrc"), "checked"])
    env = dict(os.environ, AWRY_B200_LIB=checked)
    out = subprocess.run([sys.executable, "-m", "pytest", "tests/test_gpu_hamming_strands.py", "-m", "gpu", "-x", "-q",
                          "-p", "no:cacheprovider", "-k", "not bounds_checked and not several_replicas"],
                         cwd=ROOT, env=env, capture_output=True, text=True, timeout=1800)
    tail = out.stdout[-1500:] + out.stderr[-1500:]
    assert out.returncode == 0, tail
    assert " passed" in out.stdout and "Assertion" not in out.stderr, tail
