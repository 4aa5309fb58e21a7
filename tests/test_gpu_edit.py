"""GPU parity of the edit-distance search (awry_*_edit[_strands]): text starts within k <= 3 substitutions, insertions
and deletions, found from the k + 1 exactly searched pieces of the Hamming pipeline and verified by a banded DP on the
device.  Every result is compared bit for bit with a brute-force DP at every start of the text (tests/edit_brute.c,
symbols mapped by the oracle's awo_ascii_to_index): counts by distance, hit offsets, hits in text order and each hit's
distance, k = 1, 2, 3.  Inputs: a multi-record text with N runs; reads of every length k+1 .. 300 and up to 600 with
0 .. k+1 planted substitutions, insertions and deletions (anywhere, at piece boundaries, at the first and last
symbol); homopolymer indels; lowercase / U / N / IUPAC bytes; reads hanging over either end of the text; a
repeat-rich text with tandem arrays of period 1 .. 3 verified 16 key slots at a time.  Also: k = 0 against exact
search, the distance-0 column against Hamming search, every Hamming hit against the edit hits, the device entry
points, refused reads, every error code, a too-small hit buffer, both strands against the single-strand calls on q
and rc(q), and the brute-force comparison once more against the bounds-checked build."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT, device_from_parts, mixed_queries

pytestmark = pytest.mark.gpu

COMP = bytes.maketrans(b"ACGTNacgtnUu", b"TGCANTGCANAA")


def rc(q: bytes) -> bytes:
    """the reverse complement as include/awry_b200.h defines it (bytes outside ACGTU map to N, as exact search maps them)"""
    q = bytes(c if c in b"ACGTNacgtnUu" else ord("N") for c in q)
    return q.translate(COMP)[::-1]


def pack(qs):
    from awry_b200 import fm_index as f
    return f.pack_queries(qs)


@pytest.fixture(scope="module")
def brute_lib(tmp_path_factory, po):
    so = str(tmp_path_factory.mktemp("edit") / "libedit_brute.so")
    subprocess.check_call(["gcc", "-O2", "-fopenmp", "-shared", "-fPIC", "-o", so, os.path.join(ROOT, "tests", "edit_brute.c")])
    L = C.CDLL(so)
    L.edit_brute.restype = C.c_int64
    L.edit_brute.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint32,
                             C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    lut = np.array([po.lib().awo_ascii_to_index(0, c) for c in range(256)], dtype=np.uint8)
    return L, lut


def brute(brute_lib, parts, qb, qo, k):
    """-> (counts uint64[nq, k+1], hit_off uint64[nq+1], hits uint64[n, 2], edits uint8[n])"""
    L, lut = brute_lib
    text = np.ascontiguousarray(parts.text, dtype=np.uint8)
    qb = np.ascontiguousarray(qb, dtype=np.uint8)
    qo = np.ascontiguousarray(qo, dtype=np.uint64)
    nq = len(qo) - 1
    counts = np.zeros((nq, k + 1), dtype=np.uint64)
    off = np.zeros(nq + 1, dtype=np.uint64)
    args = (lut.ctypes.data, text.ctypes.data, len(text), qb.ctypes.data, qo.ctypes.data, nq, k, counts.ctypes.data,
            off.ctypes.data)
    n = L.edit_brute(*args, None, None)
    pos = np.zeros(max(1, n), dtype=np.uint64)
    dist = np.zeros(max(1, n), dtype=np.uint8)
    L.edit_brute(*args, pos.ctypes.data, dist.ctypes.data)
    starts = np.asarray(parts.seq_starts, dtype=np.uint64) if parts.seq_starts is not None else np.zeros(1, np.uint64)
    seq = np.searchsorted(starts, pos[:n], side="right").astype(np.uint64) - np.uint64(1)
    hits = np.stack([seq, pos[:n] - starts[seq]], axis=1) if n else np.zeros((0, 2), np.uint64)
    return counts, off, hits, dist[:n]


def assert_same(dev, parts, qb, qo, k, brute_lib, want=None):
    counts, off, hits, dist = want if want is not None else brute(brute_lib, parts, qb, qo, k)
    got = dev.count_edit_packed(qb, qo, k)
    bad = np.nonzero((got != counts).any(axis=1))[0]
    assert len(bad) == 0, (k, bad[:5], got[bad[:5]], counts[bad[:5]])
    goff, ghits, gd = dev.locate_edit_packed(qb, qo, k)
    bad = np.nonzero(goff != off)[0]
    assert len(bad) == 0, (k, bad[:5], goff[bad[:5]], off[bad[:5]])
    assert np.array_equal(ghits, hits) and np.array_equal(gd, dist), k
    return counts, off, hits, dist


@pytest.fixture(scope="module")
def multi(fx):
    """several records joined by N, with N runs and isolated N inside them"""
    r = np.random.default_rng(27)
    recs = []
    for i, n in enumerate([70_000, 1, 110_000, 40, 60_000]):
        t = bytearray(bytes(fx.gen_text(0, n, 70 + i)))
        if n > 1000:
            for _ in range(6):
                t[int(r.integers(0, n))] = ord("N")
            p = int(r.integers(0, n - 300))
            t[p:p + 120] = b"N" * 120
            for _ in range(8):                            # homopolymer runs of 6 .. 14
                p, ln = int(r.integers(0, n - 20)), int(r.integers(6, 15))
                t[p:p + ln] = bytes([b"ACGT"[int(r.integers(0, 4))]]) * ln
        recs.append(bytes(t))
    text, starts = fx.concat_records(recs, 0)
    return fx.build_parts(text, 0, ratio=8, kmer_len=9, seq_starts=starts)


@pytest.fixture(scope="module")
def multi_dev(multi):
    ix = device_from_parts(multi)
    yield ix
    ix.close()


def edit(q: bytearray, at: int, op: int, r):
    """op 0: substitute q[at]; 1: insert a base in front of q[at]; 2: delete q[at]"""
    if op == 0:
        c = q[at]
        alt = [b for b in b"ACGT" if b != c]
        q[at] = alt[int(r.integers(0, len(alt)))]
    elif op == 1:
        q.insert(at, b"ACGT"[int(r.integers(0, 4))])
    else:
        del q[at]


def plant(q: bytearray, at, r, k, ops=None):
    """edits at the positions `at` (applied from the last one on, so each lands where it was aimed)"""
    for i, a in enumerate(sorted(set(int(x) for x in at), reverse=True)):
        op = int(r.integers(0, 3)) if ops is None else ops[i % len(ops)]
        if op == 2 and len(q) <= k + 1:
            op = 0
        edit(q, min(a, len(q) - 1), op, r)


def homopolymer_reads(t: bytes, k, r, n=60):
    """windows around runs of >= 4 equal bases with the run one or two bases longer or shorter"""
    qs, p = [], 0
    runs = []
    while p < len(t) - 4 and len(runs) < 4 * n:
        e = p
        while e < len(t) and t[e] == t[p]:
            e += 1
        if e - p >= 4 and t[p] in b"ACGT":
            runs.append((p, e))
        p = e
    for i, (a, e) in enumerate(runs[:: max(1, len(runs) // n)][:n]):
        lo, ln = max(0, a - int(r.integers(5, 80))), int(r.integers(max(k + 2, 30), 200))
        q = bytearray(t[lo:lo + ln])
        at = a - lo + int(r.integers(0, e - a))
        if at >= len(q):
            continue
        for _ in range(1 + (i % min(2, k))):
            if i % 2:
                q.insert(at, q[at])                       # the run one base longer
            elif len(q) > k + 2:
                del q[at]                                 # one base shorter
        qs.append(bytes(q))
    return qs


def edit_queries(parts, k, seed, n_random=700):
    r = np.random.default_rng(seed)
    t = bytes(parts.text)
    starts = [int(s) for s in parts.seq_starts]
    qs = []
    # reads with 0 .. k+1 planted edits: anywhere, one per piece, at the piece boundaries, first / last symbol
    for i in range(n_random):
        ln = int(r.integers(k + 1, 600)) if i % 3 else int(r.integers(k + 1, 60))
        p = int(r.integers(0, len(t) - ln))
        q = bytearray(t[p:p + ln])
        m = i % (k + 2)
        cuts = [j * ln // (k + 1) for j in range(k + 2)]
        kind = (i // (k + 2)) % 4
        if kind == 0:
            at = r.choice(ln, size=min(m, ln), replace=False)
        elif kind == 1:
            at = [int(r.integers(cuts[j], cuts[j + 1])) for j in range(min(m, k + 1))]
        elif kind == 2:
            at = sorted(set(min(ln - 1, c + d) for c in cuts[1:] for d in (-1, 0)))[:m]
        else:
            at = [0, ln - 1][:m]
        plant(q, at, r, k, ops=[(i // 7) % 3, (i // 5) % 3])
        if i % 17 == 5:
            q = bytearray(bytes(q).lower())
        if i % 19 == 7:
            q = bytearray(bytes(q).replace(b"T", b"U"))
        if i % 23 == 11:
            q[int(r.integers(0, len(q)))] = ord("NRnyk"[int(r.integers(0, 5))])
        qs.append(bytes(q))
    # every length k+1 .. 300 and some up to 600, an edit in every other one
    for i, ln in enumerate(list(range(k + 1, 301)) + [301, 383, 384, 385, 447, 511, 512, 513, 599, 600]):
        p = int(r.integers(0, len(t) - ln))
        q = bytearray(t[p:p + ln])
        if i % 2:
            plant(q, [int(r.integers(0, ln))], r, k, ops=[i % 3])
        qs.append(bytes(q))
    qs += homopolymer_reads(t, k, r)
    # hanging over the start or the end of the text, with a deletion or an extra base outside
    for ln in (k + 1, k + 2, 20, 64, 65, 150, 300):
        for q in (bytearray(t[:ln]), bytearray(t[len(t) - ln:])):
            qs.append(bytes(q))
            if ln > k + 1:
                d = bytearray(q)
                del d[int(r.integers(0, ln))]
                qs.append(bytes(d))
        qs.append(b"G" + t[:ln - 1])
        qs.append(b"TT" + t[:ln])
        qs.append(t[len(t) - ln + 1:] + b"A")
        qs.append(t[len(t) - ln:] + b"CC")
    for s in starts[1:]:                                 # across record delimiters
        for back in (1, 5, 40):
            a = max(0, s - back)
            q = bytearray(t[a:a + 80])
            qs.append(bytes(q))
            plant(q, [min(len(q) - 1, back + 3)], r, k, ops=[1 + back % 2])
            qs.append(bytes(q))
    for _ in range(40):                                  # random reads: mostly nothing within k
        qs.append(bytes(r.choice(np.frombuffer(b"ACGT", np.uint8), int(r.integers(k + 1, 150)))))
    return qs


@pytest.mark.parametrize("k", [1, 2, 3])
def test_edit_equals_brute_force(k, multi, multi_dev, brute_lib):
    qb, qo = pack(edit_queries(multi, k, seed=500 + k))
    counts, off, hits, dist = assert_same(multi_dev, multi, qb, qo, k, brute_lib)
    assert all((counts[:, d] > 0).sum() > 50 for d in range(k + 1))
    assert len(hits) > 1000 and (np.diff(off.astype(np.int64)) == 0).sum() > 20


@pytest.mark.parametrize("k", [1, 2])
def test_every_single_edit_of_a_read(k, multi, multi_dev, brute_lib):
    """a 100-bp read with a substitution, an insertion and a deletion at every position"""
    r = np.random.default_rng(8)
    t = bytes(multi.text)
    read = bytearray(t[2000:2100])
    qs = [bytes(read)]
    for a in range(100):
        for op in range(3):
            q = bytearray(read)
            edit(q, a, op, r)
            qs.append(bytes(q))
    qb, qo = pack(qs)
    counts, _, _, _ = assert_same(multi_dev, multi, qb, qo, k, brute_lib)
    assert (counts[1:, :2].sum(axis=1) >= 1).all()


@pytest.fixture(scope="module")
def dna_small(fx):
    text = fx.gen_text(0, 200_000, 31)
    parts = fx.build_parts(text, 0, ratio=8, kmer_len=8)
    ix = device_from_parts(parts)
    yield parts, ix
    ix.close()


def test_k0_equals_exact_search(fx, dna_small):
    parts, ix = dna_small
    qb, qo = mixed_queries(fx, parts.text, 4000, 24, seed=2)
    counts = ix.count_edit_packed(qb, qo, 0)
    assert np.array_equal(counts[:, 0], ix.count_packed(qb, qo))
    off, hits = ix.locate_packed(qb, qo, sorted_hits=True)
    eoff, ehits, ed = ix.locate_edit_packed(qb, qo, 0)
    assert np.array_equal(eoff, off) and np.array_equal(ehits, hits) and not ed.any()


@pytest.mark.parametrize("k", [1, 2, 3])
def test_against_hamming_search(k, multi, multi_dev):
    """the distance-0 column equals Hamming's, and every Hamming hit (s, h) is an edit hit (s, d <= h)"""
    qb, qo = pack(edit_queries(multi, k, seed=600 + k, n_random=400))
    ec = multi_dev.count_edit_packed(qb, qo, k)
    hc = multi_dev.count_hamming_packed(qb, qo, k)
    assert np.array_equal(ec[:, 0], hc[:, 0])
    assert (ec.sum(axis=1) >= hc.sum(axis=1)).all()
    eoff, ehits, ed = multi_dev.locate_edit_packed(qb, qo, k)
    hoff, hhits, hd = multi_dev.locate_hamming_packed(qb, qo, k)
    for q in range(len(qo) - 1):
        got = {(int(a), int(b)): int(d) for (a, b), d in zip(ehits[int(eoff[q]):int(eoff[q + 1])],
                                                             ed[int(eoff[q]):int(eoff[q + 1])])}
        for (a, b), h in zip(hhits[int(hoff[q]):int(hoff[q + 1])], hd[int(hoff[q]):int(hoff[q + 1])]):
            assert got.get((int(a), int(b)), 99) <= int(h), (q, a, b, h)


@pytest.fixture(scope="module")
def repeats(fx):
    """repeat-rich text plus tandem arrays of period 1, 2 and 3: one start is covered by many candidates"""
    from fixtures.repeats import repeat_queries, repeat_rich_text
    r = np.random.default_rng(44)
    text, regions = repeat_rich_text(200_000, seed=4, tandem_arrays=20)
    text = text.copy()
    arrays = []
    for i in range(24):
        unit = np.frombuffer(bytes(b"ACGT"[int(x)] for x in r.integers(0, 4, 1 + i % 3)), np.uint8)
        ln = int(r.integers(100, 1500))
        p = int(r.integers(0, len(text) - ln))
        text[p:p + ln] = np.resize(unit, ln)
        arrays.append((p, p + ln))
    parts = fx.build_parts(text, 0, ratio=8, kmer_len=8)
    qb, qo = repeat_queries(text, regions, 200, 60, seed=6)
    t = bytes(text)
    qs = [bytes(qb[int(qo[i]):int(qo[i + 1])]) for i in range(len(qo) - 1)]
    for i, (a, e) in enumerate(arrays):                  # inside and across the arrays' ends, with indels
        for lo, ln in ((a + 10, 40), (max(0, a - 30), 70), (max(0, e - 50), 90)):
            q = bytearray(t[lo:lo + ln])
            qs.append(bytes(q))
            plant(q, [int(r.integers(0, len(q)))], r, 3, ops=[i % 3])
            qs.append(bytes(q))
    ix = device_from_parts(parts)
    yield parts, ix, qs
    ix.close()


@pytest.mark.parametrize("k", [1, 2, 3])
def test_repeat_rich_text_and_tiny_slices(k, repeats, brute_lib, monkeypatch):
    """tandem arrays give reads hundreds of starts covered by many candidates each: every hit list equals brute force
    and is free of duplicates, also when a slice holds 16 key slots (a candidate or two)"""
    parts, ix, qs = repeats
    qb, qo = pack(qs)
    want = brute(brute_lib, parts, qb, qo, k)
    assert np.diff(want[1].astype(np.int64)).max() >= 200
    _, goff, ghits, _ = assert_same(ix, parts, qb, qo, k, brute_lib, want)
    for i in range(len(goff) - 1):
        seg = ghits[int(goff[i]):int(goff[i + 1])]
        assert len(np.unique(seg, axis=0)) == len(seg)
    monkeypatch.setenv("AWRY_B200_HAMMING_SLICE", "16")
    sub = [q for i, q in enumerate(qs) if i % 3 == 0]
    sb, so = pack(sub)
    assert_same(ix, parts, sb, so, k, brute_lib)


def test_device_entry_points(multi, multi_dev):
    import torch
    from awry_b200 import AwryError
    qs = edit_queries(multi, 3, seed=12, n_random=300)
    qb, qo = pack(qs)
    nq = len(qo) - 1
    d_qb = torch.from_numpy(qb).cuda()
    d_qo = torch.from_numpy(qo.view(np.int64)).cuda()
    want = multi_dev.count_edit_packed(qb, qo, 3)
    d_counts = torch.full((nq, 4), 7, dtype=torch.int64, device="cuda")
    multi_dev.count_edit_device(d_qb.data_ptr(), d_qo.data_ptr(), nq, 3, d_counts.data_ptr())
    multi_dev.device_check()
    assert np.array_equal(d_counts.cpu().numpy().view(np.uint64), want)
    want = multi_dev.count_edit_strands_packed(qb, qo, 2)
    d_counts = torch.full((nq, 2, 3), 7, dtype=torch.int64, device="cuda")
    multi_dev.count_edit_strands_device(d_qb.data_ptr(), d_qo.data_ptr(), nq, 2, d_counts.data_ptr())
    multi_dev.device_check()
    assert np.array_equal(d_counts.cpu().numpy().view(np.uint64), want)
    # a refused read is latched for device_check, and its counts are 0
    qb2, qo2 = pack([bytes(multi.text[500:600]), b"ACG", bytes(multi.text[900:960])])
    d_qb, d_qo = torch.from_numpy(qb2).cuda(), torch.from_numpy(qo2.view(np.int64)).cuda()
    for strands in (False, True):
        d_counts = torch.zeros((3, 2 if strands else 1, 4), dtype=torch.int64, device="cuda")
        call = multi_dev.count_edit_strands_device if strands else multi_dev.count_edit_device
        call(d_qb.data_ptr(), d_qo.data_ptr(), 3, 3, d_counts.data_ptr())
        with pytest.raises(AwryError) as e:
            multi_dev.device_check()
        assert e.value.code == -5 and "query 1" in str(e.value)
        got = d_counts.cpu().numpy()
        assert got[0, 0, 0] >= 1 and got[2, 0, 0] >= 1 and not got[1].any()
        multi_dev.device_check()


def test_errors(fx, multi, multi_dev, monkeypatch):
    from awry_b200 import AwryError
    from awry_b200 import fm_index as f
    t = bytes(multi.text)
    calls = (multi_dev.count_edit_packed, multi_dev.locate_edit_packed, multi_dev.count_edit_strands_packed,
             multi_dev.locate_edit_strands_packed)
    for k, bad in ((1, b"A"), (2, b"AC"), (3, b"ACG"), (2, b""), (1, b"AC$GT"), (1, b"AC#GT")):
        qb, qo = pack([t[100:150], bad, t[200:260]])
        for call in calls:
            with pytest.raises(AwryError) as e:
                call(qb, qo, k)
            assert e.value.code == -5 and "query 1" in str(e.value), (k, bad)
    qb, qo = pack([t[100:150]])
    for call in calls:
        with pytest.raises(AwryError) as e:
            call(qb, qo, 4)
        assert e.value.code == -1 and "max_edits" in str(e.value)
    # too small a buffer: the offsets are complete, and the retry gives the same hits
    qb, qo = pack(edit_queries(multi, 1, seed=3, n_random=200))
    hoff, hits, dist = multi_dev.locate_edit_packed(qb, qo, 1, capacity=len(qo) * 100)
    off = np.zeros(len(qo), np.uint64)
    small = np.zeros((5, 2), np.uint64)
    ed = np.zeros(5, np.uint8)
    n = C.c_uint64()
    rc_ = f.native().awry_locate_batch_edit(multi_dev.handle, qb.ctypes.data, qo.ctypes.data, len(qo) - 1, 1,
                                            off.ctypes.data, small.ctypes.data, ed.ctypes.data, 5, C.byref(n))
    assert rc_ == -8 and n.value == len(hits) and np.array_equal(off, hoff)
    assert np.array_equal(small, hits[:5]) and np.array_equal(ed, dist[:5])
    assert np.array_equal(multi_dev.locate_edit_packed(qb, qo, 1, capacity=3)[1], hits)
    # indexes the search does not exist for
    text = fx.gen_text(1, 20_000, 3)
    prot = fx.build_parts(text, 1, ratio=8, kmer_len=3)
    with device_from_parts(prot) as ix:
        for call in (ix.count_edit_packed, ix.locate_edit_packed, ix.count_edit_strands_packed):
            with pytest.raises(AwryError) as e:
                call(*pack([b"ACDEFG"]), 1)
            assert e.value.code == -6
    dna = fx.gen_text(0, 30_000, 3)
    parts = fx.build_parts(dna, 0, ratio=8, kmer_len=8)
    for var in ("AWRY_B200_TEXT", "AWRY_B200_FULL_SA", "AWRY_B200_WIDE"):
        monkeypatch.setenv(var, "1" if var == "AWRY_B200_WIDE" else "0")
        with device_from_parts(parts) as ix:
            for call in (ix.count_edit_packed, ix.locate_edit_packed, ix.count_edit_strands_packed):
                with pytest.raises(AwryError) as e:
                    call(*pack([bytes(dna[:40])]), 1)
                assert e.value.code == -6, var
        monkeypatch.delenv(var)


def interleave(fwd, rev):
    """two single-strand results (counts, hit_off, hits, edits) -> the both-strand layout"""
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


@pytest.mark.parametrize("k", [1, 2, 3])
def test_both_strands_equal_single_strand(k, multi, multi_dev, brute_lib):
    """v = 2q equals the single-strand calls on q, v = 2q + 1 those on rc(q); both equal brute force"""
    qs = edit_queries(multi, k, seed=700 + k, n_random=300)
    qs = [rc(q) if i % 2 else q for i, q in enumerate(qs)]     # true hits on both strands
    qb, qo = pack(qs)
    rb, ro = pack([rc(q) for q in qs])
    single = interleave((multi_dev.count_edit_packed(qb, qo, k),) + multi_dev.locate_edit_packed(qb, qo, k),
                        (multi_dev.count_edit_packed(rb, ro, k),) + multi_dev.locate_edit_packed(rb, ro, k))
    want = interleave(brute(brute_lib, multi, qb, qo, k), brute(brute_lib, multi, rb, ro, k))
    for a, b in zip(single, want):
        assert np.array_equal(a, b), k
    got = multi_dev.count_edit_strands_packed(qb, qo, k)
    assert np.array_equal(got, want[0])
    goff, ghits, gd = multi_dev.locate_edit_strands_packed(qb, qo, k)
    assert np.array_equal(goff, want[1]) and np.array_equal(ghits, want[2]) and np.array_equal(gd, want[3]), k
    assert (got[1::2, 1].sum(axis=1) > 0).mean() > 0.5         # reads reverse-complemented are found on strand 1


def test_on_the_bounds_checked_build():
    """the brute-force comparison against libawry_b200_checked.so (every data-dependent load bounds-checked,
    layout.cuh): no assert"""
    checked = os.path.join(ROOT, "awry_b200", "libawry_b200_checked.so")
    if os.environ.get("AWRY_B200_LIB"):
        pytest.skip("already running against another build")
    if not os.path.exists(checked):
        subprocess.check_call(["make", "-s", "-C", os.path.join(ROOT, "awry_b200", "csrc"), "checked"])
    env = dict(os.environ, AWRY_B200_LIB=checked)
    out = subprocess.run([sys.executable, "-m", "pytest", "tests/test_gpu_edit.py", "-m", "gpu", "-x", "-q",
                          "-p", "no:cacheprovider", "-k", "equals_brute_force or repeat_rich"],
                         cwd=ROOT, env=env, capture_output=True, text=True, timeout=1800)
    tail = out.stdout[-1500:] + out.stderr[-1500:]
    assert out.returncode == 0, tail
    assert " passed" in out.stdout and "Assertion" not in out.stderr, tail
