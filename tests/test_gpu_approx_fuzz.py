"""Randomised differential test of the approximate searches: Hamming (awry_*_hamming) and edit distance
(awry_*_edit), one strand and both (_strands), against the brute-force references tests/hamming_brute.c and
tests/edit_brute.c (compiled into a temporary directory, bytes mapped by the oracle's awo_ascii_to_index; both strands:
the reference on q and on rc(q), interleaved).  Every case compares, bit for bit: counts per distance, the CSR hit
offsets, the hits in text order as (record, offset) and each hit's distance.  Reads with L <= k are left out (the
calls refuse them; test_gpu_hamming.py and test_gpu_edit.py check that).

- Random small indexes (fixed seeds): 1-5 records joined by concat_records, record lengths from 1 to 4000 around the
  word sizes (1, 2, 3, 7, 8, 9, 15, 16, 17, ... 255, 256, 257, 1000, 4000); uniform, skewed and tandem-array (period
  1-3) texts with N and IUPAC bytes; kmer_len 1-9, SA ratios 2-32.  k = 0 .. 3, both metrics, both strand counts,
  through count_*_packed, locate_*_packed and count_*_device.  Reads: substrings with 0 .. 4 planted substitutions,
  insertions and deletions (anywhere, at the piece boundaries, at the first and the last symbol); the whole text and
  the whole text with 1-3 bases added or removed; reads longer than the text; reads hanging over either end by 1-3
  copies of each base; reads across record delimiters; lowercase / U / N / IUPAC reads; random reads.  In every case
  also: edit search at k = 0 equals exact search (one strand and both), the distance-0 column of edit equals
  Hamming's, and every Hamming hit (s, h) is an edit hit (s, d <= h).
- Every text length near the word boundaries: single-record texts of every length 1 .. 70 and 64j - 1 .. 64j + 8 for
  j = 2, 3, 5 (every residue of n mod 8 and mod 64, texts shorter than the reads), reads at the very start and the
  very end with a substitution, insertion or deletion at the first or the last symbol, k = 1 .. 3, both metrics, both
  strand counts.
- Routes, on one multi-record index with N runs and batches of more than 3000 reads, each against brute force:
  set_locate_variant(1) and (2), set_count_variant(1), AWRY_B200_LOCATE_CHUNK_Q=1024 (several host chunks) and
  AWRY_B200_HAMMING_SLICE=16 (on the reads of 40 symbols and more), both metrics and strand counts, count and
  locate, k = 2 and 3; and the index loaded under AWRY_B200_KMER_DEV=0, AWRY_B200_KMER_DEV=12 and
  AWRY_B200_SB_SHIFT=8.  An index sampled at ratio 1 or loaded under AWRY_B200_PAIR_INDEX=0 has no text on the
  device, and every approximate call on it refuses with AWRY_ERR_UNSUPPORTED.
- Entry points: the four count_*_device calls on a sub-batch from the middle of a larger device buffer (first offset
  neither 0 nor a multiple of 64, data pointer + 1 .. 7 bytes), on a torch.cuda.Stream() other than the default, with
  garbage in d_counts beforehand, and with nq = 1; with two GPUs, a handle over devices [0, 1] (edit search, both
  strand counts, count and locate) and the device calls with replica = 1 fed from GPU 1.
- Long and awkward reads: 1000 - 8000 bp with <= k planted edits, chimeric reads (one locus, then another), reads
  across the text's N runs, and mostly-N reads over an N run (hundreds of candidates per read).
- The whole file once more against libawry_b200_checked.so (every data-dependent load bounds-checked), without the
  replica test: no assert.

On one B200 with the brute force on 16 host cores the file took 103 s, 53 s of it the rerun on the bounds-checked
build."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT, device_from_parts
from test_gpu_edit import edit, edit_queries, interleave, rc

pytestmark = pytest.mark.gpu

METRICS = ("hamming", "edit")
COMBOS = [(m, s) for m in METRICS for s in (False, True)]
LENS = [1, 2, 3, 7, 8, 9, 15, 16, 17, 31, 63, 64, 65, 127, 128, 129, 255, 256, 257, 1000, 4000]
IUPAC = b"RYKMSWBDHV"
ACGT = np.frombuffer(b"ACGT", np.uint8)


def pack(qs):
    from awry_b200 import fm_index as f
    return f.pack_queries(qs)


@pytest.fixture(scope="module")
def refs(tmp_path_factory, po):
    """the two brute-force references, compiled into a temporary directory"""
    d = tmp_path_factory.mktemp("approx_fuzz")
    fns = {}
    for m in METRICS:
        so = str(d / f"lib{m}_brute.so")
        subprocess.check_call(["gcc", "-O2", "-fopenmp", "-shared", "-fPIC", "-o", so,
                               os.path.join(ROOT, "tests", f"{m}_brute.c")])
        fn = getattr(C.CDLL(so), f"{m}_brute")
        fn.restype = C.c_int64
        fn.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint32,
                       C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        fns[m] = fn
    lut = np.array([po.lib().awo_ascii_to_index(0, c) for c in range(256)], dtype=np.uint8)
    return fns, lut


def brute(refs, metric, parts, qs, k):
    """-> (counts uint64[nq, k+1], hit_off uint64[nq+1], hits uint64[n, 2], dist uint8[n])"""
    fns, lut = refs
    assert all(len(q) < 8192 for q in qs), "the references skip reads of 8192 symbols and more"
    qb, qo = pack(qs)
    text = np.ascontiguousarray(parts.text, dtype=np.uint8)
    nq = len(qs)
    counts = np.zeros((nq, k + 1), dtype=np.uint64)
    off = np.zeros(nq + 1, dtype=np.uint64)
    args = (lut.ctypes.data, text.ctypes.data, len(text), qb.ctypes.data, qo.ctypes.data, nq, k, counts.ctypes.data,
            off.ctypes.data)
    n = fns[metric](*args, None, None)
    pos = np.zeros(max(1, n), dtype=np.uint64)
    dist = np.zeros(max(1, n), dtype=np.uint8)
    fns[metric](*args, pos.ctypes.data, dist.ctypes.data)
    starts = np.asarray(parts.seq_starts, dtype=np.uint64)
    seq = np.searchsorted(starts, pos[:n], side="right").astype(np.uint64) - np.uint64(1)
    hits = np.stack([seq, pos[:n] - starts[seq]], axis=1) if n else np.zeros((0, 2), np.uint64)
    return counts, off, hits, dist[:n]


def expected(refs, metric, strands, parts, qs, k):
    """the reference result in the layout of the call: both strands = (q, rc(q)) per read"""
    fwd = brute(refs, metric, parts, qs, k)
    return interleave(fwd, brute(refs, metric, parts, [rc(q) for q in qs], k)) if strands else fwd


def calls(dev, metric, strands):
    sfx = "_strands" if strands else ""
    return (getattr(dev, f"count_{metric}{sfx}_packed"), getattr(dev, f"locate_{metric}{sfx}_packed"),
            getattr(dev, f"count_{metric}{sfx}_device"))


def device_counts(dev, metric, strands, qb, qo, k, lo=0, hi=None, shift=0, stream=None, replica=0, device=0):
    """count_*_device on reads lo .. hi of the batch: the caller's bytes behind `shift` garbage bytes, the offsets of
    the whole batch on the device and d_qoff pointing at entry lo, d_counts filled with garbage"""
    import torch
    hi = len(qo) - 1 if hi is None else hi
    nq = hi - lo
    dv = torch.device("cuda", device)
    with torch.cuda.device(dv):
        d_qb = torch.from_numpy(np.concatenate([np.full(shift, ord("#"), np.uint8), qb])).to(dv)
        d_qo = torch.from_numpy(np.ascontiguousarray(qo, np.uint64).view(np.int64)).to(dv)
        d_counts = torch.full((nq,) + ((2,) if strands else ()) + (k + 1,), -3, dtype=torch.int64, device=dv)
        st = stream if stream is not None else torch.cuda.current_stream(dv)
        st.wait_stream(torch.cuda.current_stream(dv))
        calls(dev, metric, strands)[2](d_qb.data_ptr() + shift, d_qo.data_ptr() + 8 * lo, nq, k,
                                       d_counts.data_ptr(), st.cuda_stream, replica)
        dev.device_check(st.cuda_stream, replica)
        st.synchronize()
        return d_counts.cpu().numpy().view(np.uint64)


def check(dev, parts, qs, k, metric, strands, refs, tag, want=None, device=True):
    """count, locate and (with `device`) the device count against the reference; -> the device results"""
    want = want if want is not None else expected(refs, metric, strands, parts, qs, k)
    wc, woff, whits, wd = want
    what = (tag, metric, "both strands" if strands else "one strand", "k=%d" % k)
    qb, qo = pack(qs)
    count, locate, _ = calls(dev, metric, strands)
    got = count(qb, qo, k)
    bad = np.nonzero((got != wc).reshape(len(qs), -1).any(axis=1))[0]
    assert len(bad) == 0, what + ("count", bad[:5], [qs[i][:80] for i in bad[:3]], got[bad[:3]], wc[bad[:3]])
    goff, ghits, gd = locate(qb, qo, k)
    bad = np.nonzero(goff != woff)[0]
    assert len(bad) == 0, what + ("hit offsets", bad[:5], goff[bad[:5]], woff[bad[:5]])
    assert np.array_equal(ghits, whits), what + ("hits",)
    assert np.array_equal(gd, wd), what + ("distances",)
    if device:
        dc = device_counts(dev, metric, strands, qb, qo, k)
        assert np.array_equal(dc, wc), what + ("device count",)
    return got, goff, ghits, gd


def relations(dev, qs, k, res, tag):
    """edit at k = 0 is exact search; edit's distance-0 column is Hamming's; a Hamming hit (s, h) is an edit hit
    (s, d <= h).  res[(metric, strands)] = (counts, hit_off, hits, dist) of the calls."""
    qb, qo = pack(qs)
    if k == 0:
        ec, eoff, ehits, ed = res[("edit", False)]
        assert np.array_equal(ec[:, 0], dev.count_packed(qb, qo)), (tag, "k=0 count")
        off, hits = dev.locate_packed(qb, qo, sorted_hits=True)
        assert np.array_equal(eoff, off) and np.array_equal(ehits, hits) and not ed.any(), (tag, "k=0 locate")
        sc, soff, shits, sd = res[("edit", True)]
        assert np.array_equal(sc[:, :, 0], dev.count_strands_packed(qb, qo)), (tag, "k=0 strands count")
        off, hits = dev.locate_strands_packed(qb, qo, sorted_hits=True)
        assert np.array_equal(soff, off) and np.array_equal(shits, hits) and not sd.any(), (tag, "k=0 strands")
    for strands in (False, True):
        ec, eoff, ehits, ed = res[("edit", strands)]
        hc, hoff, hhits, hd = res[("hamming", strands)]
        assert np.array_equal(ec[..., 0], hc[..., 0]), (tag, strands, k, "distance 0")
        # one key per hit, (query, record, offset): ascending, as the hits of a query are in text order
        ekey, hkey = [(np.repeat(np.arange(len(o) - 1, dtype=np.uint64), np.diff(o.astype(np.int64))) << np.uint64(36))
                      | (h[:, 0] << np.uint64(32)) | h[:, 1] for o, h in ((eoff, ehits), (hoff, hhits))]
        at = np.minimum(np.searchsorted(ekey, hkey), max(0, len(ekey) - 1))
        ok = (ekey[at] == hkey) & (ed[at] <= hd) if len(ekey) else np.zeros(len(hkey), bool)
        assert ok.all(), (tag, strands, k, "Hamming hit not an edit hit", hkey[~ok][:5], hd[~ok][:5])


# ---- reads --------------------------------------------------------------------------------------------------------

def rand_bases(r, n):
    return bytes(ACGT[r.integers(0, 4, n)])


def mutate(q: bytearray, r, m, where):
    """m edits of random kinds: where 0 anywhere, 1 at the piece boundaries of a random k, 2 first / last symbol"""
    if not q:
        return q
    if where == 1:
        kk = int(r.integers(1, 4))
        at = [j * len(q) // (kk + 1) + d for j in range(1, kk + 1) for d in (-1, 0)]
    elif where == 2:
        at = [0, len(q) - 1]
    else:
        at = list(r.integers(0, len(q), max(1, m)))
    for a in sorted(set(int(x) for x in r.permutation(at)[:m]), reverse=True):
        if q:
            edit(q, min(a, len(q) - 1), int(r.integers(0, 3)), r)
    return q


def odd_bytes(q: bytes, r) -> bytes:
    """lowercase, U for T, N or an IUPAC code somewhere"""
    c = int(r.integers(0, 4))
    if c == 0:
        return q.lower()
    if c == 1:
        return q.replace(b"T", b"U")
    q = bytearray(q)
    if q:
        q[int(r.integers(0, len(q)))] = (b"N" + IUPAC)[int(r.integers(0, 1 + len(IUPAC)))]
    return bytes(q)


def end_reads(t: bytes, r, lens):
    """reads at the very start and the very end of the text (edited at the first and the last symbol), longer than
    the text, and hanging over either end by 1 .. 3 copies of one base"""
    n = len(t)
    qs = []
    for ln in lens:
        if ln <= n:
            for q in (t[:ln], t[n - ln:]):
                qs.append(q)
                for at in (0, ln - 1):
                    for op in range(3):
                        e = bytearray(q)
                        edit(e, at, op, r)
                        qs.append(bytes(e))
        else:
            qs += [t + rand_bases(r, ln - n), rand_bases(r, ln - n) + t]
        for h in (1, 2, 3):
            if 0 < ln - h <= n:
                for b in b"ACGT":
                    qs += [t[n - ln + h:] + bytes([b]) * h, bytes([b]) * h + t[:ln - h]]
    return qs


def fuzz_reads(t: bytes, starts, r, n_sub=240):
    n = len(t)
    qs = []
    for i in range(n_sub):                               # substrings with 0 .. 4 planted edits
        ln = int(r.choice([2, 4, 5, 8, 9, 12, 16, 17, 24, 31, 32, 33, 48, 64, 65, 100, 150, 300]))
        p = int(r.integers(0, max(1, n - ln + 1)))
        q = mutate(bytearray(t[p:p + ln]), r, i % 5, (i // 5) % 3)
        qs.append(odd_bytes(bytes(q), r) if i % 7 == 3 else bytes(q))
    if n < 7000:                                         # the whole text, with 1 .. 3 bases added or removed
        qs.append(t)
        for d in (1, 2, 3):
            a = bytearray(t)
            for _ in range(d):
                a.insert(int(r.integers(0, len(a) + 1)), ACGT[int(r.integers(0, 4))])
            qs.append(bytes(a))
            if n > d:
                b = bytearray(t)
                for _ in range(d):
                    del b[int(r.integers(0, len(b)))]
                qs.append(bytes(b))
    qs += end_reads(t, r, sorted({2, 3, 4, 9, 17, 33, 65, min(n, 6000), min(n + 1, 6000), min(n + 3, 6000)}))
    for s in [int(x) for x in starts[1:]]:               # across record delimiters
        for back in (1, 3, 9):
            a = max(0, s - back)
            q = bytearray(t[a:a + 24])
            qs.append(bytes(q))
            qs.append(bytes(mutate(q, r, 1, 0)))
    for i in range(20):                                  # random reads, some with N and IUPAC bytes
        q = rand_bases(r, int(r.integers(2, 40)))
        qs.append(odd_bytes(q, r) if i % 2 else q)
    qs += [b"NNNNNN", b"nnnnNNNN" * 3]
    return [q for q in qs if q]


def random_text(r, ln):
    kind = int(r.integers(0, 4))
    if kind == 1:                                        # low entropy
        t = bytearray(ACGT[r.choice(4, ln, p=[0.7, 0.1, 0.1, 0.1])].tobytes())
    elif kind == 2:                                      # a tandem array of period 1 .. 3 with a few substitutions
        unit = ACGT[r.integers(0, 4, int(r.integers(1, 4)))]
        t = bytearray(np.resize(unit, ln).tobytes())
        for _ in range(int(r.integers(0, 1 + ln // 50))):
            t[int(r.integers(0, ln))] = ACGT[int(r.integers(0, 4))]
    else:
        t = bytearray(rand_bases(r, ln))
    for _ in range(int(r.integers(0, 3))):               # N and IUPAC bytes in the text
        t[int(r.integers(0, ln))] = (b"N" + IUPAC)[int(r.integers(0, 1 + len(IUPAC)))]
    if ln >= 1000 and r.random() < 0.5:                  # an N run
        p = int(r.integers(0, ln - 40))
        t[p:p + 40] = b"N" * 40
    return bytes(t)


# ---- 1. random small indexes --------------------------------------------------------------------------------------

@pytest.mark.parametrize("seed", range(24))
def test_random_index(fx, refs, seed):
    r = np.random.default_rng(9000 + seed)
    recs = [random_text(r, int(r.choice(LENS))) for _ in range(int(r.integers(1, 6)))]
    text, starts = fx.concat_records(recs, 0)
    ratio, kmer_len = int(r.choice([2, 3, 4, 8, 16, 32])), int(r.integers(1, 10))
    parts = fx.build_parts(text, 0, ratio=ratio, kmer_len=kmer_len, seq_starts=starts)
    reads = fuzz_reads(bytes(text), starts, r)
    tag = "seed %d (n=%d, records %s, ratio %d, kmer_len %d)" % (seed, len(text), [len(x) for x in recs], ratio,
                                                                  kmer_len)
    with device_from_parts(parts) as ix:
        for k in range(4):
            qs = [q for q in reads if len(q) > k]
            res = {(m, s): check(ix, parts, qs, k, m, s, refs, tag) for m, s in COMBOS}
            relations(ix, qs, k, res, tag)


# ---- 2. every text length near the word boundaries ----------------------------------------------------------------

SWEEP = list(range(1, 71)) + [64 * j + d for j in (2, 3, 5) for d in range(-1, 9)]


@pytest.mark.parametrize("n", SWEEP)
def test_text_length(fx, refs, n):
    r = np.random.default_rng(n)
    t = rand_bases(r, n) if n % 3 else random_text(r, n)
    parts = fx.build_parts(t, 0, ratio=8, kmer_len=int(1 + n % 9), seq_starts=np.zeros(1, np.uint64))
    with device_from_parts(parts) as ix:
        for k in (1, 2, 3):
            lens = sorted({k + 1, k + 2, 8, 9, 16, 17, 31, 32, 33, 63, 64, 65, n - 2, n - 1, n, n + 1, n + k + 1})
            qs = [q for q in end_reads(t, r, [ln for ln in lens if ln > k]) if len(q) > k]
            for m, s in COMBOS:
                check(ix, parts, qs, k, m, s, refs, "n=%d" % n)


# ---- 3. routes ----------------------------------------------------------------------------------------------------

@pytest.fixture(scope="module")
def mid(fx):
    """five records joined by N: N runs of 120 and 700, isolated N, homopolymers and a tandem array"""
    r = np.random.default_rng(71)
    recs = []
    for i, n in enumerate([30_000, 3, 25_000, 17, 15_000]):
        t = bytearray(bytes(fx.gen_text(0, n, 90 + i)))
        if n > 1000:
            for _ in range(6):
                t[int(r.integers(0, n))] = ord("N")
            for _ in range(8):
                p, ln = int(r.integers(0, n - 20)), int(r.integers(6, 15))
                t[p:p + ln] = bytes([b"ACGT"[int(r.integers(0, 4))]]) * ln
            p = int(r.integers(0, n - 400))
            t[p:p + 300] = np.resize(ACGT[r.integers(0, 4, 1 + i % 3)], 300).tobytes()
            p = int(r.integers(100, n - 1000))
            run = 700 if i == 0 else 120
            t[p:p + run] = b"N" * run
        recs.append(bytes(t))
    text, starts = fx.concat_records(recs, 0)
    return fx.build_parts(text, 0, ratio=8, kmer_len=9, seq_starts=starts)


@pytest.fixture(scope="module")
def mid_dev(mid):
    ix = device_from_parts(mid)
    yield ix
    ix.close()


@pytest.fixture(scope="module")
def batches(mid, refs):
    """k -> (reads, {(metric, strands): reference}); more than 3000 reads, every other one reverse-complemented"""
    out = {}

    def get(k):
        if k not in out:
            qs = edit_queries(mid, k, seed=40 + k, n_random=3600)
            qs = [rc(q) if i % 2 else q for i, q in enumerate(qs)]
            assert len(qs) > 3000
            want = {}
            for m in METRICS:
                fwd = brute(refs, m, mid, qs, k)
                want[(m, False)] = fwd
                want[(m, True)] = interleave(fwd, brute(refs, m, mid, [rc(q) for q in qs], k))
            out[k] = (qs, want)
        return out[k]
    return get


def select(want, keep):
    """the reference result of the reads where `keep` (one strand: keep[q]; both strands: keep[v // 2])"""
    counts, off, hits, dist = want
    per = len(off) // len(keep)
    kv = np.repeat(keep, per)
    lens = np.diff(off.astype(np.int64))
    kh = np.repeat(kv, lens)
    new_off = np.zeros(int(kv.sum()) + 1, np.uint64)
    new_off[1:] = np.cumsum(lens[kv]).astype(np.uint64)
    return counts[keep], new_off, hits[kh], dist[kh]


ROUTES = ["locate_variant_1", "locate_variant_2", "count_variant_1", "locate_chunk_q_1024", "slice_16"]


@pytest.mark.parametrize("k", [2, 3])
@pytest.mark.parametrize("route", ROUTES)
def test_route(route, k, mid, mid_dev, batches, refs, monkeypatch):
    from awry_b200 import fm_index as f
    qs, want = batches(k)
    try:
        if route.startswith("locate_variant"):
            f.set_locate_variant(int(route[-1]))
        elif route == "count_variant_1":
            f.set_count_variant(1)
        elif route == "locate_chunk_q_1024":
            monkeypatch.setenv("AWRY_B200_LOCATE_CHUNK_Q", "1024")
        else:                                            # (reads of a few symbols have 10^5 candidates)
            monkeypatch.setenv("AWRY_B200_HAMMING_SLICE", "16")
            keep = np.array([len(q) >= 40 for q in qs])
            qs = [q for q in qs if len(q) >= 40]
            want = {c: select(w, keep) for c, w in want.items()}
            assert len(qs) >= 3000
        for m, s in COMBOS:
            check(mid_dev, mid, qs, k, m, s, refs, route, want[(m, s)])
    finally:
        f.set_locate_variant(0)
        f.set_count_variant(0)


@pytest.mark.parametrize("var,val", [("AWRY_B200_KMER_DEV", "0"), ("AWRY_B200_KMER_DEV", "12"),
                                     ("AWRY_B200_SB_SHIFT", "8")])
def test_index_loaded_with(var, val, mid, batches, refs, monkeypatch):
    qs, want = batches(2)
    monkeypatch.setenv(var, val)
    with device_from_parts(mid) as ix:
        for m, s in COMBOS:
            check(ix, mid, qs, 2, m, s, refs, "%s=%s" % (var, val), want[(m, s)])


def test_indexes_without_the_text_refuse(fx, mid, monkeypatch):
    """the text is built only next to the pair index and the unsampled array only when the file samples the suffix
    array (ratio > 1): without them every approximate call refuses (include/awry_b200.h), on every strand count"""
    from awry_b200 import AwryError
    qb, qo = pack([bytes(mid.text[1000:1100])])
    ratio1 = fx.build_parts(bytes(mid.text[:20_000]), 0, ratio=1, kmer_len=8)
    for pair_index_off in (False, True):
        if pair_index_off:
            monkeypatch.setenv("AWRY_B200_PAIR_INDEX", "0")
        with device_from_parts(mid if pair_index_off else ratio1) as ix:
            assert ix.count_packed(qb, qo)[0] >= 1
            for m, s in COMBOS:
                for call in calls(ix, m, s)[:2]:
                    with pytest.raises(AwryError) as e:
                        call(qb, qo, 1)
                    assert e.value.code == -6, (pair_index_off, m, s)


# ---- 4. entry points ----------------------------------------------------------------------------------------------

def test_device_sub_batches_and_streams(mid, mid_dev, batches):
    import torch
    qs, want = batches(3)
    qb, qo = pack(qs)
    lo = next(i for i in range(500, 3000) if int(qo[i]) % 64)
    cases = [(lo, lo + 1700), (lo + 3, lo + 4), (len(qs) - 1, len(qs)), (0, 1)]
    stream = torch.cuda.Stream()
    for c, (m, s) in enumerate(COMBOS):
        wc = want[(m, s)][0]
        for i, (a, b) in enumerate(cases):
            shift = 1 + (c * len(cases) + i) % 7
            for st in (None, stream):
                got = device_counts(mid_dev, m, s, qb, qo, 3, a, b, shift=shift, stream=st)
                assert np.array_equal(got, wc[a:b]), (m, s, a, b, shift, st is not None)


def test_two_replicas(mid, batches, refs):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    qs, want = batches(2)
    qb, qo = pack(qs)
    ix = device_from_parts(mid, devices=[0, 1])
    try:
        for s in (False, True):
            check(ix, mid, qs, 2, "edit", s, refs, "devices [0, 1]", want[("edit", s)], device=False)
        stream = torch.cuda.Stream(device=1)
        for m, s in COMBOS:
            for st in (None, stream):
                got = device_counts(ix, m, s, qb, qo, 2, 7, len(qs), shift=5, stream=st, replica=1, device=1)
                assert np.array_equal(got, want[(m, s)][0][7:]), (m, s, st is not None)
    finally:
        ix.close()


# ---- 5. long and awkward reads ------------------------------------------------------------------------------------

def awkward_reads(mid, k, seed):
    r = np.random.default_rng(seed)
    t = bytes(mid.text)
    n = len(t)
    qs = []
    for i in range(24):                                  # 1000 - 8000 bp with <= k edits
        ln = int(r.integers(1000, 8000))
        p = int(r.integers(0, n - ln))
        q = bytearray(t[p:p + ln])
        for _ in range(i % (k + 1)):
            edit(q, int(r.integers(0, len(q))), int(r.integers(0, 3)), r)
        qs.append(bytes(q))
    for i in range(16):                                  # chimeric: one locus, then another; the DP dies late
        a, b = int(r.integers(200, 3000)), int(r.integers(5, 400))
        p, p2 = int(r.integers(0, n - a)), int(r.integers(0, n - b))
        q = bytearray(t[p:p + a] + t[p2:p2 + b]) if i % 2 else bytearray(t[p2:p2 + b] + t[p:p + a])
        if i % 3 == 0:
            edit(q, int(r.integers(0, len(q))), i % 3, r)
        qs.append(bytes(q))
    runs = []                                            # the N runs of the text
    p = t.find(b"NNNNN")
    while p >= 0:
        e = p
        while e < n and t[e] == ord("N"):
            e += 1
        runs.append((p, e))
        p = t.find(b"NNNNN", e)
    assert max(e - a for a, e in runs) >= 700
    for a, e in runs:                                    # across the N runs, and mostly N over them
        for lo, ln in ((a - 30, e - a + 60), (a - 5, 200), (e - 10, 150)):
            q = bytearray(t[max(0, lo):max(0, lo) + ln])
            qs.append(bytes(q))
            edit(q, int(r.integers(0, len(q))), int(r.integers(0, 3)), r)
            qs.append(bytes(q))
        if e - a >= 300:
            for ln in (40, 150, 299):
                q = bytearray(b"N" * ln)
                for _ in range(k):
                    q[int(r.integers(0, ln))] = ACGT[int(r.integers(0, 4))]
                qs.append(bytes(q))
                qs.append(t[a - 3:a] + bytes(q[3:]))
    return qs


@pytest.mark.parametrize("k", [1, 3])
def test_long_and_awkward_reads(k, mid, mid_dev, refs):
    qs = awkward_reads(mid, k, seed=60 + k)
    for m, s in COMBOS:
        got = check(mid_dev, mid, qs, k, m, s, refs, "awkward")[0]
        if not s:
            assert (got[:24].sum(axis=1) > 0).all() or m == "hamming", m  # the long reads are found
            assert got.sum(axis=1).max() >= 200, m       # the mostly-N reads have hundreds of hits


# ---- 6. the bounds-checked build ----------------------------------------------------------------------------------

def test_on_the_bounds_checked_build():
    """this file against libawry_b200_checked.so (every data-dependent load bounds-checked, layout.cuh): no assert"""
    checked = os.path.join(ROOT, "awry_b200", "libawry_b200_checked.so")
    if os.environ.get("AWRY_B200_LIB"):
        pytest.skip("already running against another build")
    if not os.path.exists(checked):
        subprocess.check_call(["make", "-s", "-C", os.path.join(ROOT, "awry_b200", "csrc"), "checked"])
    env = dict(os.environ, AWRY_B200_LIB=checked)
    out = subprocess.run([sys.executable, "-m", "pytest", "tests/test_gpu_approx_fuzz.py", "-m", "gpu", "-x", "-q",
                          "-p", "no:cacheprovider", "-k", "not bounds_checked and not two_replicas"],
                         cwd=ROOT, env=env, capture_output=True, text=True, timeout=3000)
    tail = out.stdout[-1500:] + out.stderr[-1500:]
    assert out.returncode == 0, tail
    assert " passed" in out.stdout and "Assertion" not in out.stderr, tail
