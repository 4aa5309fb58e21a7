"""Edit-distance search by locus: awry_count_batch_edit_loci, awry_locate_batch_edit_loci, awry_count_device_edit_loci
and awry_locate_device_edit_loci, one strand and both.

- Reference: the locus filter `loci` of test_edit_loci_abi.py applied to the hits of the brute-force reference
  tests/edit_brute.c (through the helpers of test_gpu_approx_fuzz.py), not to the library's own edit locate.  Every
  case compares bit for bit the counts per distance, the CSR offsets, the hits and their distances of all four calls
  with it, k = 0 .. 3, on: random small indexes of the fuzz suite, texts of every length 1 .. 70 and around 64j, its
  multi-record index (more than 3000 reads), the repeat-rich text (plateaus and tandem arrays), reads up to 8000 bp,
  16-slot slices and several host chunks.
- Invariants against the library's own calls: k = 0 loci are the hits of awry_locate_batch[_strands] with
  AWRY_LOCATE_SORTED; the d = 0 column is awry_count_batch[_strands]; the loci are a subset of the edit locate's hits
  with the same distances; the smallest distance per query is unchanged; reverse-strand loci of q are the
  single-strand loci of rc(q).
- Alignment: awry_align_batch / awry_align_device (metric edit) on the loci keep the header's promise, checked in
  Python against the text.
- Device entry points: sub-batches at unaligned offsets, a non-default stream, nq = 1, no hits, replica 1 (two GPUs),
  20 calls in a row, refused reads (latched; their result is the filter applied to the device edit locate's result).
- Unsupported indexes are refused as by the edit calls.
- Planted reads on a seeded random text: each comes back as one locus at its origin, where the plain edit locate
  returns several starts.
- The whole file once more against libawry_b200_checked.so."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT, device_from_parts
from test_edit_loci_abi import loci
from test_gpu_approx_fuzz import (LENS, awkward_reads, batches, end_reads, expected, fuzz_reads, mid,  # noqa: F401
                                  mid_dev, rand_bases, random_text, refs, select)
from test_gpu_edit import rc
from test_gpu_hamming import repeats  # noqa: F401

pytestmark = pytest.mark.gpu


def pack(qs):
    from awry_b200 import fm_index as f
    return f.pack_queries(qs)


def to_host(ptr, nbytes, dtype):
    out = np.zeros(max(1, nbytes), np.uint8)
    if nbytes:
        assert C.CDLL("libcudart.so").cudaMemcpy(C.c_void_p(out.ctypes.data), C.c_void_p(ptr), C.c_size_t(nbytes), 2) == 0
    return out[:nbytes].view(dtype)


def ref_loci(want, parts, k):
    """the loci of a reference result (counts, hit_off, hits, dist) in the same layout"""
    counts, off, hits, dist = want
    starts = np.asarray(parts.seq_starts, np.uint64)
    pos = starts[hits[:, 0].astype(np.int64)] + hits[:, 1] if len(hits) else np.zeros(0, np.uint64)
    new_off, keep = loci(off, pos, dist, k)
    nv = len(off) - 1
    v = np.repeat(np.arange(nv), np.diff(off.astype(np.int64)))[keep]
    c = np.zeros((nv, k + 1), np.uint64)
    np.add.at(c, (v, dist[keep].astype(np.int64)), 1)
    return c.reshape(counts.shape), new_off, hits[keep], dist[keep]


def device_locate(dev, strands, qb, qo, k, lo=0, hi=None, shift=0, stream=None, replica=0, device=0, distances=True,
                  check=True, plain=False):
    """locate_edit_loci_device (plain: locate_edit[_strands]_device) on reads lo .. hi: the bytes behind `shift`
    garbage bytes, d_qoff at entry lo of the whole batch's offsets, d_hit_off filled with garbage -> (hit_off, hits,
    distances or None); the device buffers are freed"""
    import torch
    hi = len(qo) - 1 if hi is None else hi
    nq = hi - lo
    dv = torch.device("cuda", device)
    with torch.cuda.device(dv):
        d_qb = torch.from_numpy(np.concatenate([np.full(shift, ord("#"), np.uint8), qb])).to(dv)
        d_qo = torch.from_numpy(np.ascontiguousarray(qo, np.uint64).view(np.int64)).to(dv)
        d_off = torch.full(((2 if strands else 1) * nq + 1,), -3, dtype=torch.int64, device=dv)
        st = stream if stream is not None else torch.cuda.current_stream(dv)
        st.wait_stream(torch.cuda.current_stream(dv))
        args = (d_qb.data_ptr() + shift, d_qo.data_ptr() + 8 * lo, nq, k, d_off.data_ptr())
        if plain:
            call = dev.locate_edit_strands_device if strands else dev.locate_edit_device
            hp, dp, n = call(*args, distances=distances, stream=st.cuda_stream, replica=replica)
        else:
            hp, dp, n = dev.locate_edit_loci_device(*args, strands=strands, distances=distances, stream=st.cuda_stream,
                                                    replica=replica)
        if check:
            dev.device_check(st.cuda_stream, replica)
        st.synchronize()
        if n == 0:
            assert hp is None and dp is None
        hits = to_host(hp, n * 16, np.uint64).reshape(-1, 2)
        dist = to_host(dp, n, np.uint8) if distances and n else (np.zeros(0, np.uint8) if distances else None)
        dev.device_free(hp, replica)
        dev.device_free(dp, replica)
        off = d_off.cpu().numpy().view(np.uint64)
        assert int(off[-1]) == n
        return off, hits, dist


def device_count(dev, strands, qb, qo, k, lo=0, hi=None, shift=0, stream=None, replica=0, device=0, check=True):
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
        dev.count_edit_loci_device(d_qb.data_ptr() + shift, d_qo.data_ptr() + 8 * lo, nq, k, d_counts.data_ptr(),
                                   strands=strands, stream=st.cuda_stream, replica=replica)
        if check:
            dev.device_check(st.cuda_stream, replica)
        st.synchronize()
        return d_counts.cpu().numpy().view(np.uint64)


def same(got, want, what):
    goff, ghits, gd = got
    woff, whits, wd = want[-3:]
    bad = np.nonzero(goff != woff)[0]
    assert len(bad) == 0, what + ("hit offsets", bad[:5], goff[bad[:5]], woff[bad[:5]])
    assert np.array_equal(ghits, whits), what + ("hits",)
    if gd is not None:
        assert np.array_equal(gd, wd), what + ("distances",)


def check(dev, parts, qs, k, strands, refs, tag, want=None, device=True):
    """all four calls against the loci of the brute-force reference (`want`: that reference, plain edit hits)"""
    want = want if want is not None else expected(refs, "edit", strands, parts, qs, k)
    ref = ref_loci(want, parts, k)
    what = (tag, "both strands" if strands else "one strand", "k=%d" % k)
    qb, qo = pack(qs)
    got = dev.locate_edit_loci_packed(qb, qo, k, strands=strands)
    same(got, ref, what + ("host locate",))
    assert np.array_equal(dev.count_edit_loci_packed(qb, qo, k, strands=strands), ref[0]), what + ("host count",)
    if device:
        same(device_locate(dev, strands, qb, qo, k), ref, what + ("device locate",))
        assert np.array_equal(device_count(dev, strands, qb, qo, k), ref[0]), what + ("device count",)
    return got


def invariants(dev, qs, k, tag):
    """the header's consequences, against the library's own calls"""
    qb, qo = pack(qs)
    for strands in (False, True):
        what = (tag, strands, k)
        off, hits, dist = dev.locate_edit_loci_packed(qb, qo, k, strands=strands)
        counts = dev.count_edit_loci_packed(qb, qo, k, strands=strands)
        exact = dev.count_strands_packed(qb, qo) if strands else dev.count_packed(qb, qo)
        assert np.array_equal(counts[..., 0], exact), what + ("d = 0 column",)
        if k == 0:
            eo, eh = (dev.locate_strands_packed if strands else dev.locate_packed)(qb, qo, sorted_hits=True)
            assert np.array_equal(off, eo) and np.array_equal(hits, eh), what + ("k = 0",)
        po, ph, pd = (dev.locate_edit_strands_packed if strands else dev.locate_edit_packed)(qb, qo, k)
        for v in range(len(off) - 1):
            a, b, c, d = int(off[v]), int(off[v + 1]), int(po[v]), int(po[v + 1])
            plain = {tuple(h): e for h, e in zip(ph[c:d].tolist(), pd[c:d].tolist())}
            assert all(plain.get(tuple(h)) == e for h, e in zip(hits[a:b].tolist(), dist[a:b].tolist())), what + (v,)
            assert (b == a) == (d == c), what + ("a query with hits has a locus", v)
            if b > a:
                assert int(dist[a:b].min()) == int(pd[c:d].min()), what + ("best distance", v)
        if strands:
            r_off, r_hits, r_dist = dev.locate_edit_loci_packed(*pack([rc(q) for q in qs]), k)
            for q in range(len(qs)):
                a, b = int(off[2 * q + 1]), int(off[2 * q + 2])
                c, d = int(r_off[q]), int(r_off[q + 1])
                assert np.array_equal(hits[a:b], r_hits[c:d]) and np.array_equal(dist[a:b], r_dist[c:d]), what + (q,)


# ---- 1. the reference, bit for bit ---------------------------------------------------------------------------------

@pytest.mark.parametrize("seed", range(8))
def test_random_index(fx, refs, seed):
    r = np.random.default_rng(9000 + seed)                 # the first indexes of test_gpu_approx_fuzz.py
    recs = [random_text(r, int(r.choice(LENS))) for _ in range(int(r.integers(1, 6)))]
    text, starts = fx.concat_records(recs, 0)
    ratio, kmer_len = int(r.choice([2, 3, 4, 8, 16, 32])), int(r.integers(1, 10))
    parts = fx.build_parts(text, 0, ratio=ratio, kmer_len=kmer_len, seq_starts=starts)
    reads = fuzz_reads(bytes(text), starts, r)
    with device_from_parts(parts) as ix:
        for k in range(4):
            qs = [q for q in reads if len(q) > k]
            for s in (False, True):
                check(ix, parts, qs, k, s, refs, "seed %d" % seed)
            invariants(ix, qs, k, "seed %d" % seed)


SWEEP = list(range(1, 71)) + [64 * j + d for j in (2, 3, 5) for d in (-1, 0, 1, 8)]


@pytest.mark.parametrize("n", SWEEP)
def test_text_length(fx, refs, n):
    r = np.random.default_rng(n)
    t = rand_bases(r, n) if n % 3 else random_text(r, n)
    parts = fx.build_parts(t, 0, ratio=8, kmer_len=int(1 + n % 9), seq_starts=np.zeros(1, np.uint64))
    with device_from_parts(parts) as ix:
        for k in (0, 1, 2, 3):
            lens = sorted({k + 1, k + 2, 8, 9, 17, 33, 65, n - 1, n, n + 1, n + k + 1})
            qs = [q for q in end_reads(t, r, [ln for ln in lens if ln > max(k, 1)]) if len(q) > k]
            for s in (False, True):
                check(ix, parts, qs, k, s, refs, "n=%d" % n)


@pytest.mark.parametrize("k", [0, 1, 2, 3])
def test_mid_index(k, mid, mid_dev, batches, refs):
    qs, want = batches(max(k, 1))                          # (k = 0 takes k = 1's reads)
    for s in (False, True):
        check(mid_dev, mid, qs, k, s, refs, "mid", want[("edit", s)] if k else None)
    invariants(mid_dev, qs[:600], k, "mid")


@pytest.mark.parametrize("route", ["slice_16", "locate_chunk_q_1024"])
def test_route(route, mid, mid_dev, batches, refs, monkeypatch):
    qs, want = batches(3)
    if route == "slice_16":                                # (reads of a few symbols have 10^5 candidates)
        monkeypatch.setenv("AWRY_B200_HAMMING_SLICE", "16")
        keep = np.array([len(q) >= 40 for q in qs])
        qs = [q for q in qs if len(q) >= 40]
        want = {c: select(w, keep) for c, w in want.items()}
    else:
        monkeypatch.setenv("AWRY_B200_LOCATE_CHUNK_Q", "1024")
    for s in (False, True):
        check(mid_dev, mid, qs, 3, s, refs, route, want[("edit", s)])


def test_repeat_rich_text(repeats, refs, monkeypatch):  # noqa: F811
    parts, ix, qb, qo = repeats
    qs = [bytes(qb[int(qo[i]):int(qo[i + 1])]) for i in range(len(qo) - 1)]
    monkeypatch.setenv("AWRY_B200_HAMMING_SLICE", "300")
    plateaus = 0
    for k in (1, 2, 3):
        for s in (False, True):
            want = expected(refs, "edit", s, parts, qs, k)
            got = check(ix, parts, qs, k, s, refs, "repeats", want)
            plateaus += len(want[2]) - len(got[1])
    assert plateaus > 0
    invariants(ix, qs[:200], 2, "repeats")


def test_long_and_awkward_reads(mid, mid_dev, refs):
    qs = awkward_reads(mid, 3, seed=81)
    for s in (False, True):
        check(mid_dev, mid, qs, 3, s, refs, "awkward")


# ---- 2. alignment of the loci ----------------------------------------------------------------------------------------

def apply_ops(q: bytes, a) -> bytes:
    """the window the ops of one alignment make of Q"""
    out, at = bytearray(), 0
    for t in range(int(a["n_ops"])):
        qpos, op, ts = (int(a["ops"][t][x]) for x in ("qpos", "op", "text_sym"))
        out += q[at:qpos]
        if op == ord("X"):
            out.append(ts)
            at = qpos + 1
        elif op == ord("I"):
            at = qpos + 1
        else:
            out.append(ts)
            at = qpos
    return bytes(out + q[at:])


def test_alignment_of_the_loci(mid, mid_dev, batches, refs):
    import torch
    from awry_b200 import fm_index as f
    lut = bytes(refs[1])                                   # bytes -> symbols, as exact search maps them
    qs, _ = batches(2)
    qs = qs[:800]
    qb, qo = pack(qs)
    text = bytes(mid.text)
    starts = np.asarray(mid.seq_starts, np.uint64)
    for s in (False, True):
        off, hits, dist = mid_dev.locate_edit_loci_packed(qb, qo, 2, strands=s)
        al = mid_dev.align_hits_packed(qb, qo, "edit", 2, off, hits, strands=s)
        d_qb, d_qo = torch.from_numpy(qb).cuda(), torch.from_numpy(qo.view(np.int64)).cuda()
        d_off = torch.from_numpy(off.view(np.int64)).cuda()
        d_hits = torch.from_numpy(hits.view(np.int64).reshape(-1)).cuda()
        d_out = torch.zeros(max(1, len(hits)) * f.ALIGNMENT_DTYPE.itemsize, dtype=torch.uint8, device="cuda")
        mid_dev.align_hits_device(d_qb.data_ptr(), d_qo.data_ptr(), len(qs), "edit", 2, d_off.data_ptr(),
                                  d_hits.data_ptr(), len(hits), d_out.data_ptr(), strands=s)
        torch.cuda.synchronize()
        assert d_out.cpu().numpy().tobytes()[:al.nbytes] == al.tobytes(), s
        assert np.array_equal(al["distance"], dist) and np.array_equal(al["n_ops"], dist), s
        per = 2 if s else 1
        for v in range(per * len(qs)):
            q = qs[v // per] if v % per == 0 else rc(qs[v // per])
            for h in range(int(off[v]), int(off[v + 1])):
                g = int(starts[int(hits[h, 0])] + hits[h, 1])
                window = text[g:g + int(al[h]["text_len"])].translate(lut)
                assert apply_ops(q, al[h]).translate(lut) == window, (s, v, h)


# ---- 3. device entry points ------------------------------------------------------------------------------------------

def test_sub_batches_streams_and_nq_1(mid, mid_dev, batches):
    import torch
    qs, want = batches(3)
    qb, qo = pack(qs)
    lo = next(i for i in range(500, 3000) if int(qo[i]) % 64)
    cases = [(lo, lo + 1700), (lo + 3, lo + 4), (len(qs) - 1, len(qs)), (0, 1)]
    stream = torch.cuda.Stream()
    for s in (False, True):
        ref = ref_loci(want[("edit", s)], mid, 3)
        for i, (a, b) in enumerate(cases):
            keep = np.zeros(len(qs), bool)
            keep[a:b] = True
            w = select(ref, keep)
            for st in (None, stream):
                got = device_locate(mid_dev, s, qb, qo, 3, a, b, shift=1 + i % 7, stream=st)
                same(got, w, (s, a, b, st is not None))
                assert np.array_equal(device_count(mid_dev, s, qb, qo, 3, a, b, shift=2 + i % 5, stream=st), w[0])


def test_no_hits_no_distances_and_repeated_calls(mid, mid_dev, batches, refs):
    qs, want = batches(2)
    qb, qo = pack(qs)
    r = np.random.default_rng(5)
    nb, no = pack([rand_bases(r, 80) for _ in range(40)])   # 80 random bases do not occur within 3 edits
    for s in (False, True):
        off, hits, dist = device_locate(mid_dev, s, nb, no, 3)
        assert not off.any() and len(hits) == 0, s
        assert not device_count(mid_dev, s, nb, no, 3).any()
        ref = ref_loci(want[("edit", s)], mid, 2)
        got = device_locate(mid_dev, s, qb, qo, 2, distances=False)
        assert got[2] is None
        same(got, ref, (s, "no distances"))
    first = device_locate(mid_dev, True, qb, qo, 2)
    for i in range(20):
        same(device_locate(mid_dev, True, qb, qo, 2), first, ("call", i))


def test_replica_1(mid, batches):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    qs, want = batches(2)
    qb, qo = pack(qs)
    keep = np.zeros(len(qs), bool)
    keep[7:] = True
    ix = device_from_parts(mid, devices=[0, 1])
    try:
        stream = torch.cuda.Stream(device=1)
        for s in (False, True):
            w = select(ref_loci(want[("edit", s)], mid, 2), keep)
            for st in (None, stream):
                got = device_locate(ix, s, qb, qo, 2, 7, len(qs), shift=5, stream=st, replica=1, device=1)
                same(got, w, (s, st is not None))
                assert np.array_equal(device_count(ix, s, qb, qo, 2, 7, len(qs), stream=st, replica=1, device=1), w[0])
    finally:
        ix.close()


# ---- 4. refused reads and unsupported indexes ------------------------------------------------------------------------

def test_refused_reads(mid, mid_dev):
    from awry_b200 import AwryError
    t = bytes(mid.text)
    k = 2
    good = [t[1000 + 97 * i:1000 + 97 * i + 60] for i in range(30)]
    dollar = bytearray(t[5000:5060])
    dollar[30] = ord("$")
    qs = list(good)
    qs.insert(3, b"")                                      # empty
    qs.insert(10, b"AC")                                   # L <= k
    qs.insert(20, bytes(dollar))                           # a sentinel
    qb, qo = pack(qs)
    starts = np.asarray(mid.seq_starts, np.uint64)
    for s in (False, True):
        got = device_locate(mid_dev, s, qb, qo, k, check=False)
        with pytest.raises(AwryError) as e:
            mid_dev.device_check()
        assert e.value.code == -5 and "query 3" in str(e.value), (s, str(e.value))
        mid_dev.device_check()                             # cleared
        # every read's loci, refused or not, are the filter applied to the device edit locate's result
        poff, phits, pdist = device_locate(mid_dev, s, qb, qo, k, check=False, plain=True)
        with pytest.raises(AwryError):
            mid_dev.device_check()
        pos = starts[phits[:, 0].astype(np.int64)] + phits[:, 1] if len(phits) else np.zeros(0, np.uint64)
        off, keep = loci(poff, pos, pdist, k)
        same(got, (off, phits[keep], pdist[keep]), (s, "refused reads"))
        counts = device_count(mid_dev, s, qb, qo, k, check=False)
        with pytest.raises(AwryError):
            mid_dev.device_check()
        assert np.array_equal(counts.reshape(-1, k + 1).sum(axis=1), np.diff(off.astype(np.int64))), s
        with pytest.raises(AwryError) as e:                # the host calls name the read
            mid_dev.locate_edit_loci_packed(qb, qo, k, strands=s)
        assert e.value.code == -5 and "query 3" in str(e.value)


def test_unsupported_indexes(fx, mid, monkeypatch):
    import torch
    from awry_b200 import AwryError
    qb, qo = pack([bytes(mid.text[1000:1100])])
    d_qb, d_qo = torch.from_numpy(qb).cuda(), torch.from_numpy(qo.view(np.int64)).cuda()
    d_off = torch.zeros(3, dtype=torch.int64, device="cuda")
    d_counts = torch.zeros(8, dtype=torch.int64, device="cuda")
    dna = bytes(mid.text[:20_000])
    cases = [("ratio 1", fx.build_parts(dna, 0, ratio=1, kmer_len=8), None),
             ("AWRY_B200_PAIR_INDEX=0", fx.build_parts(dna, 0, ratio=8, kmer_len=8), ("AWRY_B200_PAIR_INDEX", "0")),
             ("protein", fx.build_parts(fx.gen_text(1, 20_000, 3), 1, ratio=8, kmer_len=3), None),
             ("AWRY_B200_WIDE=1", fx.build_parts(dna, 0, ratio=8, kmer_len=8), ("AWRY_B200_WIDE", "1"))]
    for name, parts, env in cases:
        if env:
            monkeypatch.setenv(*env)
        with device_from_parts(parts) as ix:
            for s in (False, True):
                for call in (lambda: ix.locate_edit_loci_device(d_qb.data_ptr(), d_qo.data_ptr(), 1, 1, d_off.data_ptr(),
                                                                strands=s),
                             lambda: ix.count_edit_loci_device(d_qb.data_ptr(), d_qo.data_ptr(), 1, 1,
                                                               d_counts.data_ptr(), strands=s),
                             lambda: ix.locate_edit_loci_packed(qb, qo, 1, strands=s),
                             lambda: ix.count_edit_loci_packed(qb, qo, 1, strands=s)):
                    with pytest.raises(AwryError) as e:
                        call()
                    assert e.value.code == -6, (name, s)
        if env:
            monkeypatch.delenv(env[0])


# ---- 5. planted reads: one locus each, at its origin ----------------------------------------------------------------

def test_planted_reads_give_one_locus_at_their_origin(fx):
    r = np.random.default_rng(2026)
    n, L = 400_000, 100
    text = rand_bases(r, n)
    parts = fx.build_parts(text, 0, ratio=8, kmer_len=10, seq_starts=np.zeros(1, np.uint64))
    with device_from_parts(parts) as ix:
        for k in (1, 2, 3):
            origins, qs, planted = [], [], []
            for i in range(300):
                o = int(r.integers(0, n - 2 * L))
                q = bytearray(text[o:o + L])
                e = int(r.integers(0, k + 1))
                for at in sorted(r.choice(np.arange(2 * k + 2, L - 2 * k - 2), e, replace=False), reverse=True):
                    op = int(r.integers(0, 3))
                    if op == 0:
                        q[at] = ord("ACGT".replace(chr(q[at]), "")[int(r.integers(0, 3))])
                    elif op == 1:
                        q.insert(int(at), ord("ACGT"[int(r.integers(0, 4))]))
                    else:
                        del q[int(at)]
                origins.append(o)
                qs.append(bytes(q))
                planted.append(e)
            qb, qo = pack(qs)
            off, hits, dist = ix.locate_edit_loci_packed(qb, qo, k)
            poff, _, _ = ix.locate_edit_packed(qb, qo, k)
            several = fewer = 0
            for i, o in enumerate(origins):
                a, b = int(off[i]), int(off[i + 1])
                near = [h for h in range(a, b) if abs(int(hits[h, 1]) - o) <= L]
                assert len(near) == 1, (k, i, o, hits[a:b].tolist(), dist[a:b].tolist())
                h = near[0]
                assert int(hits[h, 1]) == o and int(dist[h]) <= planted[i], (k, i, o, hits[h].tolist(), int(dist[h]))
                if planted[i] < k:                         # d(o + 1) <= d(o) + 1 <= k: several starts
                    fewer += 1
                    several += int(poff[i + 1] - poff[i]) > 1
            assert fewer > 0 and several == fewer, (k, several, fewer)


# ---- 6. the bounds-checked build -------------------------------------------------------------------------------------

def test_on_the_bounds_checked_build():
    """this file against libawry_b200_checked.so (every data-dependent load bounds-checked, layout.cuh): no assert"""
    checked = os.path.join(ROOT, "awry_b200", "libawry_b200_checked.so")
    if os.environ.get("AWRY_B200_LIB"):
        pytest.skip("already running against another build")
    if not os.path.exists(checked):
        subprocess.check_call(["make", "-s", "-C", os.path.join(ROOT, "awry_b200", "csrc"), "checked"])
    env = dict(os.environ, AWRY_B200_LIB=checked)
    out = subprocess.run([sys.executable, "-m", "pytest", "tests/test_gpu_edit_loci.py", "-m", "gpu", "-x", "-q",
                          "-p", "no:cacheprovider", "-k", "not bounds_checked and not replica_1"],
                         cwd=ROOT, env=env, capture_output=True, text=True, timeout=3000)
    tail = out.stdout[-1500:] + out.stderr[-1500:]
    assert out.returncode == 0, tail
    assert " passed" in out.stdout and "Assertion" not in out.stderr, tail
