"""Read mapping: awry_map_batch and awry_map_device, Hamming and edit distance, one strand and both, k = 0 .. 3.

- Reference: `ref_map` of test_map_abi.py applied to the brute-force hits of tests/hamming_brute.c / tests/edit_brute.c
  (edit: their loci, through `loci` of test_edit_loci_abi.py), and to the library's own locate results.  Every field of
  every record is compared bit for bit, and every alignment with awry_align_batch on the primary hit.  Cases: random
  small indexes of the fuzz suite and texts of many lengths with reads at both ends, the multi-record index (more than
  3000 reads), the repeat-rich text (many equal best loci, where the hash choice matters), long and mostly-N reads,
  16-candidate slices, several host chunks, both locate variants, the count variant and the index without the device
  seed table.
- Host and device agree bit for bit; splitting a batch anywhere or reordering it leaves each read's record unchanged.
- Device entry points: sub-batches at unaligned offsets, another stream, replica 1 (two GPUs), nq = 1, a batch without
  hits, aln NULL.
- Refused reads among good ones: the host call names the read, the device call flags and latches it.
- Unsupported indexes are refused.
- Planted reads map to their origin, on their strand, at a distance no larger than their edits.
- The whole file once more against libawry_b200_checked.so."""
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT, device_from_parts
from test_edit_loci_abi import loci
from test_gpu_approx_fuzz import (LENS, awkward_reads, batches, end_reads, expected, fuzz_reads, mid,  # noqa: F401
                                  mid_dev, rand_bases, random_text, refs, select)
from test_gpu_edit import edit, rc
from test_gpu_hamming import repeats  # noqa: F401
from test_map_abi import M64, read_hash, ref_map

pytestmark = pytest.mark.gpu
METRICS = ("hamming", "edit")
COMBOS = [(m, s) for m in METRICS for s in (False, True)]


def pack(qs):
    from awry_b200 import fm_index as f
    return f.pack_queries(qs)


def global_starts(parts, hits):
    starts = np.asarray(parts.seq_starts, np.uint64)
    return starts[hits[:, 0].astype(np.int64)] + hits[:, 1] if len(hits) else np.zeros(0, np.uint64)


def hit_sets(parts, want, metric, k):
    """(hit_off, global starts, distances) of H_v from a locate result (counts, hit_off, hits, dist): the hits
    themselves (Hamming) or their loci (edit)"""
    _, off, hits, dist = want
    pos = global_starts(parts, hits)
    if metric == "edit":
        off, keep = loci(off, pos, dist, k)
        pos, dist = pos[keep], dist[keep]
    return off, pos, dist


def records(parts, ref):
    """ref_map's records -> MAPPING_DTYPE (the primary's start as (seq_idx, local_pos))"""
    from awry_b200 import fm_index as f
    out = np.zeros(len(ref), f.MAPPING_DTYPE)
    starts = np.asarray(parts.seq_starts, np.uint64)
    mapped = ref["start"] != np.uint64(M64)
    seq = np.searchsorted(starts, ref["start"][mapped], side="right").astype(np.uint64) - np.uint64(1)
    out["seq_idx"], out["local_pos"] = np.uint64(M64), np.uint64(M64)
    out["seq_idx"][mapped] = seq
    out["local_pos"][mapped] = ref["start"][mapped] - starts[seq]
    for name in ("n_best", "n_second", "distance", "strand", "mapq", "flags"):
        out[name] = ref[name]
    return out


def same_records(got, want, what):
    g = np.ascontiguousarray(got).view(np.uint8).reshape(-1, 32)
    w = np.ascontiguousarray(want).view(np.uint8).reshape(-1, 32)
    assert g.shape == w.shape, what
    bad = np.nonzero(np.any(g != w, axis=1))[0]
    assert len(bad) == 0, what + ("reads", bad[:5].tolist(), got[bad[:3]].tolist(), want[bad[:3]].tolist())


def no_alignment(k):
    from awry_b200 import fm_index as f
    a = np.zeros(1, f.ALIGNMENT_DTYPE)
    a["distance"] = k + 1
    return a[0]


def check_alignments(dev, qb, qo, metric, k, strands, recs, aln, what):
    """aln[q] = awry_align_batch on the primary hit of v = (q << strands) | strand; "no alignment" when unmapped"""
    from awry_b200 import fm_index as f
    per = 2 if strands else 1
    nq = len(recs)
    mapped = (recs["flags"] & f.MAP_UNMAPPED) == 0
    v = np.arange(nq) * per + recs["strand"].astype(np.int64)
    counts = np.zeros(per * nq, np.uint64)
    counts[v[mapped]] = 1
    off = np.zeros(per * nq + 1, np.uint64)
    off[1:] = np.cumsum(counts)
    hits = np.stack([recs["seq_idx"][mapped], recs["local_pos"][mapped]], axis=1).astype(np.uint64)
    want = dev.align_hits_packed(qb, qo, metric, k, off, hits, strands=strands)
    assert aln[mapped].tobytes() == want.tobytes(), what + ("alignments",)
    assert np.all(aln[~mapped] == no_alignment(k)), what + ("no alignment",)


def device_map(dev, qb, qo, metric, k, strands, lo=0, hi=None, shift=0, stream=None, replica=0, device=0, align=True,
               check=True):
    """map_device on reads lo .. hi: the bytes behind `shift` garbage bytes, d_qoff at entry lo of the whole batch's
    offsets, the outputs filled with garbage -> (records, alignments or None)"""
    import torch
    from awry_b200 import fm_index as f
    hi = len(qo) - 1 if hi is None else hi
    nq = hi - lo
    dv = torch.device("cuda", device)
    with torch.cuda.device(dv):
        d_qb = torch.from_numpy(np.concatenate([np.full(shift, ord("#"), np.uint8), qb])).to(dv)
        d_qo = torch.from_numpy(np.ascontiguousarray(qo, np.uint64).view(np.int64)).to(dv)
        d_out = torch.full((max(1, nq) * 32,), 0x5a, dtype=torch.uint8, device=dv)
        d_aln = torch.full((max(1, nq) * 44,), 0x5a, dtype=torch.uint8, device=dv) if align else None
        st = stream if stream is not None else torch.cuda.current_stream(dv)
        st.wait_stream(torch.cuda.current_stream(dv))
        dev.map_device(d_qb.data_ptr() + shift, d_qo.data_ptr() + 8 * lo, nq, metric, k, d_out.data_ptr(),
                       d_aln.data_ptr() if align else None, strands=strands, stream=st.cuda_stream, replica=replica)
        if check:
            dev.device_check(st.cuda_stream, replica)
        st.synchronize()
        recs = d_out.cpu().numpy()[:nq * 32].view(f.MAPPING_DTYPE)
        aln = d_aln.cpu().numpy()[:nq * 44].view(f.ALIGNMENT_DTYPE) if align else None
        return recs, aln


def library_hits(dev, metric, strands, qb, qo, k):
    """the library's own H_v: the Hamming locate, or the edit loci locate"""
    if metric == "edit":
        return dev.locate_edit_loci_packed(qb, qo, k, strands=strands)
    call = dev.locate_hamming_strands_packed if strands else dev.locate_hamming_packed
    return call(qb, qo, k)


def check(dev, parts, qs, k, metric, strands, refs, tag, want=None, device=True, own=True):
    """the host call (with and without alignments) against ref_map on the brute-force reference, its alignments
    against awry_align_batch, the device call against the host call, and ref_map on the library's own locate"""
    what = (tag, metric, "both strands" if strands else "one strand", "k=%d" % k)
    want = want if want is not None else expected(refs, metric, strands, parts, qs, k)
    ref = records(parts, ref_map(*hit_sets(parts, want, metric, k), qs, k, strands))
    qb, qo = pack(qs)
    recs, aln = dev.map_packed(qb, qo, metric, k, strands=strands)
    same_records(recs, ref, what + ("host",))
    check_alignments(dev, qb, qo, metric, k, strands, recs, aln, what)
    bare, none = dev.map_packed(qb, qo, metric, k, strands=strands, align=False)
    assert none is None and bare.tobytes() == recs.tobytes(), what
    if own:
        off, hits, dist = library_hits(dev, metric, strands, qb, qo, k)
        same_records(recs, records(parts, ref_map(off, global_starts(parts, hits), dist, qs, k, strands)),
                     what + ("library locate",))
    if device:
        drecs, daln = device_map(dev, qb, qo, metric, k, strands)
        assert drecs.tobytes() == recs.tobytes() and daln.tobytes() == aln.tobytes(), what + ("device",)
    return recs, aln


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
            for m, s in COMBOS:
                check(ix, parts, qs, k, m, s, refs, "seed %d" % seed)


SWEEP = list(range(1, 40, 3)) + [63, 64, 65, 127, 128, 129, 320, 321, 328]


@pytest.mark.parametrize("n", SWEEP)
def test_text_length(fx, refs, n):
    r = np.random.default_rng(n)
    t = rand_bases(r, n) if n % 3 else random_text(r, n)
    parts = fx.build_parts(t, 0, ratio=8, kmer_len=int(1 + n % 9), seq_starts=np.zeros(1, np.uint64))
    with device_from_parts(parts) as ix:
        for k in (0, 1, 2, 3):
            lens = sorted({k + 1, k + 2, 8, 9, 17, 33, 65, n - 1, n, n + 1})
            qs = [q for q in end_reads(t, r, [ln for ln in lens if ln > max(k, 1)]) if len(q) > k]
            for m, s in COMBOS:
                check(ix, parts, qs, k, m, s, refs, "n=%d" % n, own=False)


@pytest.mark.parametrize("k", [0, 1, 2, 3])
def test_mid_index(k, mid, mid_dev, batches, refs):
    qs, want = batches(max(k, 1))                          # (k = 0 takes k = 1's reads)
    for m, s in COMBOS:
        recs, _ = check(mid_dev, mid, qs, k, m, s, refs, "mid", want[(m, s)] if k else None)
        assert ((recs["flags"] & 1) == 0).sum() > 100 and (recs["mapq"] == (37 if k else 25)).any()


ROUTES = ["slice_16", "locate_chunk_q_1024", "locate_variant_1", "locate_variant_2", "count_variant_1", "kmer_dev_0"]


@pytest.mark.parametrize("route", ROUTES)
def test_route(route, mid, mid_dev, batches, refs, monkeypatch):
    from awry_b200 import fm_index as f
    qs, want = batches(3)
    dev = mid_dev
    try:
        if route == "slice_16":                            # (reads of a few symbols have 10^5 candidates)
            monkeypatch.setenv("AWRY_B200_HAMMING_SLICE", "16")
            keep = np.array([len(q) >= 40 for q in qs])
            qs = [q for q in qs if len(q) >= 40]
            want = {c: select(w, keep) for c, w in want.items()}
        elif route == "locate_chunk_q_1024":
            monkeypatch.setenv("AWRY_B200_LOCATE_CHUNK_Q", "1024")
        elif route.startswith("locate_variant"):
            f.set_locate_variant(int(route[-1]))
        elif route == "count_variant_1":
            f.set_count_variant(1)
        else:
            monkeypatch.setenv("AWRY_B200_KMER_DEV", "0")
            dev = device_from_parts(mid)
        for m, s in COMBOS:
            check(dev, mid, qs, 3, m, s, refs, route, want[(m, s)], own=False)
    finally:
        f.set_locate_variant(0)
        f.set_count_variant(0)
        if dev is not mid_dev:
            dev.close()


def test_repeat_rich_text(repeats, refs, monkeypatch):  # noqa: F811
    parts, ix, qb, qo = repeats
    qs = [bytes(qb[int(qo[i]):int(qo[i + 1])]) for i in range(len(qo) - 1)]
    monkeypatch.setenv("AWRY_B200_HAMMING_SLICE", "300")
    spread = 0
    for k in (1, 2):
        for m, s in COMBOS:
            recs, _ = check(ix, parts, qs, k, m, s, refs, "repeats")
            many = recs["n_best"] >= 2
            assert recs["n_best"].max() >= 20 and not recs["mapq"][many].any()
            # the primary is not always the first best start: B[h mod n_best]
            spread += int((np.array([read_hash(q) for q in qs], dtype=object)[many] % recs["n_best"][many] != 0).sum())
    assert spread > 20


@pytest.mark.parametrize("k", [1, 3])
def test_long_and_awkward_reads(k, mid, mid_dev, refs):
    qs = awkward_reads(mid, k, seed=60 + k)
    for m, s in COMBOS:
        check(mid_dev, mid, qs, k, m, s, refs, "awkward")


# ---- 2. batches: split, reordered, chunked, device entry points -----------------------------------------------------

def test_split_and_reordered_batches(mid, mid_dev, batches):
    qs, _ = batches(2)
    qs = qs[:1500]
    for m, s in COMBOS:
        whole, wa = mid_dev.map_packed(*pack(qs), m, 2, strands=s)
        perm = np.random.default_rng(3).permutation(len(qs))
        pr, pa = mid_dev.map_packed(*pack([qs[i] for i in perm]), m, 2, strands=s)
        assert pr.tobytes() == whole[perm].tobytes() and pa.tobytes() == wa[perm].tobytes(), (m, s)
        for cut in (1, 333, 1000, 1499):
            a, _ = mid_dev.map_packed(*pack(qs[:cut]), m, 2, strands=s)
            b, _ = mid_dev.map_packed(*pack(qs[cut:]), m, 2, strands=s)
            assert np.concatenate([a, b]).tobytes() == whole.tobytes(), (m, s, cut)


def test_device_sub_batches_streams_and_nq_1(mid, mid_dev, batches):
    import torch
    qs, _ = batches(3)
    qb, qo = pack(qs)
    lo = next(i for i in range(500, 3000) if int(qo[i]) % 64)
    cases = [(lo, lo + 1700), (lo + 3, lo + 4), (len(qs) - 1, len(qs)), (0, 1)]
    stream = torch.cuda.Stream()
    for c, (m, s) in enumerate(COMBOS):
        whole, wa = mid_dev.map_packed(qb, qo, m, 3, strands=s)
        for i, (a, b) in enumerate(cases):
            for st in (None, stream):
                got, ga = device_map(mid_dev, qb, qo, m, 3, s, a, b, shift=1 + (c + i) % 7, stream=st)
                assert got.tobytes() == whole[a:b].tobytes() and ga.tobytes() == wa[a:b].tobytes(), (m, s, a, b)
        got, ga = device_map(mid_dev, qb, qo, m, 3, s, lo, lo + 900, align=False)
        assert ga is None and got.tobytes() == whole[lo:lo + 900].tobytes(), (m, s)


def test_no_hits_and_repeated_calls(mid, mid_dev, batches):
    from awry_b200 import fm_index as f
    r = np.random.default_rng(5)
    nb, no = pack([rand_bases(r, 80) for _ in range(40)])   # 80 random bases do not occur within 3 edits
    for m, s in COMBOS:
        for k in (0, 3):
            for recs, aln in (mid_dev.map_packed(nb, no, m, k, strands=s), device_map(mid_dev, nb, no, m, k, s)):
                assert np.all(recs["flags"] == f.MAP_UNMAPPED) and np.all(recs["distance"] == k + 1)
                assert np.all(recs["seq_idx"] == np.uint64(M64)) and np.all(recs["local_pos"] == np.uint64(M64))
                assert not recs["n_best"].any() and not recs["mapq"].any() and not recs["pad"].any()
                assert np.all(aln == no_alignment(k))
    qs, _ = batches(2)
    qb, qo = pack(qs[:800])
    first = device_map(mid_dev, qb, qo, "edit", 2, True)
    for i in range(10):
        again = device_map(mid_dev, qb, qo, "edit", 2, True)
        assert again[0].tobytes() == first[0].tobytes() and again[1].tobytes() == first[1].tobytes(), i


def test_replica_1(mid, batches):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    qs, _ = batches(2)
    qb, qo = pack(qs)
    ix = device_from_parts(mid, devices=[0, 1])
    try:
        stream = torch.cuda.Stream(device=1)
        for m, s in COMBOS:
            whole, wa = ix.map_packed(qb, qo, m, 2, strands=s)     # (split over both replicas)
            one, oa = device_from_parts(mid).map_packed(qb, qo, m, 2, strands=s)
            assert whole.tobytes() == one.tobytes() and wa.tobytes() == oa.tobytes(), (m, s)
            for st in (None, stream):
                got, ga = device_map(ix, qb, qo, m, 2, s, 7, len(qs), shift=5, stream=st, replica=1, device=1)
                assert got.tobytes() == whole[7:].tobytes() and ga.tobytes() == wa[7:].tobytes(), (m, s)
    finally:
        ix.close()


# ---- 3. refused reads and unsupported indexes ------------------------------------------------------------------------

def test_refused_reads(mid, mid_dev):
    from awry_b200 import AwryError
    from awry_b200 import fm_index as f
    t = bytes(mid.text)
    k = 2
    good = [t[1000 + 97 * i:1000 + 97 * i + 60] for i in range(30)]
    dollar = bytearray(t[5000:5060])
    dollar[30] = ord("$")
    qs = list(good)
    qs.insert(3, b"")                                      # empty
    qs.insert(10, b"AC")                                   # L <= k
    qs.insert(20, bytes(dollar))                           # a sentinel (its pieces do occur in the text)
    bad = [3, 10, 20]
    qb, qo = pack(qs)
    for m, s in COMBOS:
        with pytest.raises(AwryError) as e:                # the host call names the read
            mid_dev.map_packed(qb, qo, m, k, strands=s)
        assert e.value.code == -5 and "query 3" in str(e.value), (m, s, str(e.value))
        recs, aln = device_map(mid_dev, qb, qo, m, k, s, check=False)
        with pytest.raises(AwryError) as e:
            mid_dev.device_check()
        assert e.value.code == -5 and "query 3" in str(e.value), (m, s, str(e.value))
        mid_dev.device_check()                             # cleared
        assert np.all(recs["flags"][bad] == f.MAP_UNMAPPED | f.MAP_REFUSED), (m, s)
        assert np.all(recs["distance"][bad] == k + 1) and not recs["n_best"][bad].any()
        assert np.all(aln[bad] == no_alignment(k))
        ok = np.setdiff1d(np.arange(len(qs)), bad)
        want, wa = mid_dev.map_packed(*pack([qs[i] for i in ok]), m, k, strands=s)
        assert recs[ok].tobytes() == want.tobytes() and aln[ok].tobytes() == wa.tobytes(), (m, s)


def test_unsupported_indexes(fx, mid, monkeypatch):
    import torch
    from awry_b200 import AwryError
    qb, qo = pack([bytes(mid.text[1000:1100])])
    d_qb, d_qo = torch.from_numpy(qb).cuda(), torch.from_numpy(qo.view(np.int64)).cuda()
    d_out = torch.zeros(64, dtype=torch.uint8, device="cuda")
    dna = bytes(mid.text[:20_000])
    cases = [("ratio 1", fx.build_parts(dna, 0, ratio=1, kmer_len=8), None),
             ("AWRY_B200_PAIR_INDEX=0", fx.build_parts(dna, 0, ratio=8, kmer_len=8), ("AWRY_B200_PAIR_INDEX", "0")),
             ("protein", fx.build_parts(fx.gen_text(1, 20_000, 3), 1, ratio=8, kmer_len=3), None),
             ("AWRY_B200_WIDE=1", fx.build_parts(dna, 0, ratio=8, kmer_len=8), ("AWRY_B200_WIDE", "1"))]
    for name, parts, env in cases:
        if env:
            monkeypatch.setenv(*env)
        with device_from_parts(parts) as ix:
            for m, s in COMBOS:
                for call in (lambda: ix.map_packed(qb, qo, m, 1, strands=s),
                             lambda: ix.map_device(d_qb.data_ptr(), d_qo.data_ptr(), 1, m, 1, d_out.data_ptr(),
                                                   strands=s)):
                    with pytest.raises(AwryError) as e:
                        call()
                    assert e.value.code == -6, (name, m, s)
        if env:
            monkeypatch.delenv(env[0])


# ---- 4. planted reads map to their origin ----------------------------------------------------------------------------

def test_planted_reads_map_to_their_origin(fx):
    from awry_b200 import fm_index as f
    r = np.random.default_rng(2027)
    n, L = 400_000, 100
    text = rand_bases(r, n)
    parts = fx.build_parts(text, 0, ratio=8, kmer_len=10, seq_starts=np.zeros(1, np.uint64))
    with device_from_parts(parts) as ix:
        for m in METRICS:
            for k in (1, 2, 3):
                origins, qs, planted = [], [], []
                for i in range(300):
                    o = int(r.integers(0, n - 2 * L))
                    q = bytearray(text[o:o + L])
                    e = i % (k + 1)
                    for at in sorted(r.choice(np.arange(2 * k + 2, L - 2 * k - 2), e, replace=False), reverse=True):
                        edit(q, int(at), 0 if m == "hamming" else int(r.integers(0, 3)), r)
                    origins.append(o)
                    qs.append(rc(bytes(q)) if i % 2 else bytes(q))
                    planted.append(e)
                recs, aln = ix.map_packed(*pack(qs), m, k, strands=True)
                for i, rec in enumerate(recs):
                    assert rec["flags"] == 0 and rec["strand"] == i % 2, (m, k, i, rec)
                    assert abs(int(rec["local_pos"]) - origins[i]) <= L and rec["distance"] <= planted[i], (m, k, i, rec)
                    assert rec["n_best"] == 1 and rec["mapq"] > 0, (m, k, i, rec)
                    assert aln[i]["distance"] == rec["distance"] and aln[i]["n_ops"] == rec["distance"]
                assert (recs["mapq"] == 37).sum() > 100, (m, k)


# ---- 5. the bounds-checked build -------------------------------------------------------------------------------------

def test_on_the_bounds_checked_build():
    """this file against libawry_b200_checked.so (every data-dependent load bounds-checked, layout.cuh): no assert"""
    checked = os.path.join(ROOT, "awry_b200", "libawry_b200_checked.so")
    if os.environ.get("AWRY_B200_LIB"):
        pytest.skip("already running against another build")
    if not os.path.exists(checked):
        subprocess.check_call(["make", "-s", "-C", os.path.join(ROOT, "awry_b200", "csrc"), "checked"])
    env = dict(os.environ, AWRY_B200_LIB=checked)
    out = subprocess.run([sys.executable, "-m", "pytest", "tests/test_gpu_map.py", "-m", "gpu", "-x", "-q",
                          "-p", "no:cacheprovider", "-k", "not bounds_checked and not replica_1"],
                         cwd=ROOT, env=env, capture_output=True, text=True, timeout=3000)
    tail = out.stdout[-1500:] + out.stderr[-1500:]
    assert out.returncode == 0, tail
    assert " passed" in out.stdout and "Assertion" not in out.stderr, tail
