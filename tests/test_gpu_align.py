"""Alignment of located hits: awry_align_batch and awry_align_device against the brute-force reference
tests/align_brute.c, on the hits of every approximate locate entry point (locate_{hamming,edit}[_strands]_packed and
_device).  Every case compares every field of every alignment bit for bit, and checks what the header promises: the
distance is the locate call's, n_ops equals it, and applying the ops to Q (rc(q) for a reverse-strand hit) gives exactly
the window text[s .. s+text_len) of the fixture's text.

- Both metrics, both strand counts, k = 0 .. 3, on the multi-record index of test_gpu_approx_fuzz.py (more than 3000
  reads, every other one reverse-complemented), a few of its random small indexes, texts shorter than the reads with
  reads at both ends, the repeat-rich text of test_gpu_hamming.py (AWRY_B200_HAMMING_SLICE=300: many slices), and reads
  up to 8000 bp, chimeric and mostly-N reads.
- Hand-placed hits get "no alignment": past the end of the text, seq_idx out of range, windows over k.
- Device call: a sub-batch from the middle of a device buffer (first offset not a multiple of 64, data pointer + 1 .. 7
  bytes), a torch.cuda.Stream() other than the default, n_hits = 0, 20 calls in a row, replica 1 of a two-GPU handle;
  refused reads among good ones (latched for device_check, their hits "no alignment"); unsupported indexes.
- The whole file once more against libawry_b200_checked.so."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT, device_from_parts
from test_gpu_approx_fuzz import (COMBOS, LENS, awkward_reads, batches, end_reads, fuzz_reads, mid,  # noqa: F401
                                  mid_dev, rand_bases, random_text, refs)
from test_gpu_hamming import repeats  # noqa: F401

pytestmark = pytest.mark.gpu
LETTERS = np.frombuffer(b"$ACGNT", np.uint8)
COMP = np.array([0, 5, 3, 2, 4, 1], np.uint8)


def fm():
    from awry_b200 import fm_index as f
    return f


def sfx(strands):
    return "_strands" if strands else ""


@pytest.fixture(scope="module")
def abrute(tmp_path_factory, po):
    so = str(tmp_path_factory.mktemp("align") / "libalign_brute.so")
    subprocess.check_call(["gcc", "-O2", "-fopenmp", "-shared", "-fPIC", "-o", so, os.path.join(ROOT, "tests", "align_brute.c")])
    fn = C.CDLL(so).align_brute
    fn.restype = C.c_int64
    fn.argtypes = [C.c_void_p] * 2 + [C.c_uint64, C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint32,
                                      C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p]
    lut = np.array([po.lib().awo_ascii_to_index(0, c) for c in range(256)], dtype=np.uint8)
    return fn, lut


def brute(abrute, parts, qs, metric, strands, k, off, hits):
    fn, lut = abrute
    qb, qo = fm().pack_queries(qs)
    text = np.ascontiguousarray(parts.text, dtype=np.uint8)
    starts = np.ascontiguousarray(parts.seq_starts, dtype=np.uint64)
    off = np.ascontiguousarray(off, np.uint64)
    hits = np.ascontiguousarray(hits, np.uint64).reshape(-1, 2)
    out = np.zeros(max(1, len(hits)), fm().ALIGNMENT_DTYPE)
    assert fn(lut.ctypes.data, text.ctypes.data, len(text), starts.ctypes.data, len(starts), qb.ctypes.data, qo.ctypes.data,
              len(qs), {"hamming": 0, "edit": 1}[metric], int(strands), k, off.ctypes.data, hits.ctypes.data,
              out.ctypes.data) == len(hits)
    return out[:len(hits)]


def replay(abrute, parts, qs, strands, off, hits, dist, al, what):
    """the header's promise for every hit: distance, n_ops, and the ops turn Q into text[s .. s+text_len)"""
    _, lut = abrute
    assert np.array_equal(al["distance"], dist), what + ("distance",)
    assert np.array_equal(al["n_ops"], dist), what + ("n_ops",)
    tl = LETTERS[lut[np.asarray(parts.text, np.uint8)]].tobytes()
    starts = np.asarray(parts.seq_starts, np.uint64)
    per = 2 if strands else 1
    for v in range(per * len(qs)):
        q = LETTERS[lut[np.frombuffer(qs[v // per], np.uint8)]]
        if strands and v % 2:
            q = LETTERS[COMP[lut[np.frombuffer(qs[v // per], np.uint8)]][::-1]]
        q = q.tobytes()
        for h in range(int(off[v]), int(off[v + 1])):
            a = al[h]
            s = int(starts[hits[h, 0]] + hits[h, 1])
            got, at = bytearray(), 0
            for t in range(int(a["n_ops"])):
                o = a["ops"][t]
                op, qp, tp = chr(o["op"]), int(o["qpos"]), int(o["tpos"])
                got += q[at:qp]
                assert tp == len(got), what + (h, "tpos")
                if op in "XI":
                    assert o["query_sym"] == q[qp], what + (h, "query_sym")
                if op in "XD":
                    assert o["text_sym"] == tl[s + tp], what + (h, "text_sym")
                    got.append(tl[s + tp])
                at = qp + (op != "D")
            got += q[at:]
            assert bytes(got) == tl[s:s + int(a["text_len"])], what + (h, "window")


def same(got, want, what):
    bad = np.nonzero(got.view(np.uint8).reshape(-1, 44) != want.view(np.uint8).reshape(-1, 44))[0]
    assert len(bad) == 0, what + ("alignments", bad[:5], got[bad[:3]], want[bad[:3]])


def to_host(ptr, nbytes):
    out = np.zeros(max(1, nbytes), np.uint8)
    if nbytes:
        assert C.CDLL("libcudart.so").cudaMemcpy(C.c_void_p(out.ctypes.data), C.c_void_p(ptr), C.c_size_t(nbytes), 2) == 0
    return out[:nbytes]


def device_align(dev, metric, strands, qb, qo, k, lo=0, hi=None, shift=0, stream=None, replica=0, device=0, check=True):
    """locate_*_device on reads lo .. hi (bytes behind `shift` garbage bytes, d_qoff at entry lo of the whole batch's
    offsets), then align_hits_device on its device outputs -> (hit_off, hits, dist, alignments)"""
    import torch
    hi = len(qo) - 1 if hi is None else hi
    nq, per = hi - lo, 2 if strands else 1
    dv = torch.device("cuda", device)
    with torch.cuda.device(dv):
        d_qb = torch.from_numpy(np.concatenate([np.full(shift, ord("#"), np.uint8), qb])).to(dv)
        d_qo = torch.from_numpy(np.ascontiguousarray(qo, np.uint64).view(np.int64)).to(dv)
        d_off = torch.full((per * nq + 1,), -3, dtype=torch.int64, device=dv)
        st = stream if stream is not None else torch.cuda.current_stream(dv)
        st.wait_stream(torch.cuda.current_stream(dv))
        hp, dp, n = getattr(dev, f"locate_{metric}{sfx(strands)}_device")(
            d_qb.data_ptr() + shift, d_qo.data_ptr() + 8 * lo, nq, k, d_off.data_ptr(), stream=st.cuda_stream,
            replica=replica)
        with torch.cuda.stream(st):
            d_out = torch.full((max(1, n) * 44,), 0xAB, dtype=torch.uint8, device=dv)
        dev.align_hits_device(d_qb.data_ptr() + shift, d_qo.data_ptr() + 8 * lo, nq, metric, k, d_off.data_ptr(),
                              hp or 0, n, d_out.data_ptr(), strands=strands, stream=st.cuda_stream, replica=replica)
        if check:
            dev.device_check(st.cuda_stream, replica)
        st.synchronize()
        hits = to_host(hp, n * 16).view(np.uint64).reshape(-1, 2)
        dist = to_host(dp, n).view(np.uint8)
        dev.device_free(hp, replica)
        dev.device_free(dp, replica)
        al = d_out.cpu().numpy()[:n * 44].copy().view(fm().ALIGNMENT_DTYPE)
        return d_off.cpu().numpy().view(np.uint64), hits, dist, al


def check(dev, parts, qs, k, metric, strands, abrute, tag, device=True):
    """host locate -> host align, and device locate -> device align, against the reference and the promise"""
    what = (tag, metric, "both strands" if strands else "one strand", "k=%d" % k)
    qb, qo = fm().pack_queries(qs)
    off, hits, dist = getattr(dev, f"locate_{metric}{sfx(strands)}_packed")(qb, qo, k)
    want = brute(abrute, parts, qs, metric, strands, k, off, hits)
    got = dev.align_hits_packed(qb, qo, metric, k, off, hits, strands=strands)
    same(got, want, what + ("host",))
    replay(abrute, parts, qs, strands, off, hits, dist, got, what)
    if device:
        doff, dhits, ddist, dal = device_align(dev, metric, strands, qb, qo, k)
        assert np.array_equal(doff, off) and np.array_equal(dhits, hits) and np.array_equal(ddist, dist), what
        same(dal, want, what + ("device",))
    return off, hits, dist, got


# ---- 1. every metric, strand count and k ---------------------------------------------------------------------------

@pytest.mark.parametrize("k", [0, 1, 2, 3])
def test_mid_index(k, mid, mid_dev, batches, abrute):
    qs, _ = batches(max(k, 1))
    for m, s in COMBOS:
        check(mid_dev, mid, qs, k, m, s, abrute, "mid")


@pytest.mark.parametrize("seed", [0, 3, 5, 11])
def test_random_index(fx, abrute, seed):
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
                check(ix, parts, qs, k, m, s, abrute, "seed %d" % seed)


@pytest.mark.parametrize("n", [1, 5, 17, 63, 64, 65, 129])
def test_short_texts_and_ends(fx, abrute, n):
    r = np.random.default_rng(n)
    t = rand_bases(r, n) if n % 3 else random_text(r, n)
    parts = fx.build_parts(t, 0, ratio=8, kmer_len=int(1 + n % 9), seq_starts=np.zeros(1, np.uint64))
    with device_from_parts(parts) as ix:
        for k in (0, 1, 3):
            lens = sorted({k + 1, k + 2, 9, 33, 65, n - 1, n, n + 1, n + k + 1})
            qs = [q for q in end_reads(t, r, [ln for ln in lens if ln > max(k, 0)]) if len(q) > k]
            for m, s in COMBOS:
                check(ix, parts, qs, k, m, s, abrute, "n=%d" % n)


def test_repeat_rich_text(repeats, abrute, monkeypatch):  # noqa: F811
    parts, ix, qb, qo = repeats
    qs = [bytes(qb[int(qo[i]):int(qo[i + 1])]) for i in range(len(qo) - 1)]
    monkeypatch.setenv("AWRY_B200_HAMMING_SLICE", "300")   # many slices of hits in one call
    for m, s in COMBOS:
        off, _, _, _ = check(ix, parts, qs, 2, m, s, abrute, "repeats")
        assert np.diff(off.astype(np.int64)).max() >= 200, (m, s)


def test_long_and_awkward_reads(mid, mid_dev, abrute):
    from test_gpu_edit import edit
    qs = awkward_reads(mid, 2, seed=80)                    # 1000 - 8000 bp, chimeric, across N runs, mostly N
    r = np.random.default_rng(81)
    t = bytes(mid.text)
    for i in range(6):                                     # 8000 bp with 0 .. 2 edits, one at the text's end
        p = len(t) - 8000 if i == 5 else int(r.integers(0, len(t) - 8000))
        q = bytearray(t[p:p + 8000])
        for _ in range(i % 3):
            edit(q, int(r.integers(0, len(q))), int(r.integers(0, 3)), r)
        qs.append(bytes(q))
    assert max(len(q) for q in qs) >= 8000
    for k in (1, 3):
        for m, s in COMBOS:
            check(mid_dev, mid, qs, k, m, s, abrute, "awkward")


# ---- 2. hand-placed hits --------------------------------------------------------------------------------------------

def test_hand_placed_hits_without_alignment(mid, mid_dev, abrute):
    t = bytes(mid.text)
    starts = np.asarray(mid.seq_starts, np.uint64)
    n = len(t)
    q = t[2000:2100]
    far = bytearray(t[3000:3100])
    for i in range(0, 100, 20):                            # 5 substitutions
        far[i] = ord("A") if far[i] != ord("A") else ord("C")
    qs = [q, bytes(far)]
    last = len(starts) - 1
    end = int(n - starts[last])                            # local position of the text's end in the last record
    hits = np.array([[0, 2000], [0, 2001],                 # the exact window, and one start off (Hamming: over k)
                     [last, end - 50], [last, end], [last, end + 7], [len(starts), 5], [1 << 40, 0], [0, (1 << 64) - 9],
                     [0, 3000]], np.uint64)                # `far` at its origin: 5 substitutions
    off = np.array([0, 8, 9], np.uint64)
    qb, qo = fm().pack_queries(qs)
    for metric in ("hamming", "edit"):
        for k in (0, 1, 3):
            got = mid_dev.align_hits_packed(qb, qo, metric, k, off, hits)
            same(got, brute(abrute, mid, qs, metric, False, k, off, hits), (metric, k))
            assert got[0]["distance"] == 0 and got[0]["text_len"] == 100, (metric, k)
            none = [3, 4, 5, 6, 7, 8] + ([1, 2] if metric == "hamming" else [])
            assert (got[none]["distance"] == k + 1).all() and not got[none]["n_ops"].any(), (metric, k)
            assert not got[none]["text_len"].any() and not got[none]["ops"].view(np.uint8).any(), (metric, k)


# ---- 3. the device entry point --------------------------------------------------------------------------------------

def test_sub_batches_streams_and_repeated_calls(mid, mid_dev, batches, abrute):
    import torch
    qs, _ = batches(3)
    qb, qo = fm().pack_queries(qs)
    lo = next(i for i in range(500, 3000) if int(qo[i]) % 64)
    stream = torch.cuda.Stream()
    for c, (m, s) in enumerate(COMBOS):
        for i, (a, b) in enumerate([(lo, lo + 1700), (lo + 3, lo + 4), (len(qs) - 1, len(qs))]):
            for st in (None, stream):
                off, hits, dist, al = device_align(mid_dev, m, s, qb, qo, 3, a, b, shift=1 + (c * 3 + i) % 7, stream=st)
                sub = qs[a:b]
                same(al, brute(abrute, mid, sub, m, s, 3, off, hits), (m, s, a, b, st is not None))
                replay(abrute, mid, sub, s, off, hits, dist, al, (m, s, a, b))
    first = device_align(mid_dev, "edit", True, qb, qo, 2)
    for i in range(20):
        got = device_align(mid_dev, "edit", True, qb, qo, 2)
        assert all(np.array_equal(x.view(np.uint8), y.view(np.uint8)) for x, y in zip(got, first)), i


def test_no_hits(mid, mid_dev):
    import torch
    r = np.random.default_rng(5)
    nohit = [rand_bases(r, 80) for _ in range(40)]
    qb, qo = fm().pack_queries(nohit)
    for m, s in COMBOS:
        off, hits, dist, al = device_align(mid_dev, m, s, qb, qo, 3)
        assert not off.any() and len(al) == 0, (m, s)
        assert len(mid_dev.align_hits_packed(qb, qo, m, 3, off, hits, strands=s)) == 0
    # n_hits = 0 with null hit and output pointers
    d_qb, d_qo = torch.from_numpy(qb).cuda(), torch.from_numpy(qo.view(np.int64)).cuda()
    d_off = torch.zeros(81, dtype=torch.int64, device="cuda")
    mid_dev.align_hits_device(d_qb.data_ptr(), d_qo.data_ptr(), 40, "edit", 3, d_off.data_ptr(), 0, 0, 0, strands=True)
    mid_dev.device_check()


def test_replica_1(mid, batches, abrute):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    qs, _ = batches(2)
    qb, qo = fm().pack_queries(qs)
    ix = device_from_parts(mid, devices=[0, 1])
    try:
        stream = torch.cuda.Stream(device=1)
        for m, s in COMBOS:
            for st in (None, stream):
                off, hits, dist, al = device_align(ix, m, s, qb, qo, 2, 7, len(qs), shift=5, stream=st, replica=1, device=1)
                same(al, brute(abrute, mid, qs[7:], m, s, 2, off, hits), (m, s, st is not None))
            # the host call splits the reads across both replicas
            check(ix, mid, qs, 2, m, s, abrute, "two replicas", device=False)
    finally:
        ix.close()


# ---- 4. refused reads and unsupported indexes ----------------------------------------------------------------------

def test_refused_reads(mid, mid_dev, abrute):
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
    qb, qo = fm().pack_queries(qs)
    for m, s in COMBOS:
        per = 2 if s else 1
        off, hits, dist, al = device_align(mid_dev, m, s, qb, qo, k, check=False)
        with pytest.raises(AwryError) as e:
            mid_dev.device_check()
        assert e.value.code == -5 and "query 3" in str(e.value), (m, s, str(e.value))
        mid_dev.device_check()                             # cleared
        same(al, brute(abrute, mid, qs, m, s, k, off, hits), (m, s))
        owner = np.repeat(np.arange(per * len(qs)) // per, np.diff(off.astype(np.int64)))
        bad = np.isin(owner, [3, 10, 20])
        assert bad.any() and (al[bad]["distance"] == k + 1).all() and not al[bad]["n_ops"].any(), (m, s)
        assert (al[~bad]["distance"] == dist[~bad]).all(), (m, s)
        # the host call refuses the batch, naming the first refused read
        with pytest.raises(AwryError) as e:
            mid_dev.align_hits_packed(qb, qo, m, k, off, hits, strands=s)
        assert e.value.code == -5 and "query 3" in str(e.value), (m, s, str(e.value))
        ok = [q for i, q in enumerate(qs) if i not in (3, 10)]
        ob, oo = fm().pack_queries(ok)
        with pytest.raises(AwryError) as e:                # the '$' read, now read 18
            mid_dev.align_hits_packed(ob, oo, m, k, np.zeros(per * len(ok) + 1, np.uint64), np.zeros((0, 2), np.uint64),
                                      strands=s)
        assert e.value.code == -5 and "query 18" in str(e.value), (m, s, str(e.value))


def test_unsupported_indexes(fx, mid, monkeypatch):
    import torch
    from awry_b200 import AwryError
    qb, qo = fm().pack_queries([bytes(mid.text[1000:1100])])
    d_qb, d_qo = torch.from_numpy(qb).cuda(), torch.from_numpy(qo.view(np.int64)).cuda()
    d_off = torch.zeros(3, dtype=torch.int64, device="cuda")
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
                with pytest.raises(AwryError) as e:
                    ix.align_hits_device(d_qb.data_ptr(), d_qo.data_ptr(), 1, m, 1, d_off.data_ptr(), 0, 0, 0, strands=s)
                assert e.value.code == -6, (name, m, s)
                with pytest.raises(AwryError) as e:
                    ix.align_hits_packed(qb, qo, m, 1, np.zeros(3 if s else 2, np.uint64), np.zeros((0, 2), np.uint64),
                                         strands=s)
                assert e.value.code == -6, (name, m, s)
        if env:
            monkeypatch.delenv(env[0])


# ---- 5. the bounds-checked build -----------------------------------------------------------------------------------

def test_on_the_bounds_checked_build():
    """this file against libawry_b200_checked.so (every data-dependent load bounds-checked, layout.cuh): no assert"""
    checked = os.path.join(ROOT, "awry_b200", "libawry_b200_checked.so")
    if os.environ.get("AWRY_B200_LIB"):
        pytest.skip("already running against another build")
    if not os.path.exists(checked):
        subprocess.check_call(["make", "-s", "-C", os.path.join(ROOT, "awry_b200", "csrc"), "checked"])
    env = dict(os.environ, AWRY_B200_LIB=checked)
    out = subprocess.run([sys.executable, "-m", "pytest", "tests/test_gpu_align.py", "-m", "gpu", "-x", "-q", "-p",
                          "no:cacheprovider", "-k", "not bounds_checked and not replica_1"],
                         cwd=ROOT, env=env, capture_output=True, text=True, timeout=3000)
    tail = out.stdout[-1500:] + out.stderr[-1500:]
    assert out.returncode == 0, tail
    assert " passed" in out.stdout and "Assertion" not in out.stderr, tail
