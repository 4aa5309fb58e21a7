"""Device-resident locate of the approximate searches: awry_locate_device_hamming, _hamming_strands, _edit and
_edit_strands.  Every case compares, bit for bit, the CSR offsets d_hit_off, the hits in text order and each hit's
distance with the brute-force references (tests/hamming_brute.c, tests/edit_brute.c, through the helpers of
test_gpu_approx_fuzz.py) and with the host-buffer call of the same metric (awry_locate_batch_*), which must agree.

- Both metrics, both strand counts, k = 0 .. 3, on the multi-record index of test_gpu_approx_fuzz.py (more than 3000
  reads, every other one reverse-complemented), on a few of its random small indexes and on texts shorter than the
  reads with reads at both ends.
- Routes: AWRY_B200_HAMMING_SLICE=16 (many slices in the count and the place pass), set_locate_variant(1) and (2),
  set_count_variant(1), the index loaded under AWRY_B200_KMER_DEV=0, and the repeat-rich text of test_gpu_hamming.py
  (reads with 200 hits and more) at AWRY_B200_HAMMING_SLICE=300.
- Entry points: a sub-batch from the middle of a device buffer (first offset not a multiple of 64, data pointer + 1 ..
  7 bytes), a torch.cuda.Stream() other than the default, garbage in d_hit_off beforehand, nq = 1, a batch without
  hits (NULL pointers, offsets 0), no distances wanted, 20 calls in a row each freed with device_free, replica 1 of a
  two-GPU handle.
- Refused reads (empty, L <= k, with '$') among good reads: the call succeeds, each read's hit range is the row sum of
  the count_*_device call on the same batch, the good reads' hits are those of the host call on the good reads alone,
  and device_check reports the first refused read once.
- Indexes the searches do not exist for return AWRY_ERR_UNSUPPORTED (-6).
- The whole file once more against libawry_b200_checked.so, which also asserts that every placed key lies inside its
  read's range."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT, device_from_parts
from test_gpu_approx_fuzz import (COMBOS, LENS, awkward_reads, batches, end_reads, expected, fuzz_reads, mid,  # noqa: F401
                                  mid_dev, rand_bases, random_text, refs, select)
from test_gpu_hamming import repeats  # noqa: F401

pytestmark = pytest.mark.gpu


def pack(qs):
    from awry_b200 import fm_index as f
    return f.pack_queries(qs)


def sfx(strands):
    return "_strands" if strands else ""


def to_host(ptr, nbytes, dtype):
    out = np.zeros(max(1, nbytes), np.uint8)
    if nbytes:
        assert C.CDLL("libcudart.so").cudaMemcpy(C.c_void_p(out.ctypes.data), C.c_void_p(ptr), C.c_size_t(nbytes), 2) == 0
    return out[:nbytes].view(dtype)


def device_locate(dev, metric, strands, qb, qo, k, lo=0, hi=None, shift=0, stream=None, replica=0, device=0,
                  distances=True, check=True):
    """locate_*_device on reads lo .. hi of the batch: the caller's bytes behind `shift` garbage bytes, the offsets of
    the whole batch on the device and d_qoff pointing at entry lo, d_hit_off filled with garbage.  -> (hit_off, hits
    uint64[n, 2], distances uint8[n] or None); the device buffers are freed."""
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
        call = getattr(dev, f"locate_{metric}{sfx(strands)}_device")
        hp, dp, n = call(d_qb.data_ptr() + shift, d_qo.data_ptr() + 8 * lo, nq, k, d_off.data_ptr(),
                         distances=distances, stream=st.cuda_stream, replica=replica)
        if check:
            dev.device_check(st.cuda_stream, replica)
        st.synchronize()
        if n == 0:
            assert hp is None and dp is None
        assert (dp is None) == (n == 0 or not distances)
        hits = to_host(hp, n * 16, np.uint64).reshape(-1, 2)
        dist = to_host(dp, n, np.uint8) if distances else None
        dev.device_free(hp, replica)
        dev.device_free(dp, replica)
        off = d_off.cpu().numpy().view(np.uint64)
        assert int(off[-1]) == n
        return off, hits, dist


def host_locate(dev, metric, strands, qb, qo, k):
    return getattr(dev, f"locate_{metric}{sfx(strands)}_packed")(qb, qo, k)


def same(got, want, what):
    goff, ghits, gd = got
    woff, whits, wd = want[-3:]
    bad = np.nonzero(goff != woff)[0]
    assert len(bad) == 0, what + ("hit offsets", bad[:5], goff[bad[:5]], woff[bad[:5]])
    assert np.array_equal(ghits, whits), what + ("hits",)
    if gd is not None:
        assert np.array_equal(gd, wd), what + ("distances",)


def check(dev, parts, qs, k, metric, strands, refs, tag, want=None, **kw):
    """the device locate against the reference and the host-buffer call"""
    want = want if want is not None else expected(refs, metric, strands, parts, qs, k)
    what = (tag, metric, "both strands" if strands else "one strand", "k=%d" % k)
    qb, qo = pack(qs)
    got = device_locate(dev, metric, strands, qb, qo, k, **kw)
    same(got, want, what + ("reference",))
    same(got, host_locate(dev, metric, strands, qb, qo, k), what + ("host call",))
    return got


# ---- 1. every metric, strand count and k ---------------------------------------------------------------------------

@pytest.mark.parametrize("k", [0, 1, 2, 3])
def test_mid_index(k, mid, mid_dev, batches, refs):
    qs, want = batches(max(k, 1))                          # (the read generator needs k >= 1: k = 0 takes k = 1's reads)
    for m, s in COMBOS:
        check(mid_dev, mid, qs, k, m, s, refs, "mid", want[(m, s)] if k else None)


@pytest.mark.parametrize("seed", [0, 5, 11])
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


@pytest.mark.parametrize("n", [1, 5, 17, 63, 64, 65, 129])
def test_short_texts_and_ends(fx, refs, n):
    r = np.random.default_rng(n)
    t = rand_bases(r, n) if n % 3 else random_text(r, n)
    parts = fx.build_parts(t, 0, ratio=8, kmer_len=int(1 + n % 9), seq_starts=np.zeros(1, np.uint64))
    with device_from_parts(parts) as ix:
        for k in (1, 3):
            lens = sorted({k + 1, k + 2, 9, 33, 65, n - 1, n, n + 1, n + k + 1})
            qs = [q for q in end_reads(t, r, [ln for ln in lens if ln > k]) if len(q) > k]
            for m, s in COMBOS:
                check(ix, parts, qs, k, m, s, refs, "n=%d" % n)


# ---- 2. routes -----------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("route", ["slice_16", "locate_variant_1", "locate_variant_2", "count_variant_1"])
def test_route(route, mid, mid_dev, batches, refs, monkeypatch):
    from awry_b200 import fm_index as f
    qs, want = batches(3)
    try:
        if route.startswith("locate_variant"):
            f.set_locate_variant(int(route[-1]))
        elif route == "count_variant_1":
            f.set_count_variant(1)
        else:                                            # (reads of a few symbols have 10^5 candidates)
            monkeypatch.setenv("AWRY_B200_HAMMING_SLICE", "16")
            keep = np.array([len(q) >= 40 for q in qs])
            qs = [q for q in qs if len(q) >= 40]
            want = {c: select(w, keep) for c, w in want.items()}
        for m, s in COMBOS:
            check(mid_dev, mid, qs, 3, m, s, refs, route, want[(m, s)])
    finally:
        f.set_locate_variant(0)
        f.set_count_variant(0)


def test_index_loaded_without_the_device_seed_table(mid, batches, refs, monkeypatch):
    qs, want = batches(2)
    monkeypatch.setenv("AWRY_B200_KMER_DEV", "0")
    with device_from_parts(mid) as ix:
        for m, s in COMBOS:
            check(ix, mid, qs, 2, m, s, refs, "AWRY_B200_KMER_DEV=0", want[(m, s)])


def test_repeat_rich_text(repeats, refs, monkeypatch):  # noqa: F811
    parts, ix, qb, qo = repeats
    qs = [bytes(qb[int(qo[i]):int(qo[i + 1])]) for i in range(len(qo) - 1)]
    monkeypatch.setenv("AWRY_B200_HAMMING_SLICE", "300")
    for m, s in COMBOS:
        want = expected(refs, m, s, parts, qs, 2)
        assert np.diff(want[1].astype(np.int64)).max() >= 200, (m, s)
        check(ix, parts, qs, 2, m, s, refs, "repeats", want)


def test_long_and_awkward_reads(mid, mid_dev, refs):
    qs = awkward_reads(mid, 2, seed=80)
    for m, s in COMBOS:
        check(mid_dev, mid, qs, 2, m, s, refs, "awkward")


# ---- 3. entry points -----------------------------------------------------------------------------------------------

def test_sub_batches_streams_and_nq_1(mid, mid_dev, batches):
    import torch
    qs, want = batches(3)
    qb, qo = pack(qs)
    lo = next(i for i in range(500, 3000) if int(qo[i]) % 64)
    cases = [(lo, lo + 1700), (lo + 3, lo + 4), (len(qs) - 1, len(qs)), (0, 1)]
    stream = torch.cuda.Stream()
    for c, (m, s) in enumerate(COMBOS):
        for i, (a, b) in enumerate(cases):
            keep = np.zeros(len(qs), bool)
            keep[a:b] = True
            w = select(want[(m, s)], keep)
            shift = 1 + (c * len(cases) + i) % 7
            for st in (None, stream):
                got = device_locate(mid_dev, m, s, qb, qo, 3, a, b, shift=shift, stream=st)
                same(got, w, (m, s, a, b, shift, st is not None))


def test_no_hits_no_distances_and_repeated_calls(mid, mid_dev, batches):
    qs, want = batches(2)
    qb, qo = pack(qs)
    r = np.random.default_rng(5)
    nohit = [rand_bases(r, 80) for _ in range(40)]          # 80 random bases do not occur within 3 edits
    nb, no = pack(nohit)
    for m, s in COMBOS:
        off, hits, dist = device_locate(mid_dev, m, s, nb, no, 3)
        assert not off.any() and len(hits) == 0 and len(dist) == 0, (m, s)
        got = device_locate(mid_dev, m, s, qb, qo, 2, distances=False)
        assert got[2] is None
        same(got, want[(m, s)], (m, s, "no distances"))
    first = device_locate(mid_dev, "edit", True, qb, qo, 2)
    for i in range(20):
        same(device_locate(mid_dev, "edit", True, qb, qo, 2), first, ("call", i))


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
        for m, s in COMBOS:
            for st in (None, stream):
                got = device_locate(ix, m, s, qb, qo, 2, 7, len(qs), shift=5, stream=st, replica=1, device=1)
                same(got, select(want[(m, s)], keep), (m, s, st is not None))
    finally:
        ix.close()


# ---- 4. refused reads and unsupported indexes ----------------------------------------------------------------------

def test_refused_reads(mid, mid_dev):
    import torch
    from awry_b200 import AwryError
    t = bytes(mid.text)
    k = 2
    good = [t[1000 + 97 * i:1000 + 97 * i + 60] for i in range(30)]
    dollar = bytearray(t[5000:5060])
    dollar[30] = ord("$")
    qs = list(good)
    qs.insert(3, b"")                                      # empty
    qs.insert(10, b"AC")                                   # L <= k
    qs.insert(20, bytes(dollar))                           # a sentinel (the count call does not give it 0: §1e)
    bad = np.zeros(len(qs), bool)
    bad[[3, 10, 20]] = True
    qb, qo = pack(qs)
    gb, go = pack(good)
    for m, s in COMBOS:
        per = 2 if s else 1
        off, hits, dist = device_locate(mid_dev, m, s, qb, qo, k, check=False)
        with pytest.raises(AwryError) as e:
            mid_dev.device_check()
        assert e.value.code == -5 and "query 3" in str(e.value), (m, s, str(e.value))
        mid_dev.device_check()                             # cleared
        d_qb, d_qo = torch.from_numpy(qb).cuda(), torch.from_numpy(qo.view(np.int64)).cuda()
        d_counts = torch.full((len(qs) * per, k + 1), 9, dtype=torch.int64, device="cuda")
        getattr(mid_dev, f"count_{m}{sfx(s)}_device")(d_qb.data_ptr(), d_qo.data_ptr(), len(qs), k, d_counts.data_ptr())
        with pytest.raises(AwryError):
            mid_dev.device_check()
        sums = d_counts.cpu().numpy().view(np.uint64).sum(axis=1)
        assert np.array_equal(np.diff(off.astype(np.int64)), sums.astype(np.int64)), (m, s)
        lens = np.diff(off.astype(np.int64)).reshape(len(qs), per)
        assert not lens[[3, 10]].any(), (m, s)             # as the header promises for the counts
        # the good reads' hits are those of the host call on the good reads alone
        woff, whits, wd = host_locate(mid_dev, m, s, gb, go, k)
        kv = np.repeat(~bad, per)
        kh = np.repeat(kv, np.diff(off.astype(np.int64)))
        assert np.array_equal(hits[kh], whits) and np.array_equal(dist[kh], wd), (m, s)
        assert np.array_equal(np.diff(off.astype(np.int64))[kv], np.diff(woff.astype(np.int64))), (m, s)


def test_unsupported_indexes(fx, mid, monkeypatch):
    import torch
    from awry_b200 import AwryError
    qb, qo = pack([bytes(mid.text[1000:1100])])
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
                    getattr(ix, f"locate_{m}{sfx(s)}_device")(d_qb.data_ptr(), d_qo.data_ptr(), 1, 1, d_off.data_ptr())
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
    out = subprocess.run([sys.executable, "-m", "pytest", "tests/test_gpu_approx_locate_device.py", "-m", "gpu", "-x",
                          "-q", "-p", "no:cacheprovider", "-k", "not bounds_checked and not replica_1"],
                         cwd=ROOT, env=env, capture_output=True, text=True, timeout=3000)
    tail = out.stdout[-1500:] + out.stderr[-1500:]
    assert out.returncode == 0, tail
    assert " passed" in out.stdout and "Assertion" not in out.stderr, tail
