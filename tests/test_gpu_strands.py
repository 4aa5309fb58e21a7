"""Both strands (awry_*_strands): query q stands for the virtual queries 2q (q) and 2q + 1 (its reverse complement).
Strand 0 must equal the single-strand calls on q and strand 1 the single-strand calls on rc(q), computed here from the
header's rule (bytes mapped as exact search maps them, complemented, reversed), and both must equal the oracle: counts,
CSR offsets and per-strand hit lists in BWT order and sorted.  Every route is compared: device-resident with the strand
wave kernel on and off, host buffers with host packing on and off, AWRY_B200_ASCII_WAVE=0, count variant 1, the three
locate pass-2 schemes, caller-pinned buffers, a wide index, an index without the text, several replicas.  Reads of
every length 1-300 at every start alignment mod 32, with lowercase / U / N / IUPAC bytes at the ends and at sector
edges, repeat-rich reads the wave kernel hands on, reads over 256 symbols and palindromic reads; refused batches name
the same query as the single-strand calls; a too-small hit buffer still returns complete offsets."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT, device_from_parts, oracle_from_parts

pytestmark = pytest.mark.gpu

_COMP = {ord("A"): ord("T"), ord("C"): ord("G"), ord("G"): ord("C"), ord("T"): ord("A")}


def rc(q: bytes) -> bytes:
    """the reverse complement as include/awry_b200.h defines it (over ACGTN)"""
    out = bytearray()
    for b in reversed(q):
        u = b - 32 if 97 <= b <= 122 else b
        if u == ord("U"):
            u = ord("T")
        out.append(_COMP.get(u, ord("N")))
    return bytes(out)


@pytest.fixture(scope="module")
def rep(fx):
    from fixtures.repeats import repeat_rich_text
    text, regions = repeat_rich_text(300_000, seed=37)
    recs = [bytes(text[:150_000]), bytes(text[150_000:])]
    joined, starts = fx.concat_records(recs, 0)
    return fx.build_parts(joined, 0, ratio=8, kmer_len=9, seq_starts=starts), regions


@pytest.fixture(scope="module")
def rep_dev(rep):
    ix = device_from_parts(rep[0])
    yield ix
    ix.close()


@pytest.fixture(autouse=True)
def defaults():
    from awry_b200 import fm_index as f
    yield
    for k in ("AWRY_B200_ASCII_WAVE", "AWRY_B200_STRAND_WAVE"):
        os.environ.pop(k, None)
    f.set_host_pack(-1)
    f.set_locate_variant(0)
    f.set_count_variant(0)


def sweep_reads(parts, regions, seed):
    """every length 1 .. 300 (either strand of the text), 10 % substitutions, lowercase; special bytes at the first /
    last byte and at offsets 31, 32, 63, 64; repeat-rich reads (handed on by the wave kernel)"""
    r = np.random.default_rng(seed)
    t = bytes(parts.text)
    n = len(t)
    qs = []
    for ln in range(1, 301):
        p = int(r.integers(0, n - ln))
        q = t[p:p + ln]
        if r.random() < 0.5:
            q = rc(q)
        qs.append(q)
        m = bytearray(q)
        for i in np.flatnonzero(r.random(ln) < 0.10):
            m[i] = ord("ACGT"[(b"ACGTN".find(bytes([m[i]])) + 1) % 4])
        qs.append(bytes(m))
        qs.append(q.lower())
        for at in {0, ln - 1, 31, 32, 63, 64}:
            if at < ln:
                s = bytearray(q)
                s[at] = ord("NnRYKuUa"[(ln + at) % 8])
                qs.append(bytes(s))
    for a, b in regions[:60]:
        for ln in (40, 150, 250, 290):
            if b - a > ln:
                p = a + int(r.integers(0, b - a - ln))
                qs.append(rc(t[p:p + ln]) if ln % 3 else t[p:p + ln])
    return [qs[i] for i in r.permutation(len(qs))]


def expected(ix_or_orc, reads, oracle=True, sorted_hits=False):
    """(counts (nq, 2), virtual CSR offsets, hits) from single-strand searches of the reads and their complements"""
    from awry_b200 import fm_index as f
    qb, qo = f.pack_queries(reads)
    rb, ro = f.pack_queries([rc(q) for q in reads])
    if oracle:
        cf, _ = ix_or_orc.count_batch(qb, qo)
        cr, _ = ix_or_orc.count_batch(rb, ro)
        of, hf, _ = ix_or_orc.locate_batch(qb, qo)
        orr, hr, _ = ix_or_orc.locate_batch(rb, ro)
    else:
        cf, cr = ix_or_orc.count_packed(qb, qo), ix_or_orc.count_packed(rb, ro)
        of, hf = ix_or_orc.locate_packed(qb, qo, sorted_hits=sorted_hits)
        orr, hr = ix_or_orc.locate_packed(rb, ro, sorted_hits=sorted_hits)
    voff, vhits = [0], []
    for i in range(len(reads)):
        for off, hits in ((of, hf), (orr, hr)):
            seg = hits[int(off[i]):int(off[i + 1])]
            vhits.append(seg)
            voff.append(voff[-1] + len(seg))
    vh = np.concatenate(vhits) if vhits else np.zeros((0, 2), np.uint64)
    return np.stack([cf, cr], axis=1).astype(np.uint64), np.array(voff, np.uint64), vh.reshape(-1, 2).astype(np.uint64)


def device_copy(qb, pad):
    import torch
    d = torch.zeros(pad + len(qb), dtype=torch.uint8, device="cuda")
    d[pad:] = torch.from_numpy(qb).cuda()
    return d


def fetch_hits(ix, ptr, n):
    import torch
    buf = torch.empty((max(1, n), 2), dtype=torch.int64, device="cuda")
    if n:
        assert C.CDLL("libcudart.so").cudaMemcpy(C.c_void_p(buf.data_ptr()), C.c_void_p(ptr), C.c_size_t(n * 16), 3) == 0
    ix.device_free(ptr)
    return buf[:n].cpu().numpy().view(np.uint64)


def both_waves(fn):
    """fn() on the generic route (AWRY_B200_STRAND_WAVE=0), then with the strand wave kernel"""
    os.environ["AWRY_B200_STRAND_WAVE"] = "0"
    try:
        old = fn()
    finally:
        os.environ.pop("AWRY_B200_STRAND_WAVE", None)
    return old, fn()


def host_results(ix, reads, sorted_hits=False):
    from awry_b200 import fm_index as f
    qb, qo = f.pack_queries(reads)
    c = ix.count_strands_packed(qb, qo)
    off, hits = ix.locate_strands_packed(qb, qo, sorted_hits=sorted_hits)
    return c, off, hits


def assert_same(got, want, what=""):
    for g, w in zip(got, want):
        assert np.array_equal(np.asarray(g), np.asarray(w)), what


def test_device_calls_every_length_and_alignment(rep, rep_dev, po):
    import torch
    from awry_b200 import fm_index as f
    reads = sweep_reads(rep[0], rep[1], seed=2)
    qb, qo = f.pack_queries(reads)
    nq = len(qo) - 1
    wc, woff, whits = expected(oracle_from_parts(po, rep[0]), reads)
    assert (wc[:, 1] > 0).sum() > 300 and (wc[:, 0] > 0).sum() > 300 and (wc > 8).sum() > 50
    c0 = rep_dev.count_packed(qb, qo)
    assert np.array_equal(c0, wc[:, 0])
    d_qo = torch.from_numpy(qo.view(np.int64)).cuda()
    st = torch.cuda.current_stream().cuda_stream
    for pad in range(32):
        d_qb = device_copy(qb, pad)
        ptr = d_qb.data_ptr() + pad

        def count():
            d_c = torch.full((2 * nq,), 7, dtype=torch.int64, device="cuda")
            rep_dev.count_strands_device(ptr, d_qo.data_ptr(), nq, d_c.data_ptr(), st)
            rep_dev.device_check(st)
            return d_c.cpu().numpy().view(np.uint64).reshape(nq, 2)

        old, new = both_waves(count)
        assert np.array_equal(old, wc) and np.array_equal(new, wc), pad
        if pad % 8 == 0:
            def locate():
                d_off = torch.zeros(2 * nq + 1, dtype=torch.int64, device="cuda")
                p, n = rep_dev.locate_strands_device(ptr, d_qo.data_ptr(), nq, d_off.data_ptr(), stream=st)
                return d_off.cpu().numpy().view(np.uint64), fetch_hits(rep_dev, p, n)

            (ooff, ohits), (noff, nhits) = both_waves(locate)
            assert np.array_equal(ooff, woff) and np.array_equal(noff, woff), pad
            assert np.array_equal(ohits, whits) and np.array_equal(nhits, whits), pad


@pytest.mark.parametrize("route", ["default", "no_host_pack", "host_pack", "no_ascii_wave", "no_strand_wave",
                                   "count_variant_1"])
@pytest.mark.parametrize("locate_variant", [0, 1, 2])
def test_host_calls_every_route(rep, rep_dev, po, route, locate_variant):
    from awry_b200 import fm_index as f
    reads = sweep_reads(rep[0], rep[1], seed=3)
    want = expected(oracle_from_parts(po, rep[0]), reads)
    f.set_locate_variant(locate_variant)
    if route == "no_host_pack":
        f.set_host_pack(0)
    elif route == "host_pack":
        f.set_host_pack(1)
    elif route == "no_ascii_wave":
        os.environ["AWRY_B200_ASCII_WAVE"] = "0"
    elif route == "no_strand_wave":
        os.environ["AWRY_B200_STRAND_WAVE"] = "0"
    elif route == "count_variant_1":
        f.set_count_variant(1)
    assert_same(host_results(rep_dev, reads), want, route)
    # sorted within each strand: what the single-strand calls return sorted
    ws = expected(rep_dev, reads, oracle=False, sorted_hits=True)
    assert_same(host_results(rep_dev, reads, sorted_hits=True), ws, route)


def test_pinned_buffers_and_capacity(rep, rep_dev, po):
    """caller-pinned buffers take the sync-free locate pipeline; a buffer one hit too small reports AWRY_ERR_CAPACITY
    with complete offsets and the needed total"""
    import torch
    from awry_b200 import fm_index as f
    reads = sweep_reads(rep[0], rep[1], seed=4)
    _, woff, whits = expected(oracle_from_parts(po, rep[0]), reads)
    qb, qo = f.pack_queries(reads)
    nq = len(qo) - 1
    p_qb = torch.from_numpy(qb).pin_memory()
    p_qo = torch.from_numpy(qo.view(np.int64)).pin_memory()
    for hp in (0, 1):
        f.set_host_pack(hp)
        p_off = torch.zeros(2 * nq + 1, dtype=torch.int64).pin_memory()
        p_hits = torch.zeros((len(whits) + 1, 2), dtype=torch.int64).pin_memory()
        n = C.c_uint64()
        rc_ = f.native().awry_locate_batch_strands(rep_dev.handle, p_qb.data_ptr(), p_qo.data_ptr(), nq, 0,
                                                   p_off.data_ptr(), p_hits.data_ptr(), len(whits) + 1, C.byref(n))
        assert rc_ == 0 and n.value == len(whits)
        assert np.array_equal(p_off.numpy().view(np.uint64), woff)
        assert np.array_equal(p_hits.numpy()[:n.value].view(np.uint64), whits)
    off = np.zeros(2 * nq + 1, np.uint64)
    hits = np.zeros((len(whits) - 1, 2), np.uint64)
    n = C.c_uint64()
    rc_ = f.native().awry_locate_batch_strands(rep_dev.handle, qb.ctypes.data, qo.ctypes.data, nq, 0, off.ctypes.data,
                                               hits.ctypes.data, len(hits), C.byref(n))
    assert rc_ == -8 and n.value == len(whits)
    assert np.array_equal(off, woff)


def test_palindromes_report_the_same_windows_on_both_strands(fx, po):
    from awry_b200 import fm_index as f
    r = np.random.default_rng(5)
    base = bytearray(fx.gen_text(0, 200_000, 55).tobytes())
    pals = []
    for i in range(300):
        s = bytes(r.choice(list(b"ACGT"), size=int(r.integers(1, 80))).astype(np.uint8))
        p = s + rc(s)
        assert rc(p) == p
        pals.append(p)
        for _ in range(1 + i % 3):  # planted 1-3 times
            at = int(r.integers(0, len(base) - len(p)))
            base[at:at + len(p)] = p
    parts = fx.build_parts(bytes(base), 0, ratio=8, kmer_len=9)
    ix = device_from_parts(parts)
    try:
        qb, qo = f.pack_queries(pals)
        c = ix.count_strands_packed(qb, qo)
        assert np.array_equal(c[:, 0], c[:, 1]) and (c[:, 0] > 0).mean() > 0.9  # (later plants may cover earlier ones)
        for sorted_hits in (False, True):
            off, hits = ix.locate_strands_packed(qb, qo, sorted_hits=sorted_hits)
            for q in range(len(pals)):
                fwd = hits[int(off[2 * q]):int(off[2 * q + 1])]
                rev = hits[int(off[2 * q + 1]):int(off[2 * q + 2])]
                assert np.array_equal(fwd, rev), q
        assert_same(host_results(ix, pals), expected(oracle_from_parts(po, parts), pals))
    finally:
        ix.close()


@pytest.mark.parametrize("env", ["AWRY_B200_WIDE", "AWRY_B200_TEXT"])
def test_wide_index_and_index_without_text(rep, po, monkeypatch, env):
    import torch
    from awry_b200 import fm_index as f
    monkeypatch.setenv(env, "1" if env == "AWRY_B200_WIDE" else "0")
    reads = sweep_reads(rep[0], rep[1], seed=6)
    want = expected(oracle_from_parts(po, rep[0]), reads)
    ix = device_from_parts(rep[0])
    try:
        if env == "AWRY_B200_WIDE":
            assert ix.row_pointer_bits() == 64
        assert_same(host_results(ix, reads), want, env)
        qb, qo = f.pack_queries(reads)
        nq = len(qo) - 1
        d_qb, d_qo = device_copy(qb, 5), torch.from_numpy(qo.view(np.int64)).cuda()
        st = torch.cuda.current_stream().cuda_stream
        d_c = torch.zeros(2 * nq, dtype=torch.int64, device="cuda")
        ix.count_strands_device(d_qb.data_ptr() + 5, d_qo.data_ptr(), nq, d_c.data_ptr(), st)
        ix.device_check(st)
        assert np.array_equal(d_c.cpu().numpy().view(np.uint64).reshape(nq, 2), want[0])
        d_off = torch.zeros(2 * nq + 1, dtype=torch.int64, device="cuda")
        p, n = ix.locate_strands_device(d_qb.data_ptr() + 5, d_qo.data_ptr(), nq, d_off.data_ptr(), stream=st)
        assert np.array_equal(d_off.cpu().numpy().view(np.uint64), want[1])
        assert np.array_equal(fetch_hits(ix, p, n), want[2])
    finally:
        ix.close()


def test_several_replicas(rep, po):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    reads = sweep_reads(rep[0], rep[1], seed=7)
    want = expected(oracle_from_parts(po, rep[0]), reads)
    ix = device_from_parts(rep[0], devices=[0, 1])
    try:
        assert_same(host_results(ix, reads), want)
        assert_same(host_results(ix, reads, sorted_hits=True), expected(ix, reads, oracle=False, sorted_hits=True))
    finally:
        ix.close()


def test_refused_batches_name_the_same_query(rep, rep_dev):
    import torch
    from awry_b200 import AwryError
    from awry_b200 import fm_index as f
    t = bytes(rep[0].text)
    reads = [t[1000 + 37 * i:1000 + 37 * i + 20 + i % 200] for i in range(3000)]
    qb0, qo0 = f.pack_queries(reads)
    want = rep_dev.count_strands_packed(qb0, qo0)
    st = torch.cuda.current_stream().cuda_stream

    def err(call):
        with pytest.raises(AwryError) as e:
            call()
        return e.value.code, str(e.value)

    for bad_at, bad in ((0, b"AC$GT"), (1777, b"#"), (2999, b"ACGT" * 70 + b"$"), (5, b""), (2400, b"")):
        qs = list(reads)
        qs[bad_at] = bad
        qs[2500] = b""
        qb, qo = f.pack_queries(qs)
        single = err(lambda: rep_dev.count_packed(qb, qo))
        assert single[0] == -5
        for hp in (0, 1):
            f.set_host_pack(hp)
            old, new = both_waves(lambda: err(lambda: rep_dev.count_strands_packed(qb, qo)))
            assert old == new == single, (old, new, single)
            old, new = both_waves(lambda: err(lambda: rep_dev.locate_strands_packed(qb, qo)))
            assert old[0] == new[0] == -5 and "query %d" % min(bad_at, 2500) in new[1], (old, new)
        f.set_host_pack(-1)
        d_qb, d_qo = device_copy(qb, 3), torch.from_numpy(qo.view(np.int64)).cuda()

        def device():
            d_c = torch.zeros(2 * len(qs), dtype=torch.int64, device="cuda")
            rep_dev.count_strands_device(d_qb.data_ptr() + 3, d_qo.data_ptr(), len(qs), d_c.data_ptr(), st)
            e = err(lambda: rep_dev.device_check(st))
            return e, d_c.cpu().numpy()

        (eo, co), (en, cn) = both_waves(device)
        d_c1 = torch.zeros(len(qs), dtype=torch.int64, device="cuda")
        rep_dev.count_device(d_qb.data_ptr() + 3, d_qo.data_ptr(), len(qs), d_c1.data_ptr(), st)
        e1 = err(lambda: rep_dev.device_check(st))
        assert eo == en == e1, (eo, en, e1)
        assert co[5000] == co[5001] == cn[5000] == cn[5001] == 0
    for bad_at, val in ((1, 10**6), (1500, 0), (2999, 10**12)):
        o = qo0.copy()
        o[bad_at] = val
        single = err(lambda: rep_dev.count_packed(qb0, o))
        assert err(lambda: rep_dev.count_strands_packed(qb0, o)) == single
        d_qb, d_qo = device_copy(qb0, 0), torch.from_numpy(o.view(np.int64)).cuda()

        def device():
            d_c = torch.full((2 * len(reads),), 9, dtype=torch.int64, device="cuda")
            rep_dev.count_strands_device(d_qb.data_ptr(), d_qo.data_ptr(), len(reads), d_c.data_ptr(), st)
            return err(lambda: rep_dev.device_check(st)), d_c.cpu().numpy()

        (eo, co), (en, cn) = both_waves(device)
        d_c1 = torch.zeros(len(reads), dtype=torch.int64, device="cuda")
        rep_dev.count_device(d_qb.data_ptr(), d_qo.data_ptr(), len(reads), d_c1.data_ptr(), st)
        e1 = err(lambda: rep_dev.device_check(st))
        assert eo == en == e1 and eo[0] == -1, (eo, en, e1)
        assert co[2 * (bad_at - 1)] == co[2 * bad_at - 1] == 0 and cn[2 * (bad_at - 1)] == cn[2 * bad_at - 1] == 0
    torch.cuda.synchronize()
    assert np.array_equal(rep_dev.count_strands_packed(qb0, qo0), want)  # no sticky error


def test_protein_index_is_unsupported(fx):
    import torch
    from awry_b200 import AwryError
    from awry_b200 import fm_index as f
    parts = fx.build_parts(fx.gen_text(1, 20_000, 9), 1, ratio=8, kmer_len=3)
    ix = device_from_parts(parts)
    try:
        qb, qo = f.pack_queries([b"ACDEF", b"KLMN"])
        for call in (lambda: ix.count_strands_packed(qb, qo), lambda: ix.locate_strands_packed(qb, qo)):
            with pytest.raises(AwryError) as e:
                call()
            assert e.value.code == -6
        d = torch.zeros(16, dtype=torch.int64, device="cuda")
        with pytest.raises(AwryError) as e:
            ix.count_strands_device(d.data_ptr(), d.data_ptr(), 1, d.data_ptr())
        assert e.value.code == -6
        with pytest.raises(AwryError) as e:
            ix.locate_strands_device(d.data_ptr(), d.data_ptr(), 1, d.data_ptr())
        assert e.value.code == -6
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
    out = subprocess.run([sys.executable, "-m", "pytest", "tests/test_gpu_strands.py", "-m", "gpu", "-x", "-q",
                          "-p", "no:cacheprovider", "-k", "not bounds_checked and not route"],
                         cwd=ROOT, env=env, capture_output=True, text=True, timeout=1800)
    tail = out.stdout[-1500:] + out.stderr[-1500:]
    assert out.returncode == 0, tail
    assert " passed" in out.stdout and "Assertion" not in out.stderr, tail
