"""GPU parity of the Hamming search (awry_count_batch_hamming / awry_locate_batch_hamming / awry_count_device_hamming):
windows within k <= 3 substitutions, found by k + 1 exactly searched pieces per read and verified against the text on
the device.  Every result is compared bit for bit with a brute-force scan over every window of the text
(tests/hamming_brute.c, symbols mapped by the oracle's awo_ascii_to_index): counts by distance, hit lists in text
order, and each hit's distance."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from conftest import ROOT, device_from_parts, mixed_queries, oracle_from_parts

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def brute_lib(tmp_path_factory, po):
    so = str(tmp_path_factory.mktemp("hamming") / "libhamming_brute.so")
    subprocess.check_call(["gcc", "-O2", "-fopenmp", "-shared", "-fPIC", "-o", so, os.path.join(ROOT, "tests", "hamming_brute.c")])
    L = C.CDLL(so)
    L.hamming_brute.restype = C.c_int64
    L.hamming_brute.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint32,
                                C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    lut = np.array([po.lib().awo_ascii_to_index(0, c) for c in range(256)], dtype=np.uint8)
    return L, lut


def brute(brute_lib, parts, qb, qo, k):
    """-> (counts uint64[nq, k+1], hit_off uint64[nq+1], hits uint64[n, 2], mismatches uint8[n])"""
    L, lut = brute_lib
    text = np.ascontiguousarray(parts.text, dtype=np.uint8)
    qb = np.ascontiguousarray(qb, dtype=np.uint8)
    qo = np.ascontiguousarray(qo, dtype=np.uint64)
    nq = len(qo) - 1
    counts = np.zeros((nq, k + 1), dtype=np.uint64)
    off = np.zeros(nq + 1, dtype=np.uint64)
    args = (lut.ctypes.data, text.ctypes.data, len(text), qb.ctypes.data, qo.ctypes.data, nq, k, counts.ctypes.data,
            off.ctypes.data)
    n = L.hamming_brute(*args, None, None)
    pos = np.zeros(max(1, n), dtype=np.uint64)
    dist = np.zeros(max(1, n), dtype=np.uint8)
    L.hamming_brute(*args, pos.ctypes.data, dist.ctypes.data)
    starts = np.asarray(parts.seq_starts, dtype=np.uint64) if parts.seq_starts is not None else np.zeros(1, np.uint64)
    seq = np.searchsorted(starts, pos[:n], side="right").astype(np.uint64) - np.uint64(1)
    hits = np.stack([seq, pos[:n] - starts[seq]], axis=1) if n else np.zeros((0, 2), np.uint64)
    return counts, off, hits, dist[:n]


def assert_same(dev, parts, qb, qo, k, brute_lib, want=None):
    counts, off, hits, dist = want if want is not None else brute(brute_lib, parts, qb, qo, k)
    got = dev.count_hamming_packed(qb, qo, k)
    bad = np.nonzero((got != counts).any(axis=1))[0]
    assert len(bad) == 0, (k, bad[:5], got[bad[:5]], counts[bad[:5]])
    goff, ghits, gd = dev.locate_hamming_packed(qb, qo, k)
    assert np.array_equal(goff, off), k
    assert np.array_equal(ghits, hits) and np.array_equal(gd, dist), k
    return counts, off, hits, dist


@pytest.fixture(scope="module")
def multi(fx):
    """several records joined by N, with N runs and isolated N inside them (as in test_gpu_text_finish.py)"""
    r = np.random.default_rng(17)
    recs = []
    for i, n in enumerate([90_000, 1, 150_000, 40, 99_999]):
        t = bytearray(bytes(fx.gen_text(0, n, 50 + i)))
        if n > 1000:
            for _ in range(6):
                t[int(r.integers(0, n))] = ord("N")
            p = int(r.integers(0, n - 300))
            t[p:p + 120] = b"N" * 120
        recs.append(bytes(t))
    text, starts = fx.concat_records(recs, 0)
    return fx.build_parts(text, 0, ratio=8, kmer_len=9, seq_starts=starts)


@pytest.fixture(scope="module")
def multi_dev(multi):
    ix = device_from_parts(multi)
    yield ix
    ix.close()


def substitute(q, at, r):
    c = q[at]
    alt = [b for b in b"ACGT" if b != c]
    q[at] = alt[int(r.integers(0, len(alt)))]


def hamming_queries(parts, k, seed, n_random=1500):
    from awry_b200 import fm_index as f
    r = np.random.default_rng(seed)
    t = bytes(parts.text)
    starts = [int(s) for s in parts.seq_starts]
    qs = []
    # reads with 0 .. k+1 planted substitutions: anywhere, in every piece, at the piece boundaries, first / last symbol
    for i in range(n_random):
        ln = int(r.integers(k + 1, 600)) if i % 3 else int(r.integers(k + 1, 60))
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
        if i % 17 == 5:
            q = bytearray(bytes(q).lower())
        if i % 19 == 7:
            q = bytearray(bytes(q).replace(b"T", b"U"))
        if i % 23 == 11:
            q[int(r.integers(0, ln))] = ord("NRnyk"[int(r.integers(0, 5))])
        qs.append(bytes(q))
    for ln in list(range(k + 1, 40)) + [64, 65, 127, 128, 129, 255, 256, 257, 600]:
        qs.append(t[:ln])                                # the very start of the text
        qs.append(t[len(t) - ln:])                       # the very end
        head = bytearray(t[:ln])
        substitute(head, ln - 1, r)
        qs.append(bytes(head))
    for s in starts[1:]:                                 # across record delimiters
        for back in (1, 5, 40):
            a = max(0, s - back)
            q = bytearray(t[a:a + 80])
            qs.append(bytes(q))
            substitute(q, min(len(q) - 1, back + 3), r)
            qs.append(bytes(q))
    for _ in range(40):                                  # random reads: mostly nothing within k
        qs.append(bytes(r.choice(np.frombuffer(b"ACGT", np.uint8), int(r.integers(k + 1, 150)))))
    p = int(r.integers(0, len(t) - 2000))
    q = bytearray(t[p:p + 1999])
    for a in r.choice(1999, size=k, replace=False):
        substitute(q, int(a), r)
    qs.append(bytes(q))                                  # about 2000 bp
    return f.pack_queries(qs)


@pytest.mark.parametrize("k", [1, 2, 3])
def test_hamming_equals_brute_force(k, multi, multi_dev, brute_lib):
    qb, qo = hamming_queries(multi, k, seed=100 + k)
    counts, off, hits, dist = assert_same(multi_dev, multi, qb, qo, k, brute_lib)
    # the planted reads reach every distance, and reads with k+1 substitutions are mostly gone
    assert all((counts[:, d] > 0).sum() > 50 for d in range(k + 1))
    assert len(hits) > 1000 and (np.diff(off.astype(np.int64)) == 0).sum() > 100


@pytest.mark.parametrize("k", [1, 2])
def test_every_substitution_of_a_read(k, multi, multi_dev, brute_lib):
    """a 120-bp read with a substitution at every position (and every pair of positions at k = 2): every alignment of
    the substitutions against the pieces and the text words"""
    from awry_b200 import fm_index as f
    r = np.random.default_rng(5)
    t = bytes(multi.text)
    p = 1000
    read = bytearray(t[p:p + 120])
    qs = [bytes(read)]
    for a in range(120):
        q = bytearray(read)
        substitute(q, a, r)
        qs.append(bytes(q))
    if k >= 2:
        for a in range(120):
            for b in range(a + 1, 120):
                q = bytearray(read)
                substitute(q, a, r)
                substitute(q, b, r)
                qs.append(bytes(q))
    qb, qo = f.pack_queries(qs)
    counts, _, _, _ = assert_same(multi_dev, multi, qb, qo, k, brute_lib)
    assert (counts[1:121, 1] >= 1).all()


def test_k0_equals_exact_search(fx, dna_small, brute_lib):
    parts, ix = dna_small
    qb, qo = mixed_queries(fx, parts.text, 4000, 24, seed=2)
    counts = ix.count_hamming_packed(qb, qo, 0)
    assert np.array_equal(counts[:, 0], ix.count_packed(qb, qo))
    off, hits = ix.locate_packed(qb, qo, sorted_hits=True)
    hoff, hhits, hd = ix.locate_hamming_packed(qb, qo, 0)
    assert np.array_equal(hoff, off) and np.array_equal(hhits, hits) and not hd.any()
    assert_same(ix, parts, qb, qo, 0, brute_lib)


@pytest.fixture(scope="module")
def dna_small(fx):
    text = fx.gen_text(0, 200_000, 31)
    parts = fx.build_parts(text, 0, ratio=8, kmer_len=8)
    ix = device_from_parts(parts)
    yield parts, ix
    ix.close()


@pytest.fixture(scope="module")
def repeats(fx):
    from fixtures.repeats import repeat_queries, repeat_rich_text
    text, regions = repeat_rich_text(300_000, seed=4, tandem_arrays=30)
    parts = fx.build_parts(text, 0, ratio=8, kmer_len=8)
    qb, qo = repeat_queries(text, regions, 600, 60, seed=6)
    ix = device_from_parts(parts)
    yield parts, ix, qb, qo
    ix.close()


def test_repeat_rich_text_and_tiny_slices(repeats, brute_lib, monkeypatch):
    """tandem arrays give reads hundreds of windows; every hit list is free of duplicates and equals brute force, also
    when the candidates are verified a few hundred at a time"""
    parts, ix, qb, qo = repeats
    want = brute(brute_lib, parts, qb, qo, 2)
    off = want[1]
    assert np.diff(off.astype(np.int64)).max() >= 200
    _, goff, ghits, _ = assert_same(ix, parts, qb, qo, 2, brute_lib, want)
    for i in range(len(goff) - 1):
        seg = ghits[int(goff[i]):int(goff[i + 1])]
        assert len(np.unique(seg, axis=0)) == len(seg)
    monkeypatch.setenv("AWRY_B200_HAMMING_SLICE", "300")
    assert_same(ix, parts, qb, qo, 2, brute_lib, want)


def test_results_do_not_depend_on_the_knobs(multi, multi_dev, brute_lib, monkeypatch):
    from awry_b200 import fm_index as f
    qb, qo = hamming_queries(multi, 2, seed=9, n_random=600)
    want = brute(brute_lib, multi, qb, qo, 2)
    try:
        for lv in (0, 1, 2):
            f.set_locate_variant(lv)
            assert_same(multi_dev, multi, qb, qo, 2, brute_lib, want)
        f.set_locate_variant(0)
        f.set_count_variant(1)
        assert_same(multi_dev, multi, qb, qo, 2, brute_lib, want)
    finally:
        f.set_locate_variant(0)
        f.set_count_variant(0)
    monkeypatch.setenv("AWRY_B200_LOCATE_CHUNK_Q", "1024")
    assert_same(multi_dev, multi, qb, qo, 2, brute_lib, want)


def test_errors(fx, multi, multi_dev, monkeypatch):
    from awry_b200 import AwryError
    from awry_b200 import fm_index as f
    t = bytes(multi.text)
    for k, bad in ((1, b"A"), (2, b"AC"), (3, b"ACG"), (2, b""), (1, b"AC$GT")):
        qb, qo = f.pack_queries([t[100:150], bad, t[200:260]])
        for call in (multi_dev.count_hamming_packed, multi_dev.locate_hamming_packed):
            with pytest.raises(AwryError) as e:
                call(qb, qo, k)
            assert e.value.code == -5 and "query 1" in str(e.value), (k, bad)
    qb, qo = f.pack_queries([t[100:150]])
    with pytest.raises(AwryError) as e:
        multi_dev.count_hamming_packed(qb, qo, 4)
    assert e.value.code == -1
    # too small a buffer: the offsets are complete, and the retry gives the same hits
    qb, qo = hamming_queries(multi, 1, seed=3, n_random=300)
    hoff, hits, dist = multi_dev.locate_hamming_packed(qb, qo, 1, capacity=len(qo) * 100)
    off = np.zeros(len(qo), np.uint64)
    small = np.zeros((5, 2), np.uint64)
    mm = np.zeros(5, np.uint8)
    n = C.c_uint64()
    rc = f.native().awry_locate_batch_hamming(multi_dev.handle, qb.ctypes.data, qo.ctypes.data, len(qo) - 1, 1,
                                              off.ctypes.data, small.ctypes.data, mm.ctypes.data, 5, C.byref(n))
    assert rc == -8 and n.value == len(hits) and np.array_equal(off, hoff)
    assert np.array_equal(small, hits[:5]) and np.array_equal(mm, dist[:5])
    assert np.array_equal(multi_dev.locate_hamming_packed(qb, qo, 1, capacity=3)[1], hits)
    # indexes the search does not exist for
    text = fx.gen_text(1, 20_000, 3)
    prot = fx.build_parts(text, 1, ratio=8, kmer_len=3)
    with device_from_parts(prot) as ix:
        with pytest.raises(AwryError) as e:
            ix.count_hamming_packed(*f.pack_queries([b"ACDEFG"]), 1)
        assert e.value.code == -6
    dna = fx.gen_text(0, 30_000, 3)
    parts = fx.build_parts(dna, 0, ratio=8, kmer_len=8)
    for var in ("AWRY_B200_TEXT", "AWRY_B200_FULL_SA", "AWRY_B200_WIDE"):
        monkeypatch.setenv(var, "1" if var == "AWRY_B200_WIDE" else "0")
        with device_from_parts(parts) as ix:
            for call in (ix.count_hamming_packed, ix.locate_hamming_packed):
                with pytest.raises(AwryError) as e:
                    call(*f.pack_queries([bytes(dna[:40])]), 1)
                assert e.value.code == -6, var
        monkeypatch.delenv(var)


def test_device_entry_point(multi, multi_dev, brute_lib):
    import torch
    from awry_b200 import AwryError
    from awry_b200 import fm_index as f
    qb, qo = hamming_queries(multi, 3, seed=12, n_random=800)
    want = multi_dev.count_hamming_packed(qb, qo, 3)
    d_qb = torch.from_numpy(qb).cuda()
    d_qo = torch.from_numpy(qo.view(np.int64)).cuda()
    d_counts = torch.full((len(qo) - 1, 4), 7, dtype=torch.int64, device="cuda")
    multi_dev.count_hamming_device(d_qb.data_ptr(), d_qo.data_ptr(), len(qo) - 1, 3, d_counts.data_ptr())
    multi_dev.device_check()
    assert np.array_equal(d_counts.cpu().numpy().view(np.uint64), want)
    qb2, qo2 = f.pack_queries([bytes(multi.text[500:600]), b"ACG", bytes(multi.text[900:960])])
    d_qb, d_qo = torch.from_numpy(qb2).cuda(), torch.from_numpy(qo2.view(np.int64)).cuda()
    d_counts = torch.zeros((3, 4), dtype=torch.int64, device="cuda")
    multi_dev.count_hamming_device(d_qb.data_ptr(), d_qo.data_ptr(), 3, 3, d_counts.data_ptr())
    with pytest.raises(AwryError) as e:
        multi_dev.device_check()
    assert e.value.code == -5 and "query 1" in str(e.value)
    got = d_counts.cpu().numpy()
    assert got[0, 0] >= 1 and got[2, 0] >= 1 and not got[1].any()
    multi_dev.device_check()


def test_several_replicas_equal_one(multi, brute_lib):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    qb, qo = hamming_queries(multi, 2, seed=21, n_random=800)
    ix = device_from_parts(multi, devices=[0, 1])
    try:
        assert_same(ix, multi, qb, qo, 2, brute_lib)
    finally:
        ix.close()


def test_on_the_bounds_checked_build():
    """this file against libawry_b200_checked.so (every data-dependent load bounds-checked, layout.cuh): no assert"""
    import sys
    checked = os.path.join(ROOT, "awry_b200", "libawry_b200_checked.so")
    if os.environ.get("AWRY_B200_LIB"):
        pytest.skip("already running against another build")
    if not os.path.exists(checked):
        subprocess.check_call(["make", "-s", "-C", os.path.join(ROOT, "awry_b200", "csrc"), "checked"])
    env = dict(os.environ, AWRY_B200_LIB=checked)
    out = subprocess.run([sys.executable, "-m", "pytest", "tests/test_gpu_hamming.py", "-m", "gpu", "-x", "-q",
                          "-p", "no:cacheprovider", "-k", "not bounds_checked and not several_replicas"],
                         cwd=ROOT, env=env, capture_output=True, text=True, timeout=1200)
    tail = out.stdout[-1500:] + out.stderr[-1500:]
    assert out.returncode == 0, tail
    assert " passed" in out.stdout and "Assertion" not in out.stderr, tail
