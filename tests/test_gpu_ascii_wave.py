"""The nucleotide wave kernel packing ASCII reads itself (launch_search_ascii): count_device, locate_device and the
host calls with host packing off must give what the separate packing pass gives (AWRY_B200_ASCII_WAVE=0, the same
process) and what the oracle gives -- counts, CSR offsets and BWT-order hit lists -- for every read length from 1 to
300 (across the 256 symbols the wave kernel stages) at every start alignment mod 32, for lowercase, N, IUPAC and U
bytes at the first and last byte and at 32-byte sector edges, for repeat-rich reads the kernel hands on, for reads
with 10 % substitutions, and for refused batches ($ / #, empty queries, non-monotone offsets): the same error and the
same first bad query, with the device usable afterwards."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT, device_from_parts, oracle_from_parts

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def rep(fx):
    from fixtures.repeats import repeat_rich_text
    text, regions = repeat_rich_text(300_000, seed=31)
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
    os.environ.pop("AWRY_B200_ASCII_WAVE", None)
    f.set_host_pack(-1)
    f.set_locate_variant(0)


def sweep_queries(parts, regions, seed):
    """every length 1 .. 300, exact and with 10 % substitutions, lowercase; special bytes at the first / last byte and
    at offsets 31, 32, 63, 64; reads from repeat-rich regions (still wide after the wave's steps: handed on)"""
    from awry_b200 import fm_index as f
    r = np.random.default_rng(seed)
    t = bytes(parts.text)
    n = len(t)
    qs = []
    for ln in range(1, 301):
        p = int(r.integers(0, n - ln))
        q = t[p:p + ln]
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
                qs.append(t[p:p + ln])
    order = r.permutation(len(qs))
    return f.pack_queries([qs[i] for i in order])


def device_copy(qb, pad):
    """the bytes at offset `pad` of a device buffer that ends with them (the last query byte is the buffer's last)"""
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


def both_paths(fn):
    """fn() with the separate packing pass, then with the wave kernel packing"""
    os.environ["AWRY_B200_ASCII_WAVE"] = "0"
    try:
        old = fn()
    finally:
        os.environ.pop("AWRY_B200_ASCII_WAVE", None)
    return old, fn()


def test_the_switch_drops_the_packing_pass(rep, rep_dev):
    import torch
    from awry_b200 import fm_index as f
    qb, qo = sweep_queries(rep[0], rep[1], seed=1)
    nq = len(qo) - 1
    d_qb, d_qo = device_copy(qb, 0), torch.from_numpy(qo.view(np.int64)).cuda()
    d_c = torch.zeros(nq, dtype=torch.int64, device="cuda")

    def packs():
        f.profile_enable(True)
        f.profile_reset()
        rep_dev.count_device(d_qb.data_ptr(), d_qo.data_ptr(), nq, d_c.data_ptr())
        torch.cuda.synchronize()
        p = f.profile_get()
        f.profile_enable(False)
        return p["pack_launches"]

    old, new = both_paths(packs)
    assert old >= 1 and new == 0


def test_device_calls_every_length_and_alignment(rep, rep_dev, po):
    import torch
    qb, qo = sweep_queries(rep[0], rep[1], seed=2)
    nq = len(qo) - 1
    orc = oracle_from_parts(po, rep[0])
    want, _ = orc.count_batch(qb, qo)
    woff, whits, _ = orc.locate_batch(qb, qo)
    assert (want == 0).sum() > 500 and (want == 1).sum() > 300 and (want > 8).sum() > 50
    d_qo = torch.from_numpy(qo.view(np.int64)).cuda()
    st = torch.cuda.current_stream().cuda_stream
    for pad in range(32):
        d_qb = device_copy(qb, pad)
        ptr = d_qb.data_ptr() + pad

        def count():
            d_c = torch.full((nq,), 7, dtype=torch.int64, device="cuda")
            rep_dev.count_device(ptr, d_qo.data_ptr(), nq, d_c.data_ptr(), st)
            rep_dev.device_check(st)
            return d_c.cpu().numpy().view(np.uint64)

        old, new = both_paths(count)
        assert np.array_equal(old, want) and np.array_equal(new, want), pad
        if pad % 8 == 0:
            def locate():
                d_off = torch.zeros(nq + 1, dtype=torch.int64, device="cuda")
                p, n = rep_dev.locate_device(ptr, d_qo.data_ptr(), nq, d_off.data_ptr(), stream=st)
                return d_off.cpu().numpy().view(np.uint64), fetch_hits(rep_dev, p, n)

            (ooff, ohits), (noff, nhits) = both_paths(locate)
            assert np.array_equal(ooff, woff) and np.array_equal(noff, woff), pad
            assert np.array_equal(ohits, whits) and np.array_equal(nhits, whits), pad


@pytest.mark.parametrize("locate_variant", [0, 1])
def test_host_calls_without_host_packing(rep, rep_dev, po, locate_variant):
    from awry_b200 import fm_index as f
    qb, qo = sweep_queries(rep[0], rep[1], seed=3)
    orc = oracle_from_parts(po, rep[0])
    want, _ = orc.count_batch(qb, qo)
    woff, whits, _ = orc.locate_batch(qb, qo)
    f.set_host_pack(0)
    f.set_locate_variant(locate_variant)
    old, new = both_paths(lambda: rep_dev.count_packed(qb, qo))
    assert np.array_equal(old, want) and np.array_equal(new, want)
    old, new = both_paths(lambda: rep_dev.locate_packed(qb, qo))
    for off, hits in (old, new):
        assert np.array_equal(off, woff) and np.array_equal(hits, whits)


def test_refused_batches_name_the_same_query(rep, rep_dev):
    import torch
    from awry_b200 import AwryError
    from awry_b200 import fm_index as f
    t = bytes(rep[0].text)
    reads = [t[1000 + 37 * i:1000 + 37 * i + 20 + i % 200] for i in range(3000)]
    qb0, qo0 = f.pack_queries(reads)
    want = rep_dev.count_packed(qb0, qo0)
    st = torch.cuda.current_stream().cuda_stream
    f.set_host_pack(0)

    def err(call):
        with pytest.raises(AwryError) as e:
            call()
        return e.value.code, str(e.value)

    for bad_at, bad in ((0, b"AC$GT"), (1777, b"#"), (2999, b"ACGT" * 70 + b"$"), (5, b""), (2400, b"")):
        qs = list(reads)
        qs[bad_at] = bad
        qs[2500] = b""                                   # a later empty query: the first one is named
        qb, qo = f.pack_queries(qs)
        old, new = both_paths(lambda: err(lambda: rep_dev.count_packed(qb, qo)))
        assert old == new and "query %d" % min(bad_at, 2500) in new[1], (old, new)
        old, new = both_paths(lambda: err(lambda: rep_dev.locate_packed(qb, qo)))
        assert old == new, (old, new)
        d_qb, d_qo = device_copy(qb, 3), torch.from_numpy(qo.view(np.int64)).cuda()

        def device():
            d_c = torch.zeros(len(qs), dtype=torch.int64, device="cuda")
            rep_dev.count_device(d_qb.data_ptr() + 3, d_qo.data_ptr(), len(qs), d_c.data_ptr(), st)
            e = err(lambda: rep_dev.device_check(st))
            return e, d_c.cpu().numpy()

        (eo, co), (en, cn) = both_paths(device)
        assert eo == en and co[2500] == 0 and cn[2500] == 0, (eo, en)
    # non-monotone offsets (device entry point: latched, named by device_check)
    for bad_at, val in ((1, 10**6), (1500, 0), (2999, 10**12)):
        o = qo0.copy()
        o[bad_at] = val
        d_qb, d_qo = device_copy(qb0, 0), torch.from_numpy(o.view(np.int64)).cuda()

        def device():
            d_c = torch.full((len(reads),), 9, dtype=torch.int64, device="cuda")
            rep_dev.count_device(d_qb.data_ptr(), d_qo.data_ptr(), len(reads), d_c.data_ptr(), st)
            return err(lambda: rep_dev.device_check(st)), d_c.cpu().numpy()

        # (the other reads' counts are not compared: with the separate packing pass, a read that the broken offsets
        # make longer than the batch overwrites the packed words of its neighbours)
        (eo, co), (en, cn) = both_paths(device)
        assert eo == en and eo[0] == -1, (eo, en)
        assert co[bad_at - 1] == 0 and cn[bad_at - 1] == 0     # a refused query gets the empty result
    torch.cuda.synchronize()
    assert np.array_equal(rep_dev.count_packed(qb0, qo0), want)     # no sticky error


def test_on_the_bounds_checked_build():
    """this file against libawry_b200_checked.so (every data-dependent load bounds-checked, layout.cuh): no assert"""
    checked = os.path.join(ROOT, "awry_b200", "libawry_b200_checked.so")
    if os.environ.get("AWRY_B200_LIB"):
        pytest.skip("already running against another build")
    if not os.path.exists(checked):
        subprocess.check_call(["make", "-s", "-C", os.path.join(ROOT, "awry_b200", "csrc"), "checked"])
    env = dict(os.environ, AWRY_B200_LIB=checked)
    out = subprocess.run([sys.executable, "-m", "pytest", "tests/test_gpu_ascii_wave.py", "-m", "gpu", "-x", "-q",
                          "-p", "no:cacheprovider", "-k", "not bounds_checked"],
                         cwd=ROOT, env=env, capture_output=True, text=True, timeout=1200)
    tail = out.stdout[-1500:] + out.stderr[-1500:]
    assert out.returncode == 0, tail
    assert " passed" in out.stdout and "Assertion" not in out.stderr, tail
