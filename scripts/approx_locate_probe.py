"""Device-resident locate of the approximate searches at full size (awry_locate_device_{hamming,edit}[_strands]).

Workload: the 3.1 Gbp synthetic index of scripts/hamming_probe.py and 10 M x 150-bp device-resident reads: for Hamming
the reads of hamming_probe.py (read q with q % 4 planted substitutions), for edit distance those of edit_probe.py (q % 4
planted substitutions, insertions and deletions); on both strands every odd read is reverse-complemented.  For each
metric, strand count and k = 0 .. 3 it times the locate-device call (outputs freed after each call) against the
count-device call of the same metric on the same reads, with CUDA events: a warm-up, then REPS rounds of one 10-call
window per arm, arms alternating; medians and spread (max - min).  Both calls synchronise inside, so a window measures
whole calls, not the enqueue.
Checks in the same run, per metric, strand count and k: the hit total equals the count total; hit_off equals the
exclusive scan of the per-read count sums; on the first SAMPLE reads the hits and distances equal the host-buffer
call's; every read with at most k planted edits has a hit at its origin on its own strand.
Then cfg3 (1 M x 50 bp, q % 4 planted edits, k = 2): the locate-device call against the host-buffer locate, one strand
and both.  The card name and power limit are printed with the numbers."""
import argparse
import ctypes as C
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))
import torch  # noqa: E402

from awry_b200 import FmIndex  # noqa: E402
from edit_probe import alternate, edited_reads  # noqa: E402
from fixtures import pyfixture_gpu as fxg  # noqa: E402
from hamming_probe import card, plant, reverse_complement_rows  # noqa: E402

def mix64(z):
    z = z + np.uint64(0x9E3779B97F4A7C15)
    z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
    z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
    return z ^ (z >> np.uint64(31))


def origins(n, L, nq, qseed):
    """the text position fixtures/fixture_gpu.cu's gen_queries_kernel cut read q from: umulhi(rnd_at(qseed, q), span)"""
    with np.errstate(over="ignore"):
        q = np.arange(nq, dtype=np.uint64)
        r = mix64(mix64(np.array([qseed], np.uint64))[0] ^ (q * np.uint64(0xD1342543DE82EF95)))
        span = np.uint64(n - L + 1)
        lo, hi = r & np.uint64(0xFFFFFFFF), r >> np.uint64(32)
        return (hi * span + ((lo * span) >> np.uint64(32))) >> np.uint64(32)


def to_torch(ptr, n, dtype, width=1):
    out = torch.empty((max(1, n), width), dtype=dtype, device="cuda")
    if n:
        nbytes = n * width * out.element_size()
        assert C.CDLL("libcudart.so").cudaMemcpy(C.c_void_p(out.data_ptr()), C.c_void_p(ptr), C.c_size_t(nbytes), 3) == 0
    return out[:n]


def reads(a, metric, nq, L, seed):
    """-> (device reads, planted edits per read, origin per read)"""
    if metric == "edit":
        # edit_probe.edited_reads cuts read q from a window of L + 3 symbols, seeded per chunk of 1 M reads; the read
        # starts behind as many window symbols as it has planted insertions (edit j of read q has kind (q // 4 + j) % 3,
        # 1 = insertion), so that text position is its origin: d(origin) <= the planted edits
        d, m = edited_reads(a.n, nq, L, seed)
        chunk = 1_000_000
        pos = np.concatenate([origins(a.n, L + 3, min(chunk, nq - c0), seed + c0) for c0 in range(0, nq, chunk)])
        q = np.arange(nq)
        n_ins = sum(((q % 4 > j) & ((q // 4 + j) % 3 == 1)).astype(np.uint64) for j in range(3))
        return d, m, pos + n_ins
    d = torch.empty(nq * L, dtype=torch.uint8, device="cuda")
    fxg.gen_queries_device(0, a.n, 3, nq, L, seed, d.data_ptr())
    return d, plant(d, nq, L, seed + 1), origins(a.n, L, nq, seed)


def calls(ix, metric, strands):
    s = "_strands" if strands else ""
    return (getattr(ix, f"count_{metric}{s}_device"), getattr(ix, f"locate_{metric}{s}_device"),
            getattr(ix, f"locate_{metric}{s}_packed"))


def check(ix, metric, strands, k, d, off, nq, L, m, origin, counts, sample, st):
    """the checks of one (metric, strands, k) on the reads of the timed run -> one line"""
    per = 2 if strands else 1
    count, locate, host = calls(ix, metric, strands)
    d_off = torch.full((per * nq + 1,), -1, dtype=torch.int64, device="cuda")
    hp, dp, n = locate(d.data_ptr(), off.data_ptr(), nq, k, d_off.data_ptr(), stream=st)
    ix.device_check(st)
    torch.cuda.synchronize()
    hits = to_torch(hp, n, torch.int64, 2)
    dist = to_torch(dp, n, torch.uint8)[:, 0]
    ix.device_free(hp)
    ix.device_free(dp)
    sums = counts.view(per * nq, k + 1).sum(dim=1)
    total_ok = n == int(sums.sum())
    scan = torch.zeros(per * nq + 1, dtype=torch.int64, device="cuda")
    scan[1:] = torch.cumsum(sums, 0)
    off_ok = bool(torch.equal(scan, d_off))
    # the first `sample` reads against the host-buffer call
    qb = d[: sample * L].cpu().numpy()
    qo = np.arange(sample + 1, dtype=np.uint64) * np.uint64(L)
    hoff, hhits, hd = host(qb, qo, k, capacity=int(d_off[per * sample]) + 1)
    e = int(hoff[-1])
    sample_ok = (np.array_equal(hoff, d_off[: per * sample + 1].cpu().numpy().view(np.uint64))
                 and np.array_equal(hhits, hits[:e].cpu().numpy().view(np.uint64)) and np.array_equal(hd, dist[:e].cpu().numpy()))
    # every read with <= k planted edits has a hit at its origin on its own strand (one record: local_pos = position)
    v = torch.repeat_interleave(torch.arange(per * nq, device="cuda"), torch.diff(d_off))
    q = v // per
    own = (v % per) == (q % 2) if strands else torch.ones_like(q, dtype=torch.bool)
    org = torch.from_numpy(origin.view(np.int64)).cuda()
    at = own & (hits[:, 1] == org[q]) & (hits[:, 0] == 0)
    found = torch.zeros(nq, dtype=torch.bool, device="cuda")
    found[q[at]] = True
    want = m <= k
    origin_ok = bool(found[want].all())
    return (f"{metric} {'both strands' if strands else 'one strand'} k = {k}: {n} hits; hit total == count total: "
            f"{total_ok}; hit_off == scan of the count sums: {off_ok}; first {sample} reads == host call: {sample_ok}; "
            f"reads with <= k planted edits found at their origin on their own strand: {origin_ok} "
            f"({int(found[want].sum())} of {int(want.sum())})")


def bench(a, ix, metric, st):
    L, nq = 150, a.nq
    t0 = time.time()
    d, m, origin = reads(a, metric, nq, L, 4 if metric == "hamming" else 5)
    off = torch.arange(0, nq + 1, dtype=torch.int64, device="cuda") * L
    print(f"{metric}: {nq} reads ready in {time.time() - t0:.1f} s", flush=True)
    for strands in (False, True):
        if strands:
            reverse_complement_rows(d, nq, L, torch.arange(nq, device="cuda") % 2 == 1)
        per = 2 if strands else 1
        count, locate, _ = calls(ix, metric, strands)
        counts = {k: torch.zeros((per * nq, k + 1), dtype=torch.int64, device="cuda") for k in range(4)}
        d_off = torch.zeros(per * nq + 1, dtype=torch.int64, device="cuda")

        def loc(k):
            hp, dp, _ = locate(d.data_ptr(), off.data_ptr(), nq, k, d_off.data_ptr(), stream=st)
            ix.device_free(hp)
            ix.device_free(dp)
        arms = {}
        for k in range(4):
            arms[f"k = {k} count"] = lambda k=k: count(d.data_ptr(), off.data_ptr(), nq, k, counts[k].data_ptr(), st)
            arms[f"k = {k} locate"] = lambda k=k: loc(k)
        med, spread = alternate(arms, a.reps)
        ix.device_check(st)
        print(f"{metric}, {'both strands' if strands else 'one strand'}, {nq / 1e6:.0f} M x {L}-bp device-resident "
              f"reads; median of {a.reps} alternating windows of 10 calls after a warm-up (spread = max - min):",
              flush=True)
        for k in range(4):
            c, lo = med[f"k = {k} count"], med[f"k = {k} locate"]
            print(f"  k = {k}: count-device {c:.3f} ms (spread {spread[f'k = {k} count']:.3f}), locate-device "
                  f"{lo:.3f} ms (spread {spread[f'k = {k} locate']:.3f}), locate / count = {lo / c:.2f}", flush=True)
        for k in range(4):
            print("  " + check(ix, metric, strands, k, d, off, nq, L, m, origin, counts[k], a.sample, st), flush=True)
    del d
    torch.cuda.empty_cache()


def cfg3(a, ix, st):
    nq, L = 1_000_000, 50
    for metric in ("hamming", "edit"):
        d, m, origin = reads(a, metric, nq, L, 7)
        off = torch.arange(0, nq + 1, dtype=torch.int64, device="cuda") * L
        for strands in (False, True):
            if strands:
                reverse_complement_rows(d, nq, L, torch.arange(nq, device="cuda") % 2 == 1)
            per = 2 if strands else 1
            count, locate, host = calls(ix, metric, strands)
            counts = torch.zeros((per * nq, 3), dtype=torch.int64, device="cuda")
            count(d.data_ptr(), off.data_ptr(), nq, 2, counts.data_ptr(), st)
            torch.cuda.synchronize()
            total = int(counts.sum())
            qb, qo = d.cpu().numpy(), np.arange(nq + 1, dtype=np.uint64) * np.uint64(L)
            d_off = torch.zeros(per * nq + 1, dtype=torch.int64, device="cuda")

            def loc():
                hp, dp, _ = locate(d.data_ptr(), off.data_ptr(), nq, 2, d_off.data_ptr(), stream=st)
                ix.device_free(hp)
                ix.device_free(dp)
            med, spread = alternate({"device": loc, "host": lambda: host(qb, qo, 2, capacity=total + 1)}, a.reps, n=3)
            line = check(ix, metric, strands, 2, d, off, nq, L, m, origin, counts, a.sample, st)
            print(f"cfg3 (1 M x 50 bp, q % 4 planted edits, k = 2) {metric} {'both strands' if strands else 'one strand'}: "
                  f"locate-device {med['device']:.3f} ms (spread {spread['device']:.3f}), host-buffer locate "
                  f"{med['host']:.3f} ms (spread {spread['host']:.3f}); {line}", flush=True)
        del d
        torch.cuda.empty_cache()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=3_100_000_000)
    ap.add_argument("--nq", type=int, default=10_000_000)
    ap.add_argument("--sample", type=int, default=10_000)
    ap.add_argument("--reps", type=int, default=5)
    a = ap.parse_args()
    print(card(), flush=True)
    st = torch.cuda.current_stream().cuda_stream
    t0 = time.time()
    parts, _ = fxg.build_parts(0, a.n, 3, ratio=8, kmer_len=13)
    ix = FmIndex.from_parts(parts.alphabet, parts.ratio, parts.bwt_len, parts.kmer_len, parts.blocks, parts.prefix_sums,
                            parts.sa_words)
    del parts
    print(f"index of {a.n} symbols ready in {time.time() - t0:.1f} s", flush=True)
    for metric in ("hamming", "edit"):
        bench(a, ix, metric, st)
    cfg3(a, ix, st)
    print(card(), flush=True)


if __name__ == "__main__":
    main()
