"""Hamming search at full size (awry_count_device_hamming / awry_locate_batch_hamming).

Workload: the 3.1 Gbp synthetic index of scripts/text_finish_probe.py and 10 M x 150-bp device-resident reads, read q
carrying exactly q % 4 substitutions (distinct positions, each base changed, planted with torch on the device).
Times the device-resident count for k = 0 .. 3 with CUDA events (10 launches after a warm-up) beside the exact
awry_count_device on the same reads; then cfg3 (1 M x 50 bp) and cfg5 (repeat-rich text, 1 M x 50 bp) at k = 2,
count and locate.  Checks: a read with d planted substitutions has a window at distance <= d when k >= d; and on
10 k sampled reads at k = 1 the distance-1 count equals the sum of exact counts (awry_count_batch) over every
single-substitution variant of the read (each position set to each other symbol of ACGTN) -- an independent check
through the exact path.  Card name and power limit are printed with the numbers."""
import argparse
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

from awry_b200 import FmIndex, fm_index as f  # noqa: E402
from fixtures import pyfixture_gpu as fxg, repeats  # noqa: E402


def plant(d_reads, nq, L, seed):
    """read q gets exactly q % 4 substitutions at distinct positions p0 + i * step (mod L), step in [1, L/4)"""
    g = torch.Generator(device="cuda").manual_seed(seed)
    reads = d_reads.view(nq, L)
    lut = torch.zeros(256, dtype=torch.int64, device="cuda")
    for i, c in enumerate(b"ACGT"):
        lut[c] = i
    acgt = torch.tensor(list(b"ACGT"), dtype=torch.uint8, device="cuda")
    m = torch.arange(nq, device="cuda") % 4
    p0 = torch.randint(0, L, (nq,), device="cuda", generator=g)
    step = torch.randint(1, L // 4, (nq,), device="cuda", generator=g)
    rows = torch.arange(nq, device="cuda")
    for i in range(3):
        sel = rows[m > i]
        pos = (p0[sel] + i * step[sel]) % L
        old = reads[sel, pos]
        shift = torch.randint(1, 4, (len(sel),), device="cuda", generator=g)
        new = acgt[(lut[old.long()] + shift) % 4]
        new = torch.where(new == old, acgt[(lut[old.long()] + 1) % 4], new)   # (a non-ACGT base: any ACGT changes it)
        reads[sel, pos] = new
    return m


def time_calls(fn, n=10):
    for _ in range(2):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=3_100_000_000)
    ap.add_argument("--nq", type=int, default=10_000_000)
    ap.add_argument("--sample", type=int, default=10_000)
    ap.add_argument("--cfg5-n", type=int, default=1_000_000_000)
    a = ap.parse_args()
    print(subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip(), flush=True)
    st = torch.cuda.current_stream().cuda_stream
    L, nq = 150, a.nq
    t0 = time.time()
    parts, _ = fxg.build_parts(0, a.n, 3, ratio=8, kmer_len=13)
    ix = FmIndex.from_parts(parts.alphabet, parts.ratio, parts.bwt_len, parts.kmer_len, parts.blocks, parts.prefix_sums,
                            parts.sa_words)
    print(f"index of {a.n} symbols built and loaded in {time.time() - t0:.1f} s; device bytes {ix.device_bytes()}", flush=True)
    d = torch.empty(nq * L, dtype=torch.uint8, device="cuda")
    fxg.gen_queries_device(0, a.n, 3, nq, L, 4, d.data_ptr())
    m = plant(d, nq, L, 5)
    off = torch.arange(0, nq + 1, dtype=torch.int64, device="cuda") * L
    exact = torch.zeros(nq, dtype=torch.int64, device="cuda")
    ms = time_calls(lambda: ix.count_device(d.data_ptr(), off.data_ptr(), nq, exact.data_ptr(), st))
    print(f"exact count (awry_count_device): {ms:.2f} ms per {nq / 1e6:.0f} M reads = {nq / ms / 1e6:.2f} G reads/s", flush=True)
    for k in range(4):
        cnt = torch.zeros((nq, k + 1), dtype=torch.int64, device="cuda")
        ms = time_calls(lambda: ix.count_hamming_device(d.data_ptr(), off.data_ptr(), nq, k, cnt.data_ptr(), st))
        ix.device_check(st)
        f.profile_enable(True)   # per-kernel split in calls of their own (event timing adds a synchronisation)
        f.profile_reset()
        per = 3
        for _ in range(per):
            ix.count_hamming_device(d.data_ptr(), off.data_ptr(), nq, k, cnt.data_ptr(), st)
        torch.cuda.synchronize()
        p = f.profile_get()
        f.profile_enable(False)
        has = torch.zeros(nq, dtype=torch.bool, device="cuda")
        for dd in range(k + 1):
            has |= cnt[:, dd] > 0
        ok = bool(has[m <= k].all())
        same0 = bool(torch.equal(cnt[:, 0], exact))
        print(f"k = {k}: {ms:.2f} ms per {nq / 1e6:.0f} M reads = {nq / ms / 1e6:.2f} G reads/s; per call: piece search "
              f"{p['search_ms'] / per:.2f} ms, verification {p['walk_ms'] / per:.2f} ms, packing {p['pack_ms'] / per:.2f} ms; "
              f"reads with <= k planted substitutions all found: {ok}; distance-0 counts == exact counts: {same0}; "
              f"windows per read by distance {[round(float(cnt[:, dd].double().mean()), 3) for dd in range(k + 1)]}", flush=True)
        if k == 1:
            c1 = cnt
    # independent check through the exact path: distance-1 count = sum of exact counts of the 4 L one-symbol variants
    rng = np.random.default_rng(1)
    sample = np.sort(rng.choice(nq, a.sample, replace=False))
    reads = d.view(nq, L)[torch.from_numpy(sample).cuda()].cpu().numpy()
    syms = np.frombuffer(b"ACGTN", np.uint8)
    var = []
    for r in reads:
        v = np.repeat(r[None, :], 4 * L, axis=0)
        for p in range(L):
            alts = syms[syms != r[p]][:4]
            v[4 * p: 4 * p + 4, p] = alts
        var.append(v)
    var = np.concatenate(var).reshape(-1)
    voff = np.arange(a.sample * 4 * L + 1, dtype=np.uint64) * np.uint64(L)
    t0 = time.time()
    vc = ix.count_packed(var, voff).reshape(a.sample, 4 * L).sum(axis=1)
    got = c1[torch.from_numpy(sample).cuda(), 1].cpu().numpy().view(np.uint64)
    print(f"k = 1 distance-1 counts of {a.sample} sampled reads == sum of exact counts over their {4 * L} variants: "
          f"{bool(np.array_equal(vc, got))} ({int((got > 0).sum())} reads with a distance-1 window; "
          f"{len(var) // L} exact queries in {time.time() - t0:.1f} s)", flush=True)
    del d, var
    # cfg3: 1 M x 50-bp reads from the same index, k = 2
    nq3, L3 = 1_000_000, 50
    d3 = torch.empty(nq3 * L3, dtype=torch.uint8, device="cuda")
    fxg.gen_queries_device(0, a.n, 3, nq3, L3, 6, d3.data_ptr())
    plant(d3, nq3, L3, 7)
    off3 = torch.arange(0, nq3 + 1, dtype=torch.int64, device="cuda") * L3
    cnt3 = torch.zeros((nq3, 3), dtype=torch.int64, device="cuda")
    ms = time_calls(lambda: ix.count_hamming_device(d3.data_ptr(), off3.data_ptr(), nq3, 2, cnt3.data_ptr(), st))
    qb3, qo3 = d3.cpu().numpy(), np.arange(nq3 + 1, dtype=np.uint64) * np.uint64(L3)
    ix.locate_hamming_packed(qb3, qo3, 2)
    t0 = time.time()
    hoff, hits, mm = ix.locate_hamming_packed(qb3, qo3, 2, capacity=int(cnt3.sum()) + 1)
    tl = time.time() - t0
    print(f"cfg3 (1 M x 50 bp, k = 2): device count {ms:.2f} ms; host-buffer locate {tl * 1e3:.1f} ms for {len(hits)} hits "
          f"(counts sum == hits: {int(cnt3.sum()) == len(hits)})", flush=True)
    del ix, d3
    torch.cuda.empty_cache()
    # cfg5: repeat-rich text, 1 M x 50-bp reads, k = 2
    n5 = a.cfg5_n
    scale = n5 / 1e9
    fams = ((300, int(100_000 * scale) + 10, 0.15), (6000, int(20_000 * scale) + 5, 0.15))
    text, regions = repeats.repeat_rich_text(n5, seed=8, tandem_arrays=max(4, int(40 * scale)), families=fams)
    parts5, _ = fxg.build_parts(0, n5, 0, ratio=32, kmer_len=13, host_text=text)
    qb5, qo5 = repeats.repeat_queries(text, regions, nq3, L3, seed=9)
    del text
    ix5 = FmIndex.from_parts(parts5.alphabet, parts5.ratio, parts5.bwt_len, parts5.kmer_len, parts5.blocks,
                             parts5.prefix_sums, parts5.sa_words)
    dq5, do5 = torch.from_numpy(qb5).cuda(), torch.from_numpy(qo5.view(np.int64)).cuda()
    cnt5 = torch.zeros((nq3, 3), dtype=torch.int64, device="cuda")
    ms = time_calls(lambda: ix5.count_hamming_device(dq5.data_ptr(), do5.data_ptr(), nq3, 2, cnt5.data_ptr(), st), n=5)
    total = int(cnt5.sum())
    print(f"cfg5 ({n5 / 1e9:.2f} Gbp repeat-rich, 1 M x 50 bp, k = 2): device count {ms:.2f} ms; {total} windows, "
          f"max {int(cnt5.sum(dim=1).max())} for one read", flush=True)
    # locate of every read would return all those windows (17 bytes each): the first reads only
    nl = 10_000
    want = int(cnt5[:nl].sum())
    ix5.locate_hamming_packed(qb5[: nl * L3], qo5[: nl + 1], 2, capacity=want + 1)
    t0 = time.time()
    hoff, hits, mm = ix5.locate_hamming_packed(qb5[: nl * L3], qo5[: nl + 1], 2, capacity=want + 1)
    tl = time.time() - t0
    key = (hits[:, 0] << np.uint64(40)) | hits[:, 1]
    first = np.zeros(len(hits), bool)
    first[hoff[:-1][hoff[:-1] < hoff[1:]].astype(np.int64)] = True
    ordered = bool((np.diff(key.astype(np.int64))[~first[1:]] > 0).all())
    print(f"cfg5 host-buffer locate of the first {nl} reads: {tl * 1e3:.1f} ms for {len(hits)} hits "
          f"(== counts: {len(hits) == want}; ascending and distinct within every read: {ordered})", flush=True)


if __name__ == "__main__":
    main()
