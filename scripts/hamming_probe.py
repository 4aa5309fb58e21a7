"""Hamming search at full size (awry_count_device_hamming / awry_locate_batch_hamming).

Workload: the 3.1 Gbp synthetic index of scripts/text_finish_probe.py and 10 M x 150-bp device-resident reads, read q
carrying exactly q % 4 substitutions (distinct positions, each base changed, planted with torch on the device).
Times the device-resident count for k = 0 .. 3 with CUDA events (10 launches after a warm-up) beside the exact
awry_count_device on the same reads; then cfg3 (1 M x 50 bp) and cfg5 (repeat-rich text, 1 M x 50 bp) at k = 2,
count and locate.  Checks: a read with d planted substitutions has a window at distance <= d when k >= d; and on
10 k sampled reads at k = 1 the distance-1 count equals the sum of exact counts (awry_count_batch) over every
single-substitution variant of the read (each position set to each other symbol of ACGTN) -- an independent check
through the exact path.  Card name and power limit are printed with the numbers.

--arm strands: the both-strand arm on the same index and reads, every odd read reverse-complemented on the device so
that both strands have true hits.  Times awry_count_device_hamming_strands at k = 0 .. 3 beside the single-strand
awry_count_device_hamming, awry_count_device_strands and awry_count_device (arms alternating, REPS windows of 10 calls,
medians), checks that strand-0 counts equal the single-strand counts and that every read with <= k substitutions is
found on its own strand, then cfg3 at k = 2: device count and host-buffer locate on both strands.
--arm single: the single-strand device count at k = 0 .. 3 only, one JSON line (for --ab).
--ab DIR: runs --arm single alternately with the library in this tree and with the awry_b200 package in DIR (another
build, e.g. the parent commit's: its Python module and its libawry_b200.so), REPS times each, and prints the medians."""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
if os.environ.get("HAMMING_PROBE_PKG"):   # --ab: the awry_b200 package of another build comes first
    sys.path.insert(0, os.environ["HAMMING_PROBE_PKG"])
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


def reverse_complement_rows(d_q, nq, L, rows):
    """reads `rows` (a bool mask over nq) of the flat byte buffer d_q replaced by their reverse complements"""
    lut = torch.arange(256, dtype=torch.uint8, device="cuda")
    for a, b in (b"AT", b"TA", b"CG", b"GC"):
        lut[a] = b
    v = d_q.view(nq, L)
    v[rows] = lut[v[rows].flip(1).long()]
    return d_q


def card():
    return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                          capture_output=True, text=True).stdout.strip().splitlines()[0]


def bench_reads(a, strands):
    """the index and the 10 M x 150-bp reads with q % 4 planted substitutions (odd reads reverse-complemented when
    `strands`)"""
    L, nq = 150, a.nq
    t0 = time.time()
    parts, _ = fxg.build_parts(0, a.n, 3, ratio=8, kmer_len=13)
    ix = FmIndex.from_parts(parts.alphabet, parts.ratio, parts.bwt_len, parts.kmer_len, parts.blocks, parts.prefix_sums,
                            parts.sa_words)
    print(f"index of {a.n} symbols built and loaded in {time.time() - t0:.1f} s", file=sys.stderr, flush=True)
    d = torch.empty(nq * L, dtype=torch.uint8, device="cuda")
    fxg.gen_queries_device(0, a.n, 3, nq, L, 4, d.data_ptr())
    m = plant(d, nq, L, 5)
    if strands:
        reverse_complement_rows(d, nq, L, torch.arange(nq, device="cuda") % 2 == 1)
    off = torch.arange(0, nq + 1, dtype=torch.int64, device="cuda") * L
    return ix, d, off, m


def alternate(arms, reps, n=10):
    """arms: name -> fn; REPS rounds, each arm one window of n calls per round -> name -> median ms"""
    ms = {name: [] for name in arms}
    for _ in range(reps):
        for name, fn in arms.items():
            ms[name].append(time_calls(fn, n))
    return {name: statistics.median(v) for name, v in ms.items()}, {name: max(v) - min(v) for name, v in ms.items()}


def arm_single(a):
    """the single-strand device count at k = 0 .. 3 (both-strand reads), one JSON line on stdout"""
    st = torch.cuda.current_stream().cuda_stream
    ix, d, off, _ = bench_reads(a, True)
    nq = a.nq
    cnt = {k: torch.zeros((nq, k + 1), dtype=torch.int64, device="cuda") for k in range(4)}
    arms = {k: (lambda k=k: ix.count_hamming_device(d.data_ptr(), off.data_ptr(), nq, k, cnt[k].data_ptr(), st))
            for k in range(4)}
    med, _ = alternate(arms, a.reps)
    ix.device_check(st)
    digest = [int((cnt[k] * torch.arange(1, k + 2, device="cuda")).sum()) for k in range(4)]
    print(json.dumps({"lib": f.library_path(), "ms": [med[k] for k in range(4)], "digest": digest}), flush=True)


def run_ab(a):
    """--arm single alternately with this tree's library and with the package in a.ab"""
    other = os.path.abspath(a.ab)
    print(card(), flush=True)
    res = {"this tree": [], os.path.relpath(other, ROOT): []}
    for _ in range(a.ab_rounds):
        for name in res:
            env = dict(os.environ)
            env.pop("HAMMING_PROBE_PKG", None)
            env.pop("AWRY_B200_LIB", None)
            if name != "this tree":
                env["HAMMING_PROBE_PKG"] = other
                env["AWRY_B200_LIB"] = os.path.join(other, "awry_b200", "libawry_b200.so")
            out = subprocess.run([sys.executable, os.path.abspath(__file__), "--arm", "single", "--reps", str(a.reps),
                                  "--n", str(a.n), "--nq", str(a.nq)], env=env, capture_output=True, text=True, check=True)
            line = json.loads(out.stdout.strip().splitlines()[-1])
            res[name].append(line)
            print(f"{os.path.relpath(line['lib'], ROOT)}: k = 0 .. 3 " + " ".join(f"{x:.3f}" for x in line["ms"]) + " ms",
                  flush=True)
    for name, lines in res.items():
        med = [statistics.median(l["ms"][k] for l in lines) for k in range(4)]
        print(f"median over {len(lines)} processes, {name}: " + " ".join(f"k={k} {med[k]:.3f} ms" for k in range(4)),
              flush=True)
    digests = {json.dumps(l["digest"]) for lines in res.values() for l in lines}
    print(f"per-distance count digests identical across builds: {len(digests) == 1}", flush=True)


def arm_strands(a):
    print(card(), flush=True)
    st = torch.cuda.current_stream().cuda_stream
    L, nq = 150, a.nq
    ix, d, off, m = bench_reads(a, True)
    odd = torch.arange(nq, device="cuda") % 2 == 1
    exact = torch.zeros(nq, dtype=torch.int64, device="cuda")
    exact2 = torch.zeros((nq, 2), dtype=torch.int64, device="cuda")
    one = {k: torch.zeros((nq, k + 1), dtype=torch.int64, device="cuda") for k in range(4)}
    two = {k: torch.zeros((nq, 2, k + 1), dtype=torch.int64, device="cuda") for k in range(4)}
    arms = {"exact single strand (awry_count_device)":
            lambda: ix.count_device(d.data_ptr(), off.data_ptr(), nq, exact.data_ptr(), st),
            "exact both strands (awry_count_device_strands)":
            lambda: ix.count_strands_device(d.data_ptr(), off.data_ptr(), nq, exact2.data_ptr(), st)}
    for k in range(4):
        arms[f"k = {k} single strand (awry_count_device_hamming)"] = \
            lambda k=k: ix.count_hamming_device(d.data_ptr(), off.data_ptr(), nq, k, one[k].data_ptr(), st)
        arms[f"k = {k} both strands (awry_count_device_hamming_strands)"] = \
            lambda k=k: ix.count_hamming_strands_device(d.data_ptr(), off.data_ptr(), nq, k, two[k].data_ptr(), st)
    med, spread = alternate(arms, a.reps)
    ix.device_check(st)
    print(f"10 M x 150-bp device-resident reads, read q with q % 4 substitutions, odd reads reverse-complemented; "
          f"median of {a.reps} alternating windows of 10 calls (spread = max - min):", flush=True)
    for name in arms:
        print(f"  {name}: {med[name]:.3f} ms (spread {spread[name]:.3f})", flush=True)
    for k in range(4):
        same = bool(torch.equal(two[k][:, 0], one[k]))
        found = torch.where(odd, two[k][:, 1].sum(dim=1) > 0, two[k][:, 0].sum(dim=1) > 0)
        ok = bool(found[m <= k].all())
        same0 = bool(torch.equal(two[k][:, :, 0], exact2))
        print(f"k = {k}: both strands / single strand = {med[f'k = {k} both strands (awry_count_device_hamming_strands)'] / med[f'k = {k} single strand (awry_count_device_hamming)']:.2f}; "
              f"strand-0 counts == awry_count_device_hamming: {same}; distance-0 counts == awry_count_device_strands: "
              f"{same0}; reads with <= k substitutions found on their own strand: {ok}; windows per read by strand and "
              f"distance {[[round(float(two[k][:, s, dd].double().mean()), 3) for dd in range(k + 1)] for s in (0, 1)]}",
              flush=True)
    del d
    # cfg3: 1 M x 50-bp reads, k = 2, odd reads reverse-complemented
    nq3, L3 = 1_000_000, 50
    d3 = torch.empty(nq3 * L3, dtype=torch.uint8, device="cuda")
    fxg.gen_queries_device(0, a.n, 3, nq3, L3, 6, d3.data_ptr())
    plant(d3, nq3, L3, 7)
    reverse_complement_rows(d3, nq3, L3, torch.arange(nq3, device="cuda") % 2 == 1)
    off3 = torch.arange(0, nq3 + 1, dtype=torch.int64, device="cuda") * L3
    c1 = torch.zeros((nq3, 3), dtype=torch.int64, device="cuda")
    c2 = torch.zeros((nq3, 2, 3), dtype=torch.int64, device="cuda")
    med3, _ = alternate({
        "single": lambda: ix.count_hamming_device(d3.data_ptr(), off3.data_ptr(), nq3, 2, c1.data_ptr(), st),
        "both": lambda: ix.count_hamming_strands_device(d3.data_ptr(), off3.data_ptr(), nq3, 2, c2.data_ptr(), st)},
        a.reps)
    qb3, qo3 = d3.cpu().numpy(), np.arange(nq3 + 1, dtype=np.uint64) * np.uint64(L3)
    tl = {}
    for name, fn, cap in (("single", ix.locate_hamming_packed, int(c1.sum()) + 1),
                          ("both", ix.locate_hamming_strands_packed, int(c2.sum()) + 1)):
        fn(qb3, qo3, 2, capacity=cap)
        t0 = time.time()
        hoff, hits, mm = fn(qb3, qo3, 2, capacity=cap)
        tl[name] = (time.time() - t0, len(hits))
    print(f"cfg3 (1 M x 50 bp, k = 2, odd reads reverse-complemented): device count {med3['single']:.3f} ms single strand, "
          f"{med3['both']:.3f} ms both strands; host-buffer locate {tl['single'][0] * 1e3:.1f} ms single strand "
          f"({tl['single'][1]} hits), {tl['both'][0] * 1e3:.1f} ms both strands ({tl['both'][1]} hits; counts sum == "
          f"hits: {int(c2.sum()) == tl['both'][1]}; strand-0 counts == single strand: {bool(torch.equal(c2[:, 0], c1))})",
          flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=3_100_000_000)
    ap.add_argument("--nq", type=int, default=10_000_000)
    ap.add_argument("--sample", type=int, default=10_000)
    ap.add_argument("--cfg5-n", type=int, default=1_000_000_000)
    ap.add_argument("--arm", choices=["all", "strands", "single"], default="all")
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--ab", default=None)
    ap.add_argument("--ab-rounds", type=int, default=3)
    a = ap.parse_args()
    if a.ab:
        return run_ab(a)
    if a.arm == "single":
        return arm_single(a)
    if a.arm == "strands":
        return arm_strands(a)
    print(card(), flush=True)
    st = torch.cuda.current_stream().cuda_stream
    L, nq = 150, a.nq
    ix, d, off, m = bench_reads(a, False)
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
