"""Edit-distance search at full size (awry_count_device_edit, awry_*_batch_edit).

Workload: the 3.1 Gbp synthetic index of scripts/hamming_probe.py and 10 M x 150-bp device-resident reads, read q
carrying exactly q % 4 planted edits: substitutions, insertions and deletions in turn (edit i of read q has kind
(q // 4 + i) % 3), at distinct positions, cut from a 153-symbol window of the text so that every read keeps 150 bytes.
Times awry_count_device_edit at k = 0 .. 3 with CUDA events, alternating with awry_count_device_hamming at the same k
and with the exact awry_count_device (a warm-up, then REPS rounds of one 10-call window per arm; medians and spread).
Checks in the same run: the distance-0 counts equal the exact counts; a read with e planted edits has a start at
distance <= e for every k >= e; and the total within <= k of every read is at least its Hamming total.  Then cfg3
(1 M x 50 bp, q % 4 planted edits) at k = 2: device count beside Hamming, and the host-buffer locate.  The card name
and power limit are printed with the numbers."""
import argparse
import os
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

from awry_b200 import FmIndex, fm_index as f  # noqa: E402
from fixtures import pyfixture_gpu as fxg  # noqa: E402


def card():
    return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                          capture_output=True, text=True).stdout.strip().splitlines()[0]


def edited_reads(n, nq, L, seed, chunk=1_000_000):
    """nq reads of L bytes on the device, read q = a window of the text with q % 4 edits at distinct positions -> (flat
    uint8 reads, planted edits per read).  A deletion skips a text symbol, an insertion adds a random base, so every
    read is cut from a window of L + 3 symbols and stays L long."""
    W = L + 3
    out = torch.empty(nq * L, dtype=torch.uint8, device="cuda")
    acgt = torch.tensor(list(b"ACGT"), dtype=torch.uint8, device="cuda")
    g = torch.Generator(device="cuda").manual_seed(seed)
    win = torch.empty(chunk * W, dtype=torch.uint8, device="cuda")
    i = torch.arange(L, device="cuda")
    for c0 in range(0, nq, chunk):
        m = min(chunk, nq - c0)
        fxg.gen_queries_device(0, n, 3, m, W, seed + c0, win.data_ptr())
        q = torch.arange(c0, c0 + m, device="cuda")
        e = q % 4
        p0 = torch.randint(0, L, (m,), device="cuda", generator=g)
        step = torch.randint(1, L // 4, (m,), device="cuda", generator=g)
        shift = torch.zeros((m, L), dtype=torch.int64, device="cuda")   # source = i + n_ins + dels <= i - ins before i
        ins_at = torch.zeros((m, L), dtype=torch.bool, device="cuda")
        sub_at = torch.zeros((m, L), dtype=torch.bool, device="cuda")
        n_ins = torch.zeros(m, dtype=torch.int64, device="cuda")
        for j in range(3):
            live = e > j
            pos = (p0 + j * step) % L
            kind = (q // 4 + j) % 3
            hit = (i[None, :] >= pos[:, None]) & live[:, None]
            shift += (hit & (kind == 2)[:, None]).long()                     # deletion: later symbols come one further
            after = (i[None, :] > pos[:, None]) & live[:, None] & (kind == 1)[:, None]
            shift -= after.long()                                            # insertion: later symbols one closer
            n_ins += (live & (kind == 1)).long()
            ins_at |= (i[None, :] == pos[:, None]) & (live & (kind == 1))[:, None]
            sub_at |= (i[None, :] == pos[:, None]) & (live & (kind == 0))[:, None]
        src = i[None, :] + n_ins[:, None] + shift
        w = win[: m * W].view(m, W)
        r = torch.gather(w, 1, src.clamp(0, W - 1))
        rnd = acgt[torch.randint(0, 4, (m, L), device="cuda", generator=g)]
        r = torch.where(ins_at, rnd, r)
        lut = torch.zeros(256, dtype=torch.int64, device="cuda")
        for k, c in enumerate(b"ACGT"):
            lut[c] = k
        changed = acgt[(lut[r.long()] + torch.randint(1, 4, (m, L), device="cuda", generator=g)) % 4]
        r = torch.where(sub_at, changed, r)
        out[c0 * L:(c0 + m) * L] = r.reshape(-1)
    return out, torch.arange(nq, device="cuda") % 4


def time_calls(fn, n=10):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n


def alternate(arms, reps, n=10):
    """a warm-up of every arm, then REPS rounds of one n-call window per arm -> (median ms, spread) per arm"""
    for fn in arms.values():
        fn()
        fn()
    torch.cuda.synchronize()
    ms = {name: [] for name in arms}
    for _ in range(reps):
        for name, fn in arms.items():
            ms[name].append(time_calls(fn, n))
    return {k: statistics.median(v) for k, v in ms.items()}, {k: max(v) - min(v) for k, v in ms.items()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=3_100_000_000)
    ap.add_argument("--nq", type=int, default=10_000_000)
    ap.add_argument("--reps", type=int, default=5)
    a = ap.parse_args()
    print(card(), flush=True)
    st = torch.cuda.current_stream().cuda_stream
    L, nq = 150, a.nq
    t0 = time.time()
    parts, _ = fxg.build_parts(0, a.n, 3, ratio=8, kmer_len=13)
    ix = FmIndex.from_parts(parts.alphabet, parts.ratio, parts.bwt_len, parts.kmer_len, parts.blocks, parts.prefix_sums,
                            parts.sa_words)
    del parts
    d, m = edited_reads(a.n, nq, L, 5)
    off = torch.arange(0, nq + 1, dtype=torch.int64, device="cuda") * L
    print(f"index of {a.n} symbols and {nq} reads ready in {time.time() - t0:.1f} s", flush=True)
    exact = torch.zeros(nq, dtype=torch.int64, device="cuda")
    ham = {k: torch.zeros((nq, k + 1), dtype=torch.int64, device="cuda") for k in range(4)}
    ed = {k: torch.zeros((nq, k + 1), dtype=torch.int64, device="cuda") for k in range(4)}
    arms = {"exact (awry_count_device)": lambda: ix.count_device(d.data_ptr(), off.data_ptr(), nq, exact.data_ptr(), st)}
    for k in range(4):
        arms[f"k = {k} Hamming (awry_count_device_hamming)"] = \
            lambda k=k: ix.count_hamming_device(d.data_ptr(), off.data_ptr(), nq, k, ham[k].data_ptr(), st)
        arms[f"k = {k} edit (awry_count_device_edit)"] = \
            lambda k=k: ix.count_edit_device(d.data_ptr(), off.data_ptr(), nq, k, ed[k].data_ptr(), st)
    med, spread = alternate(arms, a.reps)
    ix.device_check(st)
    print(f"{nq / 1e6:.0f} M x {L}-bp device-resident reads, read q with q % 4 planted edits (substitution, insertion, "
          f"deletion in turn); median of {a.reps} alternating windows of 10 calls after a warm-up (spread = max - min):",
          flush=True)
    for name in arms:
        print(f"  {name}: {med[name]:.3f} ms (spread {spread[name]:.3f})", flush=True)
    for k in range(4):
        same0 = bool(torch.equal(ed[k][:, 0], exact))
        found = ed[k].sum(dim=1) > 0
        ok = bool(found[m <= k].all())
        ge = bool((ed[k].sum(dim=1) >= ham[k].sum(dim=1)).all())
        hfound = float((ham[k].sum(dim=1) > 0)[m <= k].double().mean())
        ratio = med[f"k = {k} edit (awry_count_device_edit)"] / med[f"k = {k} Hamming (awry_count_device_hamming)"]
        print(f"k = {k}: edit / Hamming = {ratio:.2f}; distance-0 counts == exact counts: {same0}; reads with <= k "
              f"planted edits have a start at distance <= k: {ok} (Hamming finds {hfound:.3f} of them); per-read total "
              f">= Hamming total: {ge}; starts per read by distance "
              f"{[round(float(ed[k][:, dd].double().mean()), 3) for dd in range(k + 1)]}", flush=True)
    # per-stage split at k = 3 (profiling adds synchronisations: calls of their own)
    for name, fn in (("Hamming", ix.count_hamming_device), ("edit", ix.count_edit_device)):
        f.profile_enable(True)
        f.profile_reset()
        for _ in range(3):
            fn(d.data_ptr(), off.data_ptr(), nq, 3, ed[3].data_ptr(), st)
        torch.cuda.synchronize()
        p = f.profile_get()
        f.profile_enable(False)
        print(f"k = 3 {name} per call: piece search {p['search_ms'] / 3:.2f} ms, verification {p['walk_ms'] / 3:.2f} ms, "
              f"packing {p['pack_ms'] / 3:.2f} ms", flush=True)
    del d, ham, ed
    torch.cuda.empty_cache()
    # cfg3: 1 M x 50-bp reads, q % 4 planted edits, k = 2
    nq3, L3 = 1_000_000, 50
    d3, _ = edited_reads(a.n, nq3, L3, 7)
    off3 = torch.arange(0, nq3 + 1, dtype=torch.int64, device="cuda") * L3
    c_h = torch.zeros((nq3, 3), dtype=torch.int64, device="cuda")
    c_e = torch.zeros((nq3, 3), dtype=torch.int64, device="cuda")
    med3, _ = alternate({
        "hamming": lambda: ix.count_hamming_device(d3.data_ptr(), off3.data_ptr(), nq3, 2, c_h.data_ptr(), st),
        "edit": lambda: ix.count_edit_device(d3.data_ptr(), off3.data_ptr(), nq3, 2, c_e.data_ptr(), st)}, a.reps)
    qb3, qo3 = d3.cpu().numpy(), np.arange(nq3 + 1, dtype=np.uint64) * np.uint64(L3)
    tl = {}
    for name, fn, cap in (("hamming", ix.locate_hamming_packed, int(c_h.sum()) + 1),
                          ("edit", ix.locate_edit_packed, int(c_e.sum()) + 1)):
        fn(qb3, qo3, 2, capacity=cap)
        t0 = time.time()
        _, hits, _ = fn(qb3, qo3, 2, capacity=cap)
        tl[name] = (time.time() - t0, len(hits))
    print(f"cfg3 (1 M x 50 bp, q % 4 planted edits, k = 2): device count {med3['edit']:.3f} ms edit, "
          f"{med3['hamming']:.3f} ms Hamming; host-buffer locate {tl['edit'][0] * 1e3:.1f} ms edit ({tl['edit'][1]} hits; "
          f"counts sum == hits: {int(c_e.sum()) == tl['edit'][1]}), {tl['hamming'][0] * 1e3:.1f} ms Hamming "
          f"({tl['hamming'][1]} hits)", flush=True)


if __name__ == "__main__":
    main()
