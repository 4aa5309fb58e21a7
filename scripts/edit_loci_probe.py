"""Edit-distance search by locus at full size (awry_locate_device_edit_loci, awry_count_device_edit_loci).

Workload: the 3.1 Gbp synthetic index of scripts/hamming_probe.py and the 10 M x 150-bp device-resident reads of
edit_probe.py (read q with q % 4 planted substitutions, insertions and deletions; on both strands every odd read is
reverse-complemented), then cfg3 (1 M x 50 bp, the same planting).  For one strand and both and k = 1 .. 3 it times,
in one alternating run with CUDA events (a warm-up, then REPS rounds of one 10-call window per arm; medians and
spread = max - min), the plain edit locate-device call against the loci locate-device call (outputs freed after each
call), and the plain edit count-device call against the loci count-device call.  Every call synchronises inside, so a
window measures whole calls.
Reported with the times: the hit and locus totals and their ratio.  Checked in the same run: on the first SAMPLE reads
the device loci (offsets, hits, distances) equal the host call's, and every read with at most k planted edits has a
locus at distance <= its planted edits within L of its origin on its own strand.  The card name and power limit are
printed with the numbers."""
import argparse
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))
import torch  # noqa: E402

from approx_locate_probe import reads, to_torch  # noqa: E402
from awry_b200 import FmIndex  # noqa: E402
from edit_probe import alternate  # noqa: E402
from fixtures import pyfixture_gpu as fxg  # noqa: E402
from hamming_probe import card, reverse_complement_rows  # noqa: E402


def check(ix, strands, k, d, off, nq, L, m, origin, sample, st):
    """the checks of one (strands, k) on the reads of the timed run -> (locus total, one line)"""
    per = 2 if strands else 1
    d_off = torch.full((per * nq + 1,), -1, dtype=torch.int64, device="cuda")
    hp, dp, n = ix.locate_edit_loci_device(d.data_ptr(), off.data_ptr(), nq, k, d_off.data_ptr(), strands=strands,
                                           stream=st)
    ix.device_check(st)
    torch.cuda.synchronize()
    hits = to_torch(hp, n, torch.int64, 2)
    dist = to_torch(dp, n, torch.uint8)[:, 0]
    ix.device_free(hp)
    ix.device_free(dp)
    qb = d[: sample * L].cpu().numpy()
    qo = np.arange(sample + 1, dtype=np.uint64) * np.uint64(L)
    hoff, hhits, hd = ix.locate_edit_loci_packed(qb, qo, k, strands=strands, capacity=int(d_off[per * sample]) + 1)
    e = int(hoff[-1])
    sample_ok = (np.array_equal(hoff, d_off[: per * sample + 1].cpu().numpy().view(np.uint64))
                 and np.array_equal(hhits, hits[:e].cpu().numpy().view(np.uint64))
                 and np.array_equal(hd, dist[:e].cpu().numpy()))
    # a locus within L of the origin, on the read's own strand, at distance <= its planted edits (one record)
    v = torch.repeat_interleave(torch.arange(per * nq, device="cuda"), torch.diff(d_off))
    q = v // per
    own = (v % per) == (q % 2) if strands else torch.ones_like(q, dtype=torch.bool)
    org = torch.from_numpy(origin.view(np.int64)).cuda()
    mm = m.to(torch.int64) if torch.is_tensor(m) else torch.from_numpy(np.asarray(m, np.int64)).cuda()
    at = own & ((hits[:, 1] - org[q]).abs() <= L) & (hits[:, 0] == 0) & (dist.to(torch.int64) <= mm[q])
    found = torch.zeros(nq, dtype=torch.bool, device="cuda")
    found[q[at]] = True
    want = mm <= k
    return n, (f"first {sample} reads == host call: {sample_ok}; reads with <= k planted edits with a locus at distance "
               f"<= their edits within {L} of their origin on their own strand: {bool(found[want].all())} "
               f"({int(found[want].sum())} of {int(want.sum())})")


def run(a, ix, st, nq, L, seed, tag):
    t0 = time.time()
    d, m, origin = reads(a, "edit", nq, L, seed)
    off = torch.arange(0, nq + 1, dtype=torch.int64, device="cuda") * L
    print(f"{tag}: {nq} reads ready in {time.time() - t0:.1f} s", flush=True)
    for strands in (False, True):
        if strands:
            reverse_complement_rows(d, nq, L, torch.arange(nq, device="cuda") % 2 == 1)
        per = 2 if strands else 1
        counts = {k: torch.zeros((per * nq, k + 1), dtype=torch.int64, device="cuda") for k in range(1, 4)}
        d_off = torch.zeros(per * nq + 1, dtype=torch.int64, device="cuda")
        plain_count = ix.count_edit_strands_device if strands else ix.count_edit_device
        plain_locate = ix.locate_edit_strands_device if strands else ix.locate_edit_device

        def loc(k, loci):
            if loci:
                hp, dp, n = ix.locate_edit_loci_device(d.data_ptr(), off.data_ptr(), nq, k, d_off.data_ptr(),
                                                       strands=strands, stream=st)
            else:
                hp, dp, n = plain_locate(d.data_ptr(), off.data_ptr(), nq, k, d_off.data_ptr(), stream=st)
            ix.device_free(hp)
            ix.device_free(dp)
            return n
        arms = {}
        for k in range(1, 4):
            arms[f"k = {k} locate"] = lambda k=k: loc(k, False)
            arms[f"k = {k} loci locate"] = lambda k=k: loc(k, True)
            arms[f"k = {k} count"] = lambda k=k: plain_count(d.data_ptr(), off.data_ptr(), nq, k, counts[k].data_ptr(), st)
            arms[f"k = {k} loci count"] = lambda k=k: ix.count_edit_loci_device(
                d.data_ptr(), off.data_ptr(), nq, k, counts[k].data_ptr(), strands=strands, stream=st)
        med, spread = alternate(arms, a.reps)
        ix.device_check(st)
        print(f"{tag}, {'both strands' if strands else 'one strand'}, {nq / 1e6:g} M x {L}-bp device-resident reads; "
              f"median of {a.reps} alternating windows of 10 calls after a warm-up (spread = max - min):", flush=True)
        for k in range(1, 4):
            n_hits = loc(k, False)
            n_loci, line = check(ix, strands, k, d, off, nq, L, m, origin, a.sample, st)
            ix.count_edit_loci_device(d.data_ptr(), off.data_ptr(), nq, k, counts[k].data_ptr(), strands=strands,
                                      stream=st)
            torch.cuda.synchronize()
            counted = int(counts[k].sum())
            p, pl, c, cl = (med[f"k = {k} {x}"] for x in ("locate", "loci locate", "count", "loci count"))
            sp = {x: spread[f"k = {k} {x}"] for x in ("locate", "loci locate", "count", "loci count")}
            print(f"  k = {k}: locate-device {p:.3f} ms (spread {sp['locate']:.3f}), loci locate-device {pl:.3f} ms "
                  f"(spread {sp['loci locate']:.3f}), loci / plain = {pl / p:.3f}; count-device {c:.3f} ms (spread "
                  f"{sp['count']:.3f}), loci count-device {cl:.3f} ms (spread {sp['loci count']:.3f}), loci / plain = "
                  f"{cl / c:.3f}", flush=True)
            print(f"    {n_hits} hits, {n_loci} loci (hits / loci = {n_hits / max(1, n_loci):.2f}); loci count total == "
                  f"loci locate total: {counted == n_loci}; {line}", flush=True)
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
    run(a, ix, st, a.nq, 150, 5, "edit")
    run(a, ix, st, min(a.nq, 1_000_000), 50, 7, "cfg3")
    print(card(), flush=True)


if __name__ == "__main__":
    main()
