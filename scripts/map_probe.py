"""Read mapping at full size (awry_map_device) against the locate it replaces.

Workload: the 3.1 Gbp synthetic index of scripts/hamming_probe.py and its 10 M x 150-bp device-resident reads (DESIGN.md
§1e): read q carries q % 4 planted substitutions (Hamming) or substitutions, insertions and deletions (edit, as
edit_probe.py), and every odd read is reverse-complemented.  Both strands.  For each metric and k = 0 .. 3 it times, in
one alternating run with CUDA events (a warm-up, then REPS rounds of one 10-call window per arm; medians and spread =
max - min), the map call without and with alignments against the locate a mapper would otherwise start from:
awry_locate_device_hamming_strands, or awry_locate_device_edit_loci with strands = 1 (outputs freed after each call).
Reported with the times: the keys placed and sorted under the bound (each read's best distance + 1) against the
unbounded hit total, from the device counts.  Checked in the same run: on the first SAMPLE reads the device records and
alignments equal the host call's and the Python reference (tests/test_map_abi.py: ref_map) applied to the host locate's
hits; every read with at most k planted edits maps to its origin strand within L of its origin, at a distance no larger
than its edits.  The card name and power limit are printed with the numbers."""
import argparse
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))
sys.path.insert(0, os.path.join(ROOT, "tests"))
import torch  # noqa: E402

from approx_locate_probe import reads  # noqa: E402
from awry_b200 import FmIndex  # noqa: E402
from awry_b200 import fm_index as f  # noqa: E402
from edit_probe import alternate  # noqa: E402
from fixtures import pyfixture_gpu as fxg  # noqa: E402
from hamming_probe import card, reverse_complement_rows  # noqa: E402
from test_map_abi import M64, ref_map  # noqa: E402


def bounded_keys(counts, nq):
    """(keys under the bound, unbounded hits) from the device counts ((2 nq) x (k+1)), as the bound kernel sums them"""
    k = counts.shape[1] - 1
    c = counts.view(nq, 2, k + 1)
    any_d = (c.sum(dim=1) > 0)
    best = torch.where(any_d.any(dim=1), any_d.to(torch.int8).argmax(dim=1), torch.full((nq,), -1, device="cuda"))
    lim = torch.where(best >= 0, torch.clamp(best + 1, max=k), torch.full_like(best, -1))
    d = torch.arange(k + 1, device="cuda")
    keep = d[None, :] <= lim[:, None]
    return int((c.sum(dim=1) * keep).sum()), int(c.sum())


def checks(ix, metric, k, d, off, nq, L, planted, origin, sample, st):
    recs = torch.empty(nq * 32, dtype=torch.uint8, device="cuda")
    aln = torch.empty(nq * 44, dtype=torch.uint8, device="cuda")
    ix.map_device(d.data_ptr(), off.data_ptr(), nq, metric, k, recs.data_ptr(), aln.data_ptr(), stream=st)
    ix.device_check(st)
    torch.cuda.synchronize()
    r = recs.cpu().numpy().view(f.MAPPING_DTYPE)
    a = aln.cpu().numpy().view(f.ALIGNMENT_DTYPE)
    qb = d[: sample * L].cpu().numpy()
    qo = np.arange(sample + 1, dtype=np.uint64) * np.uint64(L)
    hr, ha = ix.map_packed(qb, qo, metric, k)
    host_ok = hr.tobytes() == r[:sample].tobytes() and ha.tobytes() == a[:sample].tobytes()
    if metric == "edit":
        hoff, hits, dist = ix.locate_edit_loci_packed(qb, qo, k, strands=True)
    else:
        hoff, hits, dist = ix.locate_hamming_strands_packed(qb, qo, k)
    qs = [bytes(qb[i * L:(i + 1) * L]) for i in range(sample)]
    ref = ref_map(hoff, hits[:, 1], dist, qs, k, True)     # (one record: the global start is local_pos)
    mapped = ref["start"] != np.uint64(M64)
    ref_ok = (np.array_equal(ref["start"][mapped], r["local_pos"][:sample][mapped])
              and all(np.array_equal(ref[x], r[x][:sample]) for x in ("n_best", "n_second", "distance", "strand",
                                                                       "mapq", "flags")))
    q = np.arange(nq)
    want = planted <= k
    near = ((r["flags"] == 0) & (r["strand"] == q % 2) & (np.abs(r["local_pos"].astype(np.int64) -
                                                                  origin.astype(np.int64)) <= L)
            & (r["distance"] <= planted))
    unique = (r["n_best"] == 1).sum()
    return (f"first {sample} reads: device == host call: {host_ok}, == ref_map on the host locate: {ref_ok}; reads "
            f"with <= k planted edits mapped to their origin strand within {L} at distance <= their edits: "
            f"{int(near[want].sum())} of {int(want.sum())}; mapped {int((r['flags'] == 0).sum())}, unique "
            f"{int(unique)}, mapq 37: {int((r['mapq'] == 37).sum())}")


def run(a, ix, st, nq, L, metric, seed):
    t0 = time.time()
    d, m, origin = reads(a, metric, nq, L, seed)
    planted = m.cpu().numpy().astype(np.int64) if torch.is_tensor(m) else np.asarray(m, np.int64)
    reverse_complement_rows(d, nq, L, torch.arange(nq, device="cuda") % 2 == 1)
    off = torch.arange(0, nq + 1, dtype=torch.int64, device="cuda") * L
    print(f"{metric}: {nq} reads ready in {time.time() - t0:.1f} s", flush=True)
    recs = torch.empty(nq * 32, dtype=torch.uint8, device="cuda")
    aln = torch.empty(nq * 44, dtype=torch.uint8, device="cuda")
    d_off = torch.zeros(2 * nq + 1, dtype=torch.int64, device="cuda")

    def locate(k):
        if metric == "edit":
            hp, dp, n = ix.locate_edit_loci_device(d.data_ptr(), off.data_ptr(), nq, k, d_off.data_ptr(), strands=True,
                                                   stream=st)
        else:
            hp, dp, n = ix.locate_hamming_strands_device(d.data_ptr(), off.data_ptr(), nq, k, d_off.data_ptr(),
                                                         stream=st)
        ix.device_free(hp)
        ix.device_free(dp)
        return n
    for k in range(4):
        arms = {
            "locate": lambda: locate(k),
            "map": lambda: ix.map_device(d.data_ptr(), off.data_ptr(), nq, metric, k, recs.data_ptr(), stream=st),
            "map + aln": lambda: ix.map_device(d.data_ptr(), off.data_ptr(), nq, metric, k, recs.data_ptr(),
                                               aln.data_ptr(), stream=st),
        }
        med, spread = alternate(arms, a.reps)
        ix.device_check(st)
        counts = torch.zeros((2 * nq, k + 1), dtype=torch.int64, device="cuda")
        count = ix.count_edit_strands_device if metric == "edit" else ix.count_hamming_strands_device
        count(d.data_ptr(), off.data_ptr(), nq, k, counts.data_ptr(), st)
        torch.cuda.synchronize()
        keys, starts = bounded_keys(counts, nq)
        n_loc = locate(k)
        print(f"{metric}, both strands, k = {k}, {nq / 1e6:g} M x {L}-bp device-resident reads; median of {a.reps} "
              f"alternating windows of 10 calls after a warm-up (spread = max - min):", flush=True)
        lo, mp, ma = med["locate"], med["map"], med["map + aln"]
        print(f"  locate-device {lo:.3f} ms (spread {spread['locate']:.3f}); map-device {mp:.3f} ms (spread "
              f"{spread['map']:.3f}), map / locate = {mp / lo:.3f}; map-device with alignments {ma:.3f} ms (spread "
              f"{spread['map + aln']:.3f}), / locate = {ma / lo:.3f}", flush=True)
        print(f"  keys placed and sorted: {keys} under the bound against {starts} unbounded "
              f"({'starts' if metric == 'edit' else 'windows'}; {starts / max(1, keys):.2f} x); the locate returns "
              f"{n_loc} {'loci' if metric == 'edit' else 'hits'}", flush=True)
        print("  " + checks(ix, metric, k, d, off, nq, L, planted, origin, a.sample, st), flush=True)
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
    run(a, ix, st, a.nq, 150, "hamming", 5)
    run(a, ix, st, a.nq, 150, "edit", 5)
    print(card(), flush=True)


if __name__ == "__main__":
    main()
