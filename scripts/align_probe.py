"""Alignment of located hits at full size (awry_align_device, DESIGN.md §1f).

Workload: the §1e workload of scripts/approx_locate_probe.py -- the 3.1 Gbp synthetic index and 10 M x 150-bp
device-resident reads with q % 4 planted edits (substitutions for Hamming, substitutions / insertions / deletions for
edit distance); on both strands every odd read is reverse-complemented.  For each metric, strand count and k = 0 .. 3 it
runs the locate-device call once, then times awry_align_device on its hits against that locate call (outputs freed
after each call), with CUDA events: a warm-up, then REPS rounds of one 10-call window per arm, arms alternating; medians
and spread (max - min).  Both calls are timed as whole calls (the locate synchronises inside; the align window ends in
a stream synchronisation).
Checks in the same run, for every hit: the alignment's distance and n_ops equal the locate call's distance; on the hits
of the first SAMPLE reads, copied to the host with the text they name, applying the ops to Q (rc(q) for a
reverse-strand hit) gives exactly text[s .. s+text_len).  The card name and power limit are printed with the numbers."""
import argparse
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))
import torch  # noqa: E402

from approx_locate_probe import calls, reads, to_torch  # noqa: E402
from awry_b200 import FmIndex  # noqa: E402
from awry_b200 import fm_index as f  # noqa: E402
from edit_probe import alternate  # noqa: E402
from fixtures import pyfixture_gpu as fxg  # noqa: E402
from hamming_probe import card, reverse_complement_rows  # noqa: E402

COMP = bytes.maketrans(b"ACGTN", b"TGCAN")


def replay(al, hits, off, d, text, L, sample, strands):
    """the ops of the first `sample` reads' hits turn Q into the window -> (hits checked, all good)"""
    per = 2 if strands else 1
    e = int(off[per * sample])
    pos = hits[:e, 1].cpu().numpy()
    span = L + 3
    idx = torch.from_numpy(pos.astype(np.int64)).cuda()[:, None] + torch.arange(span, device="cuda")[None, :]
    win = text[idx.clamp(max=text.numel() - 1)].cpu().numpy()
    qs = d[: sample * L].cpu().numpy().reshape(sample, L)
    a = al[:e]
    good = True
    for v in range(per * sample):
        q = qs[v // per].tobytes().upper()
        if strands and v % 2:
            q = q.translate(COMP)[::-1]
        for h in range(int(off[v]), int(off[v + 1])):
            got, at = bytearray(), 0
            for t in range(int(a[h]["n_ops"])):
                o = a[h]["ops"][t]
                op, qp = chr(o["op"]), int(o["qpos"])
                got += q[at:qp]
                if op in "XD":
                    got.append(int(o["text_sym"]))
                at = qp + (op != "D")
            got += q[at:]
            good &= bytes(got) == win[h, : int(a[h]["text_len"])].tobytes()
    return e, good


def bench(a, ix, metric, st, text):
    L, nq = 150, a.nq
    d, _, _ = reads(a, metric, nq, L, 4 if metric == "hamming" else 5)
    off = torch.arange(0, nq + 1, dtype=torch.int64, device="cuda") * L
    for strands in (False, True):
        if strands:
            reverse_complement_rows(d, nq, L, torch.arange(nq, device="cuda") % 2 == 1)
        per = 2 if strands else 1
        _, locate, _ = calls(ix, metric, strands)
        d_off = torch.zeros(per * nq + 1, dtype=torch.int64, device="cuda")
        print(f"{metric}, {'both strands' if strands else 'one strand'}, {nq / 1e6:.0f} M x {L}-bp device-resident reads; "
              f"median of {a.reps} alternating windows of 10 calls after a warm-up (spread = max - min):", flush=True)
        for k in range(4):
            hp, dp, n = locate(d.data_ptr(), off.data_ptr(), nq, k, d_off.data_ptr(), stream=st)
            d_out = torch.empty(max(1, n) * 44, dtype=torch.uint8, device="cuda")
            hit_off = d_off.clone()
            scratch = torch.zeros(per * nq + 1, dtype=torch.int64, device="cuda")

            def align():
                ix.align_hits_device(d.data_ptr(), off.data_ptr(), nq, metric, k, hit_off.data_ptr(), hp, n,
                                     d_out.data_ptr(), strands=strands, stream=st)
                torch.cuda.current_stream().synchronize()

            def loc():
                h2, d2, _ = locate(d.data_ptr(), off.data_ptr(), nq, k, scratch.data_ptr(), stream=st)
                ix.device_free(h2)
                ix.device_free(d2)
            med, spread = alternate({"align": align, "locate": loc}, a.reps)
            ix.device_check(st)
            al_t, lo_t = med["align"], med["locate"]
            # checks: every hit's distance; the sample's ops against the text
            torch.cuda.synchronize()
            al_dev = d_out[: n * 44].view(n, 44)
            dist = to_torch(dp, n, torch.uint8)[:, 0]
            dist_ok = bool(torch.equal(al_dev[:, 4], dist)) and bool(torch.equal(al_dev[:, 5], dist))
            hits = to_torch(hp, n, torch.int64, 2)
            al = al_dev.cpu().numpy().copy().view(f.ALIGNMENT_DTYPE)[:, 0]
            checked, ops_ok = replay(al, hits, hit_off.cpu().numpy(), d, text, L, a.sample, strands)
            ix.device_free(hp)
            ix.device_free(dp)
            print(f"  k = {k}: {n} hits; align-device {al_t:.3f} ms (spread {spread['align']:.3f}), "
                  f"{n / (al_t * 1e-3) / 1e9:.2f} G hits/s; locate-device {lo_t:.3f} ms (spread {spread['locate']:.3f}); "
                  f"align / locate = {al_t / lo_t:.3f}; every hit's distance and n_ops == the locate's: {dist_ok}; "
                  f"ops reproduce the window on the {checked} hits of the first {a.sample} reads: {ops_ok}", flush=True)
            del d_out
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
    text = torch.empty(a.n, dtype=torch.uint8, device="cuda")          # the same synthetic text, for the checks
    assert fxg.lib().fxg_gen_text_device(0, a.n, 3, text.data_ptr(), 0) == 0
    torch.cuda.synchronize()
    print(f"index of {a.n} symbols ready in {time.time() - t0:.1f} s", flush=True)
    for metric in ("hamming", "edit"):
        bench(a, ix, metric, st, text)
    print(card(), flush=True)


if __name__ == "__main__":
    main()
