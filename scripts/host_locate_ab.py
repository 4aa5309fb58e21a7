"""A/B of the host-buffer approximate locates (awry_locate_batch_{hamming,edit}[_strands], awry_locate_batch_edit_loci)
between this tree's library and another build of it, normally the parent commit's:

    git worktree add /tmp/parent HEAD~1 && make -C /tmp/parent/awry_b200/csrc
    python scripts/host_locate_ab.py --other /tmp/parent/awry_b200/libawry_b200.so

Both libraries are loaded into one process (the other one through AWRY_B200_LIB), each with its own copy of every
index; the Python wrappers of this tree serve both, since the C signatures are the same.  Per workload: a warm-up call
of each library, whose outputs (hit_off, hits, distances) must be identical, then REPS rounds of one window of N calls
per library, the order of the two swapped every round.  The calls return to the host, so a host clock around them
measures whole calls.  Medians and spread (max - min) per library.  Then one profiled call per library splits its time
into the library's own spans: packing (reads and pieces), the exact search of the pieces and the verification passes;
the rest is sorting, compaction, copies and synchronisations.

Workloads:
- cfg5: the first 10 k reads of hamming_probe.py's cfg5 (1 Gbp repeat-rich text, up to ~10^4 hits per read), k = 2,
  Hamming and edit.
- cfg3: the 3.1 Gbp synthetic index of hamming_probe.py, 1 M x 50-bp reads with q % 4 planted edits (the reads of
  approx_locate_probe.py's cfg3: substitutions for Hamming, edits for edit distance), k = 2: Hamming and edit on one
  strand and both, and the edit loci on one strand and both; on both strands every odd read is reverse-complemented.
- The same index, 1 M x 150-bp reads (q % 4 planted edits), k = 0 .. 3, Hamming and edit, one strand.
The card name and power limit are printed with the numbers."""
import argparse
import os
import statistics
import sys
import time
from types import SimpleNamespace

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))
import torch  # noqa: E402

from approx_locate_probe import reads  # noqa: E402
from awry_b200 import FmIndex, fm_index as f  # noqa: E402
from fixtures import pyfixture_gpu as fxg, repeats  # noqa: E402
from hamming_probe import card, reverse_complement_rows  # noqa: E402


def load(path):
    """the library at `path`, loaded next to any other (fm_index keeps one current library: f._LIB)"""
    os.environ["AWRY_B200_LIB"] = path
    f._LIB = None
    lib = f.native()
    del os.environ["AWRY_B200_LIB"]
    return lib


class Pair:
    """one index per library, built from the same parts"""

    def __init__(self, libs, parts):
        self.libs, self.ix = libs, {}
        for name, lib in libs.items():
            f._LIB = lib
            self.ix[name] = FmIndex.from_parts(parts.alphabet, parts.ratio, parts.bwt_len, parts.kmer_len, parts.blocks,
                                               parts.prefix_sums, parts.sa_words)

    def call(self, name, method, *args, **kw):
        f._LIB = self.libs[name]
        return getattr(self.ix[name], method)(*args, **kw)

    def close(self):
        for name, ix in self.ix.items():
            f._LIB = self.libs[name]
            ix.close()


def ab(pair, label, method, qb, qo, k, reps, n, **kw):
    """warm-up and output check, then alternating timed windows and one profiled call per library -> one line each"""
    out = {name: pair.call(name, method, qb, qo, k, **kw) for name in pair.libs}
    a, b = out.values()
    same = all(np.array_equal(x, y) for x, y in zip(a, b))
    total = len(a[1])
    del out, a, b
    kw = dict(kw, capacity=total + 1)
    ms = {name: [] for name in pair.libs}
    names = list(pair.libs)
    for r in range(reps):
        for name in (names if r % 2 == 0 else names[::-1]):
            t0 = time.perf_counter()
            for _ in range(n):
                got = pair.call(name, method, qb, qo, k, **kw)
            ms[name].append((time.perf_counter() - t0) * 1e3 / n)
            assert len(got[1]) == total, (label, name, len(got[1]), total)
            del got
    med = {name: statistics.median(v) for name, v in ms.items()}
    print(f"{label}: {total} hits, outputs identical: {same}", flush=True)
    for name in names:
        f._LIB = pair.libs[name]
        f.profile_enable(True)
        f.profile_reset()
        t0 = time.perf_counter()
        pair.call(name, method, qb, qo, k, **kw)
        t = (time.perf_counter() - t0) * 1e3
        p = f.profile_get()
        f.profile_enable(False)
        print(f"  {name:6s} {med[name]:9.2f} ms (spread {max(ms[name]) - min(ms[name]):.2f}, median of {reps} windows of "
              f"{n}); one profiled call {t:.2f} ms: packing {p['pack_ms']:.2f}, piece search {p['search_ms']:.2f}, "
              f"verification {p['walk_ms']:.2f} ms in {p['walk_launches']} launches, other {t - p['pack_ms'] - p['search_ms'] - p['walk_ms']:.2f} ms; "
              f"d2h {p['d2h_bytes'] / 1e6:.1f} MB", flush=True)
    print(f"  this / other = {med['this'] / med['other']:.3f}", flush=True)
    return same


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--other", required=True, help="the other build's libawry_b200.so (e.g. the parent commit's)")
    ap.add_argument("--n", type=int, default=3_100_000_000)
    ap.add_argument("--cfg5-n", type=int, default=1_000_000_000)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--cfg5-reps", type=int, default=3)
    a = ap.parse_args()
    print(card(), flush=True)
    this = os.path.join(os.path.dirname(os.path.abspath(f.__file__)), "libawry_b200.so")
    libs = {"other": load(os.path.abspath(a.other)), "this": load(this)}
    print(f"other = {os.path.relpath(a.other, ROOT)}, this = {os.path.relpath(this, ROOT)}", flush=True)
    ok = True
    # cfg5: hamming_probe.py's repeat-rich text and reads, the first 10 k reads
    n5 = a.cfg5_n
    scale = n5 / 1e9
    fams = ((300, int(100_000 * scale) + 10, 0.15), (6000, int(20_000 * scale) + 5, 0.15))
    text, regions = repeats.repeat_rich_text(n5, seed=8, tandem_arrays=max(4, int(40 * scale)), families=fams)
    parts5, _ = fxg.build_parts(0, n5, 0, ratio=32, kmer_len=13, host_text=text)
    qb5, qo5 = repeats.repeat_queries(text, regions, 1_000_000, 50, seed=9)
    del text
    pair = Pair(libs, parts5)
    del parts5
    nl = 10_000
    for metric in ("hamming", "edit"):
        ok &= ab(pair, f"cfg5 ({n5 / 1e9:.2f} Gbp repeat-rich, first {nl} reads x 50 bp, k = 2) {metric} one strand",
                 f"locate_{metric}_packed", qb5[: nl * 50], qo5[: nl + 1], 2, a.cfg5_reps, 1)
    pair.close()
    torch.cuda.empty_cache()
    t0 = time.time()
    parts, _ = fxg.build_parts(0, a.n, 3, ratio=8, kmer_len=13)
    pair = Pair(libs, parts)
    del parts
    print(f"two indexes of {a.n} symbols ready in {time.time() - t0:.1f} s", flush=True)
    g = SimpleNamespace(n=a.n)
    # cfg3
    nq, L = 1_000_000, 50
    for metric in ("hamming", "edit"):
        d, _, _ = reads(g, metric, nq, L, 7)
        for strands in (False, True):
            if strands:
                reverse_complement_rows(d, nq, L, torch.arange(nq, device="cuda") % 2 == 1)
            qb, qo = d.cpu().numpy(), np.arange(nq + 1, dtype=np.uint64) * np.uint64(L)
            s = "_strands" if strands else ""
            side = "both strands" if strands else "one strand"
            ok &= ab(pair, f"cfg3 (1 M x 50 bp, k = 2) {metric} {side}", f"locate_{metric}{s}_packed", qb, qo, 2, a.reps, 3)
            if metric == "edit":
                ok &= ab(pair, f"cfg3 (1 M x 50 bp, k = 2) edit loci {side}", "locate_edit_loci_packed", qb, qo, 2, a.reps,
                         3, strands=strands)
        del d
    # 1 M x 150 bp, k = 0 .. 3, one strand
    nq, L = 1_000_000, 150
    for metric in ("hamming", "edit"):
        d, _, _ = reads(g, metric, nq, L, 4 if metric == "hamming" else 5)
        qb, qo = d.cpu().numpy(), np.arange(nq + 1, dtype=np.uint64) * np.uint64(L)
        del d
        for k in range(4):
            ok &= ab(pair, f"1 M x 150 bp on {a.n / 1e9:.1f} Gbp, k = {k}, {metric} one strand", f"locate_{metric}_packed",
                     qb, qo, k, a.reps, 1)
    pair.close()
    print(f"all outputs identical: {ok}", flush=True)
    print(card(), flush=True)
    return 0 if ok else 1


if __name__ == "__main__":
    sys.exit(main())
