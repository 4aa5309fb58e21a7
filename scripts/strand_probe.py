"""Cost of searching both strands, on the bench workload (bench.py's index and reads: 10 M x 150-bp device-resident
reads against the 3.1 Gbp synthetic text, k = 13, SA ratio 8).

  single:  awry_count_device (the strand the index holds)
  strands: awry_count_device_strands with the strand flavour of the ASCII wave kernel
  generic: awry_count_device_strands with AWRY_B200_STRAND_WAVE=0 (pack_kernel + strand_words_kernel + search)

The arms alternate within one process, REPS times, each a window of STEPS back-to-back calls timed with CUDA events
after a warm-up.  Twice: on the bench reads (all from the indexed strand), and on a mixed set in which every odd read
is reverse-complemented on the device.  Checks on the mixed set: every read is found on its own strand (forward reads
in slot 2q, complemented ones in slot 2q + 1), strand-0 counts equal awry_count_device's, and both strand arms agree.
Then cfg3 locate (1 M x 50-bp reads, same index): awry_locate_device against awry_locate_device_strands (both
routes), with the same checks on the hit totals.  Card name and power limit are printed with the numbers.
Usage: python scripts/strand_probe.py [--reps 7 --steps 10]"""
import argparse
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
os.environ.setdefault("AWRY_B200_LEAN_SA", "1")   # the bench index carries it too
import torch  # noqa: E402

import bench  # noqa: E402
from awry_b200 import FmIndex  # noqa: E402
from fixtures import pyfixture_gpu as fxg  # noqa: E402


def reverse_complement_rows(d_q, nq, L, rows):
    """reads `rows` (a bool mask over nq) of the flat byte buffer d_q replaced by their reverse complements"""
    lut = torch.arange(256, dtype=torch.uint8, device="cuda")
    for a, b in (b"AT", b"TA", b"CG", b"GC"):
        lut[a] = b
    m = d_q.view(nq, L)
    m[rows] = lut[m[rows].flip(1).long()]
    return d_q


def timed(fn, env, steps):
    os.environ["AWRY_B200_STRAND_WAVE"] = env
    for _ in range(3):
        fn()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


def compare(title, arms, reps, steps):
    ms = {name: [] for name, _, _ in arms}
    for _ in range(reps):
        for name, fn, env in arms:
            ms[name].append(timed(fn, env, steps))
    print(title)
    for name, _, _ in arms:
        v = ms[name]
        print(f"  {name:8s} ms/call min {min(v):.3f} median {statistics.median(v):.3f} spread {max(v) - min(v):.3f}"
              f"   windows {' '.join(f'{x:.3f}' for x in v)}")
    base = statistics.median(ms[arms[0][0]])
    for name, _, _ in arms[1:]:
        print(f"  {name} / {arms[0][0]}: {statistics.median(ms[name]) / base:.3f}")
    if len(arms) == 3:
        print(f"  {arms[1][0]} vs {arms[2][0]}: {100 * (1 - statistics.median(ms[arms[1][0]]) / statistics.median(ms[arms[2][0]])):.1f} % less time")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--text-len", type=int, default=3_100_000_000)
    ap.add_argument("--reads", type=int, default=10_000_000)
    ap.add_argument("--read-len", type=int, default=150)
    ap.add_argument("--locate-reads", type=int, default=1_000_000)
    ap.add_argument("--locate-len", type=int, default=50)
    a = ap.parse_args()
    print(subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip(), flush=True)
    parts, _ = fxg.build_parts(0, a.text_len, bench.TEXT_SEED, ratio=8, kmer_len=13)
    ix = FmIndex.from_parts(parts.alphabet, parts.ratio, parts.bwt_len, parts.kmer_len, parts.blocks, parts.prefix_sums,
                            parts.sa_words)
    st = torch.cuda.current_stream().cuda_stream
    nq, L = a.reads, a.read_len
    d_off = torch.arange(0, nq + 1, dtype=torch.int64, device="cuda") * L
    d_c1 = torch.zeros(nq, dtype=torch.int64, device="cuda")
    d_c2 = torch.zeros(2 * nq, dtype=torch.int64, device="cuda")
    odd = torch.arange(nq, device="cuda") % 2 == 1
    for label, mixed in (("bench reads (all on the indexed strand)", False),
                         ("mixed: every odd read reverse-complemented", True)):
        d_q = bench.device_reads(fxg, 0, a.text_len, bench.TEXT_SEED, nq, L, bench.QUERY_SEED)
        if mixed:
            reverse_complement_rows(d_q, nq, L, odd)
        single = lambda: ix.count_device(d_q.data_ptr(), d_off.data_ptr(), nq, d_c1.data_ptr(), st)  # noqa: E731
        both = lambda: ix.count_strands_device(d_q.data_ptr(), d_off.data_ptr(), nq, d_c2.data_ptr(), st)  # noqa: E731
        single()
        res = {}
        for env in ("1", "0"):
            os.environ["AWRY_B200_STRAND_WAVE"] = env
            both()
            ix.device_check(st)
            res[env] = d_c2.clone().view(nq, 2)
        ix.device_check(st)
        c1 = d_c1.clone()
        r = res["1"]
        fwd_ok = bool((r[~odd, 0] >= 1).all()) if mixed else bool((r[:, 0] >= 1).all())
        rev_ok = bool((r[odd, 1] >= 1).all()) if mixed else True
        print(f"{label}: routes identical {bool(torch.equal(res['1'], res['0']))}; strand 0 == awry_count_device "
              f"{bool(torch.equal(r[:, 0], c1))}; forward reads found on strand 0 {fwd_ok}; complemented reads found "
              f"on strand 1 {rev_ok}; reads with a reverse-strand hit {int((r[:, 1] > 0).sum())} of {nq}", flush=True)
        compare(f"awry_count_device vs awry_count_device_strands, {nq} x {L}-bp reads, {a.text_len}-bp text, {label}; "
                f"{a.reps} alternating windows of {a.steps} calls",
                [("single", single, "1"), ("strands", both, "1"), ("generic", both, "0")], a.reps, a.steps)
        del d_q
    # cfg3 locate
    nl, ll = a.locate_reads, a.locate_len
    d_q = bench.device_reads(fxg, 0, a.text_len, bench.TEXT_SEED, nl, ll, bench.QUERY_SEED + 1)
    reverse_complement_rows(d_q, nl, ll, torch.arange(nl, device="cuda") % 2 == 1)
    d_lo = torch.arange(0, nl + 1, dtype=torch.int64, device="cuda") * ll
    d_h1 = torch.zeros(nl + 1, dtype=torch.int64, device="cuda")
    d_h2 = torch.zeros(2 * nl + 1, dtype=torch.int64, device="cuda")
    totals = {}

    def loc1():
        p, n = ix.locate_device(d_q.data_ptr(), d_lo.data_ptr(), nl, d_h1.data_ptr(), stream=st)
        ix.device_free(p)
        totals["single"] = n

    def loc2():
        p, n = ix.locate_strands_device(d_q.data_ptr(), d_lo.data_ptr(), nl, d_h2.data_ptr(), stream=st)
        ix.device_free(p)
        totals["strands" + os.environ["AWRY_B200_STRAND_WAVE"]] = n

    compare(f"cfg3 locate: awry_locate_device vs awry_locate_device_strands, {nl} x {ll}-bp reads (odd ones "
            f"reverse-complemented), BWT order; {a.reps} alternating windows of {a.steps} calls",
            [("single", loc1, "1"), ("strands", loc2, "1"), ("generic", loc2, "0")], a.reps, a.steps)
    ix.device_check(st)
    print(f"cfg3 hit totals: single {totals['single']}, strands {totals['strands1']}, generic {totals['strands0']}")
    ix.close()


if __name__ == "__main__":
    main()
