"""A/B of the two ways awry_count_device packs ASCII reads, on the bench workload (bench.py's index and reads: 10 M x
150-bp reads against the 3.1 Gbp synthetic text, k = 13, SA ratio 8).

  old: pack_kernel writes the 4-bit words, the wave kernel reads them back (AWRY_B200_ASCII_WAVE=0)
  new: the wave kernel stages each read into its ring straight from the ASCII bytes

The arms alternate within one process, REPS times, each a window of STEPS back-to-back calls timed with CUDA events
after a warm-up; the profile counters of one more window give the pack / search split.  Prints min, median and spread
(max - min) per arm, the new arm's gain, and whether both arms' counts are identical.  Card name and power limit are
printed with the numbers.  Usage: python scripts/ascii_wave_probe.py [--reps 7 --steps 10]"""
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
from awry_b200 import FmIndex, fm_index as f  # noqa: E402
from fixtures import pyfixture_gpu as fxg  # noqa: E402

ARMS = (("old", "0"), ("new", "1"))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--text-len", type=int, default=3_100_000_000)
    ap.add_argument("--reads", type=int, default=10_000_000)
    ap.add_argument("--read-len", type=int, default=150)
    a = ap.parse_args()
    print(subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip(), flush=True)
    parts, _ = fxg.build_parts(0, a.text_len, bench.TEXT_SEED, ratio=8, kmer_len=13)
    ix = FmIndex.from_parts(parts.alphabet, parts.ratio, parts.bwt_len, parts.kmer_len, parts.blocks, parts.prefix_sums,
                            parts.sa_words)
    nq, L = a.reads, a.read_len
    d_q = bench.device_reads(fxg, 0, a.text_len, bench.TEXT_SEED, nq, L, bench.QUERY_SEED)
    d_off = torch.arange(0, nq + 1, dtype=torch.int64, device="cuda") * L
    st = torch.cuda.current_stream().cuda_stream
    counts = {}
    for name, env in ARMS:
        os.environ["AWRY_B200_ASCII_WAVE"] = env
        d_c = torch.zeros(nq, dtype=torch.int64, device="cuda")
        ix.count_device(d_q.data_ptr(), d_off.data_ptr(), nq, d_c.data_ptr(), st)
        ix.device_check(st)
        counts[name] = d_c
    same = bool(torch.equal(counts["old"], counts["new"]))
    d_c = counts["new"]

    def window(env):
        os.environ["AWRY_B200_ASCII_WAVE"] = env
        for _ in range(3):
            ix.count_device(d_q.data_ptr(), d_off.data_ptr(), nq, d_c.data_ptr(), st)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        for _ in range(a.steps):
            ix.count_device(d_q.data_ptr(), d_off.data_ptr(), nq, d_c.data_ptr(), st)
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / a.steps

    ms = {name: [] for name, _ in ARMS}
    for _ in range(a.reps):
        for name, env in ARMS:
            ms[name].append(window(env))
    split = {}
    for name, env in ARMS:
        os.environ["AWRY_B200_ASCII_WAVE"] = env
        f.profile_enable(True)
        f.profile_reset()
        window(env)
        p = f.profile_get()
        f.profile_enable(False)
        n = max(1, p["search_launches"])
        split[name] = (p["pack_ms"] / n, p["search_ms"] / n)
    ix.device_check(st)
    print(f"awry_count_device, {nq} x {L}-bp reads, {a.text_len}-bp text; {a.reps} alternating windows of {a.steps} calls")
    for name, _ in ARMS:
        v = ms[name]
        print(f"{name}: ms/call min {min(v):.3f} median {statistics.median(v):.3f} spread {max(v) - min(v):.3f}   "
              f"pack {split[name][0]:.3f} ms + search {split[name][1]:.3f} ms per call (profile counters)   "
              f"windows {' '.join(f'{x:.3f}' for x in v)}")
    gain = 1 - statistics.median(ms["new"]) / statistics.median(ms["old"])
    print(f"new vs old: median {100 * gain:.1f} % less time per call; counts identical: {same}")
    ix.close()


if __name__ == "__main__":
    main()
