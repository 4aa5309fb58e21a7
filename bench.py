#!/usr/bin/env python
"""bench.py -- headline benchmark of the batched FM-index search path (BASELINE.json configs[1]):
parallel_count of 10 M synthetic 150-bp reads against a 3.1 Gbp synthetic DNA text, k = 13 seed
table, SA ratio 8.

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --gpus N --steps K ...   # the reference's CPU algorithm (oracle port)
    python bench.py ... --dump-outputs DIR                    # also writes the headline counts for comparing builds

One process per GPU (torchrun for N > 1); the index is replicated per GPU, every rank searches its
own 10 M-read batch (weak scaling), no collective on the data path.  A "step" is one pass of the hot
path over the rank's batch.  Rank 0 prints ONE JSON line.

`value`  = device-resident reads/s (CUDA events, max over ranks).
`e2e`    = the same metric through the C ABI from pinned HOST ASCII to host counts.  At N = 1 that is one
           awry_count_batch call per step; at N > 1 it is ONE awry_count_batch call per step over the
           N x 10 M reads of all ranks, issued by rank 0 on a handle with N replicas (the library's own
           multi-GPU path: fm_index.rs:455-487 is one call over one batch), the other ranks idle; the
           per-process figure (every rank calling with its own batch) is reported as `e2e_per_process`.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

# the bench index carries all three locate schemes (unsampled array, position-sampled array + walk blocks, the
# file's row samples) so that the locate legs can time each on the same handle; the count path does not read them
os.environ.setdefault("AWRY_B200_LEAN_SA", "1")

TEXT_SEED = 3          # BASELINE.md cfg2
QUERY_SEED = 4
ALG_BYTES_PER_BLOCK = 104   # SURVEY.md 8(d): 3 x 32 B planes + one 8-B milestone per rank-block access
DUMP_ROWS = 1 << 21         # --dump-outputs: 2 x 16 MB of float64 at most
DUMP_SEED = 5


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="awry_b200", choices=["awry_b200", "reference"])
    ap.add_argument("--text-len", type=int, default=3_100_000_000)
    ap.add_argument("--reads", type=int, default=10_000_000, help="reads per GPU per step")
    ap.add_argument("--read-len", type=int, default=150)
    ap.add_argument("--kmer", type=int, default=13)
    ap.add_argument("--sa-ratio", type=int, default=8)
    ap.add_argument("--cpu-sample", type=int, default=4_000_000, help="reads timed on the CPU oracle (rank 0, N=1)")
    ap.add_argument("--ref-reads-per-step", type=int, default=1_000_000)
    ap.add_argument("--locate-reads", type=int, default=1_000_000, help="cfg3: queries of the locate leg")
    ap.add_argument("--locate-len", type=int, default=50)
    ap.add_argument("--count-variant", type=int, default=0, choices=[0, 1],
                    help="0 = the library's default count path (one-row intervals finished in the text), 1 = backward "
                         "search to the last symbol for the headline leg too (ncu captures of that kernel)")
    ap.add_argument("--no-locate", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-secondary", action="store_true", help="skip the cfg4 (protein) and cfg5 (repeat-rich) legs")
    ap.add_argument("--no-inprocess", action="store_true", help="N > 1: skip rank 0's one-call-over-N-replicas leg")
    ap.add_argument("--cfg4-len", type=int, default=2_000_000_000)
    ap.add_argument("--cfg5-len", type=int, default=1_000_000_000)
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the counts of the headline leg's last step (rank 0's batch) to "
                         "DIR/counts.npy and the reads they belong to to DIR/count_rows.npy, both float64; batches above "
                         f"{DUMP_ROWS} reads are sampled with a fixed seed")
    a = ap.parse_args()
    if a.dump_outputs and a.impl != "awry_b200":
        ap.error("--dump-outputs writes the outputs of --impl awry_b200")
    return a


def dump_counts(out_dir, counts):
    """--dump-outputs: the per-read counts a caller of the headline path receives, as float64 (exact below 2**53).
    The same arguments give the same reads, so two builds can be compared file for file."""
    n = len(counts)
    rows = np.arange(n)
    if n > DUMP_ROWS:
        rows = np.sort(np.random.default_rng(DUMP_SEED).choice(n, DUMP_ROWS, replace=False))
    np.save(os.path.join(out_dir, "counts.npy"), counts[rows].astype(np.float64))
    np.save(os.path.join(out_dir, "count_rows.npy"), rows.astype(np.float64))


def dist_env():
    return int(os.environ.get("RANK", 0)), int(os.environ.get("LOCAL_RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe).  The sampler is
    started ahead of the region and `wait_ready()` returns once its first line has arrived; only samples whose
    timestamp falls inside [mark_begin(), mark_end()] are reported (all of them if none does)."""
    Q = ("timestamp,index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.proc = None
        self.lines = []
        self.t0 = self.t1 = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.gpu), "-lms", "50"], stdout=subprocess.PIPE, text=True)
            self.thr = threading.Thread(target=self._pump, daemon=True)
            self.thr.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append((time.time(), line.strip()))

    def wait_ready(self, timeout=3.0):
        t = time.time()
        while self.proc and not self.lines and time.time() - t < timeout:
            time.sleep(0.01)

    def mark_begin(self):
        self.t0 = time.time()

    def mark_end(self):
        self.t1 = time.time()

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.12)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]

        def parse(rows):
            sm, mx, reasons = [], [], set()
            for _, ln in rows:
                f = [x.strip() for x in ln.split(",")]
                if len(f) < 10:
                    continue
                try:
                    sm.append(float(f[2]))
                    mx.append(float(f[3]))
                except ValueError:
                    continue
                for name, v in zip(names, f[6:10]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            return sm, mx, reasons
        # a line is printed right after its sample is taken: arrival time ~ sample time
        inside = [r for r in self.lines if self.t0 is not None and self.t0 - 0.01 <= r[0] <= (self.t1 or 1e18) + 0.06]
        sm, mx, reasons = parse(inside if inside else self.lines)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "samples_in_timed_region": len(inside), "reasons": sorted(reasons)}


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs, stream copy)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md, 6.65 TB/s)"


def traffic_from_profiles(kernel, in_text=None):
    """DRAM bytes per launch of a kernel from the committed `ncu --set full` capture of this bench command
    (profiles/*_traffic.json, written by scripts/ncu_summary.py), or None.  `in_text`: the pair kernel exists
    with (last template argument 1) and without (0, or absent in captures older than the argument) the
    finish-in-the-text step."""
    import glob
    for path in sorted(glob.glob(os.path.join(ROOT, "profiles", "*_traffic.json"))):
        try:
            d = json.load(open(path))
        except Exception:
            continue
        name = str(d.get("kernel", ""))
        if not name.startswith(kernel) or not d.get("dram_bytes_per_launch"):
            continue
        if in_text is not None and name.rstrip().endswith(", 1>") != in_text:
            continue
        return d
    return None


def workload_name(a):
    return (f"parallel_count {a.reads} x {a.read_len}-bp reads vs {a.text_len}-bp synthetic DNA text, "
            f"k={a.kmer} seed table, SA ratio {a.sa_ratio}")


def config_of(a):
    """identical in both arms (the driver compares them)"""
    return {"workload": workload_name(a), "reads_per_gpu_per_step": a.reads,
            "l2": "inputs larger than L2 (1.5 GB of reads per step; 4.1 GB pair blocks, 8.6 GB seed table, 12.4 GB suffix array, "
                  "1.55 GB text, all read at random)",
            "index": "replicated per GPU; ranks search disjoint batches; no collective on the data path"}


def build_host_index(a, device):
    """reference-layout index arrays in host memory (fixture; FmIndex::new stand-in)"""
    import torch
    if torch.cuda.is_available():
        from fixtures import pyfixture_gpu as fxg
        parts, phases = fxg.build_parts(0, a.text_len, TEXT_SEED, ratio=a.sa_ratio, kmer_len=a.kmer, device=device)
        return parts, phases
    from fixtures import pyfixture as fx
    text = fx.gen_text(0, a.text_len, TEXT_SEED)
    return fx.build_parts(text, 0, ratio=a.sa_ratio, kmer_len=a.kmer), {"total": None}


def device_reads(fxg, alphabet, text_len, text_seed, nq, L, qseed, mut_ppm=0):
    import torch
    d = torch.empty(nq * L, dtype=torch.uint8, device="cuda")
    fxg.gen_queries_device(alphabet, text_len, text_seed, nq, L, qseed, d.data_ptr(), mut_ppm=mut_ppm)
    return d


def query_positions(text_len, nq, L, qseed):
    """text position of synthetic read q (the generator of fixtures/fixture_gpu.cu, restated): the check that
    the index the CPU arm searches was built right does not go through the product library"""
    M = (1 << 64) - 1

    def mix64(z):
        z = (z + 0x9E3779B97F4A7C15) & M
        z = ((z ^ (z >> 30)) * 0xBF58476D1CE4E5B9) & M
        z = ((z ^ (z >> 27)) * 0x94D049BB133111EB) & M
        return z ^ (z >> 31)
    span = text_len - L + 1
    return [(mix64(mix64(qseed) ^ ((q * 0xD1342543DE82EF95) & M)) * span) >> 64 for q in range(nq)]


def check_index_by_known_positions(orc, a, qb, nq_check=512):
    """every synthetic read is text[p .. p+L) for a p the generator fixes: the oracle's locate on the index
    under test must report p among the read's hits (tests blocks, prefix sums and sampled SA together,
    independently of the library that built them)"""
    L = a.read_len
    pos = query_positions(a.text_len, nq_check, L, QUERY_SEED)
    qo = np.arange(nq_check + 1, dtype=np.uint64) * np.uint64(L)
    off, hits, _ = orc.locate_batch(qb[: nq_check * L], qo)
    for q in range(nq_check):
        if pos[q] not in set(int(x) for x in hits[int(off[q]):int(off[q + 1]), 1]):
            return False
    return True


def run_reference(a):
    """--impl reference: the reference's CPU search path (C port in oracle/, all host threads)"""
    rank, local_rank, world = dist_env()
    if rank != 0:
        return 0
    from oracle import pyoracle as po
    import torch
    if torch.cuda.is_available():
        torch.cuda.set_device(0)
    reduced = not torch.cuda.is_available()
    if reduced:
        a.text_len = min(a.text_len, 20_000_000)
    parts, _ = build_host_index(a, 0)
    orc = po.OracleIndex.from_parts(parts.alphabet, parts.ratio, parts.bwt_len, parts.kmer_len, parts.blocks,
                                    parts.prefix_sums, parts.sa_words)
    nq = a.ref_reads_per_step
    full = None
    if reduced:
        from fixtures import pyfixture as fx
        text = fx.gen_text(0, a.text_len, TEXT_SEED)
        qb, _, _ = fx.gen_substring_queries(text, nq, a.read_len, QUERY_SEED)
        index_ok = None
    else:
        from fixtures import pyfixture_gpu as fxg
        qb_all = device_reads(fxg, 0, a.text_len, TEXT_SEED, a.reads, a.read_len, QUERY_SEED).cpu().numpy()
        qb = qb_all[: nq * a.read_len]
        # the index comes from the GPU builder (no CPU suffix sort handles 3.1 Gbp in minutes): verify it
        # without the product library before timing anything on it
        index_ok = check_index_by_known_positions(orc, a, qb_all)
    qo = np.arange(nq + 1, dtype=np.uint64) * np.uint64(a.read_len)
    cores = po.lib().awo_hw_threads()
    for _ in range(a.warmup):
        orc.count_batch(qb, qo)
    t0 = time.perf_counter()
    for _ in range(a.steps):
        counts, st = orc.count_batch(qb, qo)
    dt = time.perf_counter() - t0
    value = nq * a.steps / dt
    if not reduced:
        # the whole 10 M-read batch once, so the sample's rate can be checked against the full workload
        qo_all = np.arange(a.reads + 1, dtype=np.uint64) * np.uint64(a.read_len)
        t1 = time.perf_counter()
        c_all, _ = orc.count_batch(qb_all, qo_all)
        dt_all = time.perf_counter() - t1
        full = {"reads": a.reads, "seconds": dt_all, "reads_per_s": a.reads / dt_all, "every_read_found": bool(c_all.min() >= 1)}
    sample = (f"{nq} reads per step (bounded sample of the {a.reads}-read batch; the full batch is timed once in "
              f"`full_batch_once`), plain backward search as the reference executes it (no table use, "
              f"kmer_lookup_table.rs:90-110), {cores} pthreads with dynamic chunking standing in for rayon")
    line = {
        "impl": "reference", "metric": "count queries/s", "value": value, "unit": "reads/s", "n_gpus": a.gpus,
        "steps": a.steps, "warmup": a.warmup, "ms_per_step": dt / a.steps * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "u64", "data": "synthetic",
        "config": config_of(a), "reads_per_step": nq, "reduced_text": reduced,
        "cpu_baseline": {"value": value, "unit": "reads/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": "reads/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "full_batch_once": full,
        "index_check": {"located_known_positions": index_ok,
                        "how": "the oracle's locate of 512 reads reports the text position each read was cut from "
                               "(positions restated from the generator's seed in bench.py); the index arrays "
                               "come from the GPU builder, the timed region is pure oracle/"},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)
    return 0


# ---------------------------------------------------------------------------------------------- legs

def timed_device_leg(torch, barrier, fn, steps, warmup=3):
    for _ in range(warmup):
        fn()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    barrier()
    return e0.elapsed_time(e1)


def pinned_like(torch, n, dtype):
    return torch.empty(n, dtype=dtype, pin_memory=True)


def secondary_cfg4(a, torch, f, fxg, po, stream, peak):
    """BASELINE cfg4: count + locate of 10 M 12-residue peptides vs a 2 G-residue protein text, k = 5"""
    from awry_b200 import FmIndex
    n, k, L, nq, nl = a.cfg4_len, 5, 12, 10_000_000, 1_000_000
    parts, _ = fxg.build_parts(1, n, 6, ratio=8, kmer_len=k)
    with FmIndex.from_parts(parts.alphabet, parts.ratio, parts.bwt_len, parts.kmer_len, parts.blocks,
                            parts.prefix_sums, parts.sa_words) as ix:
        d_q = device_reads(fxg, 1, n, 6, nq, L, 7)
        d_off = torch.arange(0, nq + 1, dtype=torch.int64, device="cuda") * L
        d_cnt = torch.zeros(nq, dtype=torch.int64, device="cuda")
        f.profile_enable(True)
        f.profile_reset()
        ms = timed_device_leg(torch, torch.cuda.synchronize,
                              lambda: ix.count_device(d_q.data_ptr(), d_off.data_ptr(), nq, d_cnt.data_ptr(), stream), a.steps)
        prof = f.profile_get()
        f.profile_enable(False)
        ix.device_check(stream)
        ns = 200_000
        orc = po.OracleIndex.from_parts(parts.alphabet, parts.ratio, parts.bwt_len, parts.kmer_len, parts.blocks,
                                        parts.prefix_sums, parts.sa_words)
        sb = d_q[: ns * L].cpu().numpy()
        so = np.arange(ns + 1, dtype=np.uint64) * np.uint64(L)
        t0 = time.perf_counter()
        want, st = orc.count_batch(sb, so)
        cpu_dt = time.perf_counter() - t0
        parity = bool(np.array_equal(want, d_cnt[:ns].cpu().numpy().view(np.uint64)))
        # steps per peptide: L - k seeded steps, one 128-B device block each; algorithmic bytes 168 B per
        # distinct reference block (5 x 32-B planes + one 8-B milestone, SURVEY 8(d))
        kernel_ms = prof["search_ms"] / max(1, prof["search_launches"])
        touches = st["seeded_touches"] / ns
        alg_bytes = nq * (L + 8 + 16 + 168 * touches)
        tr = traffic_from_profiles("search_amino")
        phys = tr["dram_bytes_per_launch"] if tr and nq == 10_000_000 else None
        # DRAM lines per launch from the ncu capture; without one: L - k block reads + offsets, packed words, seed entry, result
        requests = phys / 128 if phys else nq * ((L - k) + 4.5)
        # e2e through the C ABI from pinned host ASCII
        h_q = pinned_like(torch, nq * L, torch.uint8)
        h_q.copy_(d_q)
        h_off = pinned_like(torch, nq + 1, torch.int64)
        h_off.copy_(d_off)
        h_cnt = pinned_like(torch, nq, torch.int64)
        torch.cuda.synchronize()
        qb, qo, out = h_q.numpy(), h_off.numpy().view(np.uint64), h_cnt.numpy().view(np.uint64)
        for _ in range(2):
            ix.count_packed(qb, qo, out=out)
        t0 = time.perf_counter()
        for _ in range(a.steps):
            ix.count_packed(qb, qo, out=out)
        e2e_dt = (time.perf_counter() - t0) / a.steps
        # locate: 1 M peptides
        d_lq = device_reads(fxg, 1, n, 6, nl, L, 8)
        d_loff = torch.arange(0, nl + 1, dtype=torch.int64, device="cuda") * L
        d_hoff = torch.zeros(nl + 1, dtype=torch.int64, device="cuda")
        res = {}
        for variant in (1, 0):
            f.set_locate_variant(variant)
            try:
                def once():
                    ptr, nh = ix.locate_device(d_lq.data_ptr(), d_loff.data_ptr(), nl, d_hoff.data_ptr(), stream=stream)
                    ix.device_free(ptr)
                    return nh
                nh = once()
                lms = timed_device_leg(torch, torch.cuda.synchronize, once, a.steps, warmup=1) / a.steps
            finally:
                f.set_locate_variant(0)
            res[variant] = (lms, nh)
        out_d = {
            "workload": f"count + locate of {nq} x {L}-residue peptides vs {n}-residue synthetic protein text, k={k}, SA ratio 8 (cfg4)",
            "count_reads_per_s": nq * a.steps / (ms * 1e-3), "count_ms_per_step": ms / a.steps,
            "e2e_reads_per_s": nq / e2e_dt, "e2e_ms_per_step": e2e_dt * 1e3,
            "roofline": {"bound": "hbm (random 128-B block reads: request-bound)",
                         "kernel": str(tr.get("kernel")) if tr else "search_amino_wave_kernel",
                         "path": "device seed table (k = 6 at this size), one-symbol steps until the interval is one row wide, then "
                                 "SA[row] and a byte-wise comparison with the text on the device",
                         "kernel_ms": kernel_ms, "traffic": phys,
                         "achieved": (phys / (kernel_ms * 1e-3) / 1e9) if phys else None,
                         "peak": peak, "unit": "GB/s", "frac": (phys / (kernel_ms * 1e-3) / 1e9 / peak) if phys else None,
                         "algorithmic_equivalent_gbs": alg_bytes / (kernel_ms * 1e-3) / 1e9,
                         "line_requests_per_s": requests / (kernel_ms * 1e-3),
                         "lf_steps_per_s": nq * (L - k) / (kernel_ms * 1e-3)},
            "cpu_baseline": {"value": ns / cpu_dt, "unit": "reads/s", "cores": po.lib().awo_hw_threads(), "kind": "port",
                             "sample": f"first {ns} peptides ({cpu_dt:.2f} s)"},
            "parity_vs_oracle_on_sample": parity,
            "locate": {"queries": nl, "hits": res[0][1], "gather_hits_per_s": res[0][1] / (res[0][0] * 1e-3),
                       "gather_ms_per_step": res[0][0], "lf_walk_hits_per_s": res[1][1] / (res[1][0] * 1e-3),
                       "lf_walk_ms_per_step": res[1][0]},
        }
    return out_d


def secondary_cfg5(a, torch, f, fxg, po, stream):
    """BASELINE cfg5: repeat-rich DNA, SA ratio 32, 1 M x 50-bp queries with heavily skewed hit counts"""
    from awry_b200 import FmIndex
    from fixtures import repeats
    n, nq, L = a.cfg5_len, 1_000_000, 50
    scale = n / 1e9
    fams = ((300, int(100_000 * scale) + 10, 0.15), (6000, int(20_000 * scale) + 5, 0.15))
    text, regions = repeats.repeat_rich_text(n, seed=8, tandem_arrays=max(4, int(40 * scale)), families=fams)
    parts, _ = fxg.build_parts(0, n, 0, ratio=32, kmer_len=13, host_text=text)
    qb, qo = repeats.repeat_queries(text, regions, nq, L, seed=9)
    del text
    with FmIndex.from_parts(parts.alphabet, parts.ratio, parts.bwt_len, parts.kmer_len, parts.blocks,
                            parts.prefix_sums, parts.sa_words) as ix:
        d_q = torch.from_numpy(qb).cuda()
        d_off = torch.from_numpy(qo.astype(np.int64)).cuda()
        d_hoff = torch.zeros(nq + 1, dtype=torch.int64, device="cuda")
        res = {}
        f.profile_enable(True)
        for variant in (1, 2, 0):
            f.set_locate_variant(variant)
            try:
                def once():
                    ptr, nh = ix.locate_device(d_q.data_ptr(), d_off.data_ptr(), nq, d_hoff.data_ptr(), stream=stream)
                    ix.device_free(ptr)
                    return nh
                nh = once()
                f.profile_reset()
                steps = max(1, min(a.steps, 3))
                lms = timed_device_leg(torch, torch.cuda.synchronize, once, steps, warmup=0) / steps
                p = f.profile_get()
            finally:
                f.set_locate_variant(0)
            res[variant] = (lms, nh, p["walk_ms"] / max(1, p["walk_launches"]), p["search_ms"] / max(1, p["search_launches"]))
        f.profile_enable(False)
        lean_r = ix.lean_sa_ratio()
        cnt = np.diff(d_hoff.cpu().numpy().view(np.uint64))
        ns = 2000
        orc = po.OracleIndex.from_parts(parts.alphabet, parts.ratio, parts.bwt_len, parts.kmer_len, parts.blocks,
                                        parts.prefix_sums, parts.sa_words)
        t0 = time.perf_counter()
        woff, whits, st = orc.locate_batch(qb[: ns * L], qo[: ns + 1])
        cpu_dt = time.perf_counter() - t0
        parity = bool(np.array_equal(np.diff(woff), cnt[:ns]))
        walk = st["walk_steps"] / max(1, st["hits"])
        out = {
            "workload": f"parallel_locate {nq} x {L}-bp queries vs {n}-bp repeat-rich synthetic DNA, SA ratio 32 (cfg5)",
            "hits": res[0][1], "hits_per_query": {"min": int(cnt.min()), "median": float(np.median(cnt)),
                                                  "mean": float(cnt.mean()), "max": int(cnt.max())},
            "gather": {"hits_per_s": res[0][1] / (res[0][0] * 1e-3), "ms_per_step": res[0][0], "pass2_kernel_ms": res[0][2],
                       "roofline": {"bound": "hbm", "algorithmic_bytes_per_hit": 4 + 16,
                                    "achieved_gbs": res[0][1] * 20 / (res[0][2] * 1e-3) / 1e9}},
            "bounded_walk": {"what": "walk blocks + suffix array sampled by text position (derived at load time): at most "
                                     "ratio - 1 LF steps per hit, consecutive hits of an interval walked side by side",
                             "hits_per_s": res[2][1] / (res[2][0] * 1e-3), "ms_per_step": res[2][0], "pass2_kernel_ms": res[2][2],
                             "device_bytes": ix.device_bytes()["lean_sa"], "unsampled_array_bytes": ix.device_bytes()["full_sa"],
                             "position_sampling_distance": lean_r,
                             "roofline": {"bound": "hbm (random 128-B walk-block reads)", "mean_walk_len": (lean_r - 1) / 2,
                                          "block_reads_per_hit": (lean_r - 1) / 2 + 1,
                                          "algorithmic_bytes_per_hit": 104 * ((lean_r - 1) / 2 + 1) + 20,
                                          "achieved_gbs": res[2][1] * (104 * ((lean_r - 1) / 2 + 1) + 20) / (res[2][2] * 1e-3) / 1e9,
                                          "block_reads_per_s": res[2][1] * ((lean_r - 1) / 2 + 1) / (res[2][2] * 1e-3)}},
            "lf_walk": {"hits_per_s": res[1][1] / (res[1][0] * 1e-3), "ms_per_step": res[1][0], "pass2_kernel_ms": res[1][2],
                        "mean_walk_len": walk,
                        "roofline": {"bound": "hbm (random block reads)", "algorithmic_bytes_per_hit": 104 * walk + 20,
                                     "achieved_gbs": res[1][1] * (104 * walk + 20) / (res[1][2] * 1e-3) / 1e9,
                                     "lf_steps_per_s": res[1][1] * walk / (res[1][2] * 1e-3)}},
            "search_kernel_ms": res[0][3],
            "cpu_baseline": {"value": int(woff[-1]) / cpu_dt, "unit": "hits/s", "cores": po.lib().awo_hw_threads(),
                             "kind": "port", "sample": f"first {ns} queries ({int(woff[-1])} hits, {cpu_dt:.2f} s)"},
            "hit_counts_match_oracle_on_sample": parity,
        }
    return out


def inprocess_leg(a, torch, f, fxg, parts, world, rank_sums, rank_hit_totals):
    """N > 1, rank 0 only: ONE handle with N replicas, ONE call per step over the reads of all ranks"""
    from awry_b200 import FmIndex
    nq, L = a.reads, a.read_len
    t0 = time.time()
    ix = FmIndex.from_parts(parts.alphabet, parts.ratio, parts.bwt_len, parts.kmer_len, parts.blocks,
                            parts.prefix_sums, parts.sa_words, devices=list(range(world)))
    t_index = time.time() - t0
    total = world * nq
    h_q = pinned_like(torch, total * L, torch.uint8)
    for r in range(world):
        d = device_reads(fxg, 0, a.text_len, TEXT_SEED, nq, L, QUERY_SEED + 1000 * r)
        h_q[r * nq * L:(r + 1) * nq * L].copy_(d)
        del d
    h_off = pinned_like(torch, total + 1, torch.int64)
    h_off.copy_(torch.arange(0, total + 1, dtype=torch.int64) * L)
    h_cnt = pinned_like(torch, total, torch.int64)
    torch.cuda.synchronize()
    qb, qo, out = h_q.numpy(), h_off.numpy().view(np.uint64), h_cnt.numpy().view(np.uint64)
    hw = os.cpu_count() or 16
    f.set_host_threads(min(hw, 256))        # this process owns the host now: the other ranks wait on a socket
    res = {"index_on_n_devices_s": round(t_index, 2), "host_threads": f.host_threads(), "host_cores": hw}
    try:
        # what the HOST can deliver, measured alone: the packer on all threads, and raw pinned -> device copies on
        # all N links at once.  ASCII reads cross host memory once either way (read by the cores or by the DMA
        # engines), so these two rates bound `ascii` below whatever the GPUs could search.
        import ctypes as C
        nb = nq * L
        pk_dst = pinned_like(torch, nb // 4 + 64, torch.uint8).numpy()      # pinned and touched, like the library's staging
        pk_exc = np.zeros(1 << 16, dtype=np.uint64)
        pk_n = C.c_uint64()

        def pack_once(r):
            rc = f.native().awry_host_pack_dna(qb[r * nb:].ctypes.data, nb, pk_dst.ctypes.data, pk_exc.ctypes.data, len(pk_exc),
                                               C.byref(pk_n))
            assert rc == 0
        pack_once(0)
        t0 = time.perf_counter()
        for r in range(world):
            pack_once(r)
        pack_gbs = world * nb / (time.perf_counter() - t0) / 1e9
        dsts = []
        for r in range(world):
            with torch.cuda.device(r):
                dsts.append((torch.empty(nb, dtype=torch.uint8, device=f"cuda:{r}"), torch.cuda.Stream(device=r)))
        def raw_all():
            for r, (dt_, st_) in enumerate(dsts):
                with torch.cuda.device(r), torch.cuda.stream(st_):
                    dt_.copy_(h_q[r * nb:(r + 1) * nb], non_blocking=True)
            for r, (dt_, st_) in enumerate(dsts):
                st_.synchronize()
        raw_all()
        t0 = time.perf_counter()
        raw_all()
        raw_gbs = world * nb / (time.perf_counter() - t0) / 1e9
        del dsts
        res["host_limits"] = {"pack_all_threads_gbs": pack_gbs, "raw_h2d_all_links_gbs": raw_gbs,
                              "reads_per_s_if_only_packed": pack_gbs * 1e9 / L, "reads_per_s_if_only_raw": raw_gbs * 1e9 / L}
        for _ in range(3):
            ix.count_packed(qb, qo, out=out)
        f.profile_reset()
        t0 = time.perf_counter()
        for _ in range(a.steps):
            ix.count_packed(qb, qo, out=out)
        dt = (time.perf_counter() - t0) / a.steps
        p = f.profile_get()
        sums = [int(out[r * nq:(r + 1) * nq].sum(dtype=np.uint64)) for r in range(world)]
        res["ascii"] = {"value": total / dt, "unit": "reads/s", "ms_per_step": dt * 1e3,
                        "h2d_bytes_per_step": p["h2d_bytes"] // a.steps, "d2h_bytes_per_step": p["d2h_bytes"] // a.steps,
                        "counts_equal_per_rank_device_counts": sums == rank_sums}
        # pre-packed input (awry_count_batch_packed2): the reads packed once, outside the timed region
        crumbs_np, exc = f.host_pack_dna(qb)
        h_c = pinned_like(torch, len(crumbs_np) + 64, torch.uint8)
        h_c[:len(crumbs_np)].copy_(torch.from_numpy(crumbs_np))
        cr = h_c.numpy()
        del crumbs_np
        for _ in range(2):
            ix.count_prepacked(cr, qo, exc, out=out)
        f.profile_reset()
        t0 = time.perf_counter()
        for _ in range(a.steps):
            ix.count_prepacked(cr, qo, exc, out=out)
        dt2 = (time.perf_counter() - t0) / a.steps
        p2 = f.profile_get()
        sums2 = [int(out[r * nq:(r + 1) * nq].sum(dtype=np.uint64)) for r in range(world)]
        res["prepacked"] = {"value": total / dt2, "unit": "reads/s", "ms_per_step": dt2 * 1e3,
                            "h2d_bytes_per_step": p2["h2d_bytes"] // a.steps, "d2h_bytes_per_step": p2["d2h_bytes"] // a.steps,
                            "counts_equal_per_rank_device_counts": sums2 == rank_sums}
        if not a.no_locate and rank_hit_totals:
            nl, ll = a.locate_reads, a.locate_len
            tl = world * nl
            hl_q = pinned_like(torch, tl * ll, torch.uint8)
            for r in range(world):
                d = device_reads(fxg, 0, a.text_len, TEXT_SEED, nl, ll, QUERY_SEED + 1 + 1000 * r)
                hl_q[r * nl * ll:(r + 1) * nl * ll].copy_(d)
                del d
            hl_off = pinned_like(torch, tl + 1, torch.int64)
            hl_off.copy_(torch.arange(0, tl + 1, dtype=torch.int64) * ll)
            want_hits = sum(rank_hit_totals)
            hoff = pinned_like(torch, tl + 1, torch.int64).numpy().view(np.uint64)
            hits = torch.zeros((want_hits + 1024, 2), dtype=torch.int64, pin_memory=True).numpy().view(np.uint64)
            torch.cuda.synchronize()
            lq, lo = hl_q.numpy(), hl_off.numpy().view(np.uint64)
            n_h = ix.locate_packed_into(lq, lo, hoff, hits)
            t0 = time.perf_counter()
            for _ in range(a.steps):
                n_h = ix.locate_packed_into(lq, lo, hoff, hits)
            dtl = (time.perf_counter() - t0) / a.steps
            per_rank = [int(hoff[(r + 1) * nl] - hoff[r * nl]) for r in range(world)]
            res["locate"] = {"hits_per_s": n_h / dtl, "ms_per_step": dtl * 1e3, "queries": tl, "hits": n_h,
                             "hit_totals_equal_per_rank": per_rank == rank_hit_totals}
    finally:
        f.set_host_threads(0)
        ix.close()
    return res


def main():
    a = parse_args()
    if a.impl == "reference":
        return run_reference(a)
    rank, local_rank, world = dist_env()
    if a.dump_outputs and rank == 0:
        os.makedirs(a.dump_outputs, exist_ok=True)     # fail before the set-up, not after the timed steps
    import torch
    import torch.distributed as dist
    if not torch.cuda.is_available():
        print("bench.py: no CUDA device; the awry_b200 search path has no CPU fallback", file=sys.stderr)
        return 2
    torch.cuda.set_device(local_rank)
    gloo = None
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
        try:   # host-side waits that do not spin on a core (see the in-process leg)
            gloo = dist.new_group(backend="gloo")
        except Exception:  # noqa: BLE001 -- no usable interface for gloo: wait on NCCL instead (spins, still correct)
            gloo = None
    from awry_b200 import FmIndex, fm_index as f
    from fixtures import pyfixture_gpu as fxg

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- setup (untimed): index fixture, device replica, reads in HBM and in pinned host memory
    t_setup = time.time()
    parts, phases = build_host_index(a, local_rank)
    ix = FmIndex.from_parts(parts.alphabet, parts.ratio, parts.bwt_len, parts.kmer_len, parts.blocks,
                            parts.prefix_sums, parts.sa_words, devices=[local_rank])
    nq, L = a.reads, a.read_len
    qseed = QUERY_SEED + 1000 * rank           # every rank searches its own batch
    d_q = device_reads(fxg, 0, a.text_len, TEXT_SEED, nq, L, qseed)
    d_off = torch.arange(0, nq + 1, dtype=torch.int64, device="cuda") * L
    d_cnt = torch.zeros(nq, dtype=torch.int64, device="cuda")
    stream = torch.cuda.current_stream().cuda_stream
    torch.cuda.synchronize()
    setup_s = time.time() - t_setup
    dev_bytes = ix.device_bytes()

    def step_device():
        ix.count_device(d_q.data_ptr(), d_off.data_ptr(), nq, d_cnt.data_ptr(), stream)

    # ---- kernel-only figure: inputs resident in HBM, CUDA events on the launching stream
    f.set_count_variant(a.count_variant)
    in_text = a.count_variant == 0 and dev_bytes.get("text", 0) > 0   # the default path finishes one-row intervals in the text
    for _ in range(max(a.warmup, 3)):
        step_device()
    barrier()
    f.profile_enable(True)
    f.profile_reset()
    sampler = ClockSampler(local_rank)
    sampler.start()
    sampler.wait_ready()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    sampler.mark_begin()
    e0.record()
    for _ in range(a.steps):
        step_device()
    e1.record()
    barrier()
    sampler.mark_end()
    ms_total = e0.elapsed_time(e1)
    clocks = sampler.stop()
    prof = f.profile_get()
    f.profile_enable(False)
    ix.device_check(stream)
    if a.dump_outputs and rank == 0:
        dump_counts(a.dump_outputs, d_cnt.cpu().numpy().view(np.uint64))
    t_ms = torch.tensor([ms_total], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t_ms, op=dist.ReduceOp.MAX)
    ms_max = float(t_ms.item())
    value = world * nq * a.steps / (ms_max * 1e-3)

    # ---- the same leg with backward search to the last symbol (awry_set_count_variant(1)): the kernel the
    # north star describes, one block read per two symbols of every read; same counts
    lf_only = None
    if in_text:
        d_cnt_lf = torch.zeros(nq, dtype=torch.int64, device="cuda")
        f.set_count_variant(1)
        try:
            for _ in range(3):
                ix.count_device(d_q.data_ptr(), d_off.data_ptr(), nq, d_cnt_lf.data_ptr(), stream)
            barrier()
            f.profile_enable(True)
            f.profile_reset()
            l0, l1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            l0.record()
            for _ in range(a.steps):
                ix.count_device(d_q.data_ptr(), d_off.data_ptr(), nq, d_cnt_lf.data_ptr(), stream)
            l1.record()
            barrier()
            prof_lf = f.profile_get()
            f.profile_enable(False)
        finally:
            f.set_count_variant(0)
        t_l = torch.tensor([l0.elapsed_time(l1)], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(t_l, op=dist.ReduceOp.MAX)
        lf_only = {"value": world * nq * a.steps / (float(t_l.item()) * 1e-3), "unit": "reads/s",
                   "ms_per_step": float(t_l.item()) / a.steps,
                   "kernel_ms": prof_lf["search_ms"] / max(1, prof_lf["search_launches"]),
                   "counts_equal_default_path": bool(torch.equal(d_cnt_lf, d_cnt))}
        del d_cnt_lf

    # ---- end-to-end figure: C-ABI call with pinned HOST buffers, H2D + D2H inside the timed region
    e2e = e2e_packed = None
    if not a.no_e2e:
        h_q = pinned_like(torch, nq * L, torch.uint8)
        h_q.copy_(d_q)
        h_off = pinned_like(torch, nq + 1, torch.int64)
        h_off.copy_(d_off)
        h_cnt = pinned_like(torch, nq, torch.int64)
        torch.cuda.synchronize()
        qb = h_q.numpy()
        qo = h_off.numpy().view(np.uint64)
        out = h_cnt.numpy().view(np.uint64)
        for _ in range(2):
            ix.count_packed(qb, qo, out=out)
        f.profile_reset()
        barrier()
        t0 = time.perf_counter()
        for _ in range(a.steps):
            ix.count_packed(qb, qo, out=out)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        p2 = f.profile_get()
        t_e = torch.tensor([dt], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(t_e, op=dist.ReduceOp.MAX)
        e2e = {"value": world * nq * a.steps / float(t_e.item()), "unit": "reads/s",
               "h2d_bytes_per_step": p2["h2d_bytes"] // a.steps, "d2h_bytes_per_step": p2["d2h_bytes"] // a.steps,
               "ms_per_step": float(t_e.item()) / a.steps * 1e3, "host_buffers": "pinned",
               "host_pack": ("bases packed to 2 bits by the host thread pool before the copy"
                             if p2["h2d_bytes"] // a.steps < nq * L else "ASCII bytes copied as they are"),
               "host_threads": f.host_threads()}
        assert np.array_equal(out, d_cnt.cpu().numpy().view(np.uint64)), "e2e and device-resident counts differ"
        # the same call on reads the caller already holds as 2-bit codes (awry_count_batch_packed2)
        crumbs_np, exc = f.host_pack_dna(qb)
        h_c = pinned_like(torch, len(crumbs_np) + 64, torch.uint8)
        h_c[:len(crumbs_np)].copy_(torch.from_numpy(crumbs_np))
        cr = h_c.numpy()
        out[:] = 0
        for _ in range(2):
            ix.count_prepacked(cr, qo, exc, out=out)
        f.profile_reset()
        barrier()
        t0 = time.perf_counter()
        for _ in range(a.steps):
            ix.count_prepacked(cr, qo, exc, out=out)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        p3 = f.profile_get()
        t_e = torch.tensor([dt], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(t_e, op=dist.ReduceOp.MAX)
        e2e_packed = {"value": world * nq * a.steps / float(t_e.item()), "unit": "reads/s",
                      "h2d_bytes_per_step": p3["h2d_bytes"] // a.steps, "d2h_bytes_per_step": p3["d2h_bytes"] // a.steps,
                      "ms_per_step": float(t_e.item()) / a.steps * 1e3,
                      "input": "reads pre-packed to 2 bits per base by the caller (pinned), awry_count_batch_packed2"}
        assert np.array_equal(out, d_cnt.cpu().numpy().view(np.uint64)), "pre-packed and device-resident counts differ"
        del h_q, h_c, qb, cr

    # ---- secondary run of cfg2 (SURVEY.md 8(d)): 10 % of the reads carry one random substitution, so their
    # search ends early with an empty interval; same timing rules as the headline figure
    mutated = None
    if not a.no_locate:
        d_qm = device_reads(fxg, 0, a.text_len, TEXT_SEED, nq, L, qseed, mut_ppm=100_000)
        d_cm = torch.zeros(nq, dtype=torch.int64, device="cuda")
        for _ in range(3):
            ix.count_device(d_qm.data_ptr(), d_off.data_ptr(), nq, d_cm.data_ptr(), stream)
        barrier()
        m0, m1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        m0.record()
        for _ in range(a.steps):
            ix.count_device(d_qm.data_ptr(), d_off.data_ptr(), nq, d_cm.data_ptr(), stream)
        m1.record()
        barrier()
        t_m = torch.tensor([m0.elapsed_time(m1)], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(t_m, op=dist.ReduceOp.MAX)
        zero = int((d_cm == 0).sum())
        mutated = {"workload": "same batch, 10 % of the reads with one substitution (early exit)",
                   "reads_per_s": world * nq * a.steps / (float(t_m.item()) * 1e-3),
                   "ms_per_step": float(t_m.item()) / a.steps, "reads_without_a_hit": zero}
        del d_qm, d_cm

    # ---- secondary metric (BASELINE cfg3): parallel_locate of 1 M x 50-bp queries, same index
    locate = None
    n_hits = 0
    if not a.no_locate:
        nl, ll = a.locate_reads, a.locate_len
        d_lq = device_reads(fxg, 0, a.text_len, TEXT_SEED, nl, ll, QUERY_SEED + 1 + 1000 * rank)
        d_loff = torch.arange(0, nl + 1, dtype=torch.int64, device="cuda") * ll
        d_hoff = torch.zeros(nl + 1, dtype=torch.int64, device="cuda")

        def locate_leg(variant):
            """device-resident two-pass locate, CUDA events; variant 0 = default pass 2, 1 = LF-walk"""
            f.set_locate_variant(variant)
            try:
                nh = 0
                for _ in range(2):
                    ptr, nh = ix.locate_device(d_lq.data_ptr(), d_loff.data_ptr(), nl, d_hoff.data_ptr(), stream=stream)
                    ix.device_free(ptr)
                f.profile_enable(True)
                f.profile_reset()
                barrier()
                l0, l1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                l0.record()
                for _ in range(a.steps):
                    ptr, nh = ix.locate_device(d_lq.data_ptr(), d_loff.data_ptr(), nl, d_hoff.data_ptr(), stream=stream)
                    ix.device_free(ptr)
                l1.record()
                barrier()
                prof_l = f.profile_get()
                f.profile_enable(False)
            finally:
                f.set_locate_variant(0)
            t = torch.tensor([l0.elapsed_time(l1)], dtype=torch.float64, device="cuda")
            if world > 1:
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
            return float(t.item()) / a.steps, prof_l, nh

        walk_lms, walk_lp, n_hits = locate_leg(1)
        lean_lms, lean_lp, n_hits3 = locate_leg(2)
        lms, lp, n_hits2 = locate_leg(0)
        assert n_hits == n_hits2 == n_hits3
        unsampled = ix.device_bytes()["full_sa"] > 0
        # end to end through the C ABI: pinned host queries in, CSR offsets + hits out to the host
        hl_q = pinned_like(torch, nl * ll, torch.uint8)
        hl_q.copy_(d_lq)
        hl_off = pinned_like(torch, nl + 1, torch.int64)
        hl_off.copy_(d_loff)
        torch.cuda.synchronize()
        lqb, lqo = hl_q.numpy(), hl_off.numpy().view(np.uint64)
        hoff_h = torch.zeros(nl + 1, dtype=torch.int64, pin_memory=True).numpy().view(np.uint64)
        hits_h = torch.zeros((n_hits + 1024, 2), dtype=torch.int64, pin_memory=True).numpy().view(np.uint64)
        for _ in range(2):
            ix.locate_packed_into(lqb, lqo, hoff_h, hits_h)
        f.profile_reset()
        barrier()
        t0 = time.perf_counter()
        for _ in range(a.steps):
            n_e2e = ix.locate_packed_into(lqb, lqo, hoff_h, hits_h)
        dt = (time.perf_counter() - t0) / a.steps
        pl = f.profile_get()
        t_le = torch.tensor([dt], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(t_le, op=dist.ReduceOp.MAX)
        assert np.array_equal(hoff_h, d_hoff.cpu().numpy().view(np.uint64)), "e2e and device-resident hit offsets differ"
        locate = {"workload": f"parallel_locate {nl} x {ll}-bp queries, SA ratio {a.sa_ratio} (cfg3)",
                  "pass2": "gather from the unsampled suffix array (rebuilt on the device at load time)" if unsampled
                           else "LF-walk to the sampled rows",
                  "hits_per_query": n_hits / nl, "hits_per_s": world * n_hits / (lms * 1e-3),
                  "queries_per_s": world * nl / (lms * 1e-3), "ms_per_step": lms,
                  "pass2_kernel_ms": lp["walk_ms"] / max(1, lp["walk_launches"]),
                  "search_kernel_ms": lp["search_ms"] / max(1, lp["search_launches"]),
                  "e2e": {"hits_per_s": world * n_e2e / float(t_le.item()), "ms_per_step": float(t_le.item()) * 1e3,
                          "h2d_bytes_per_step": pl["h2d_bytes"] // a.steps, "d2h_bytes_per_step": pl["d2h_bytes"] // a.steps,
                          "path": "awry_locate_batch_into, pinned buffers: hits written by the gather kernel straight "
                                  "into the caller's buffer, one wait per call"},
                  "lf_walk_variant": {"hits_per_s": world * n_hits / (walk_lms * 1e-3), "ms_per_step": walk_lms,
                                      "walk_kernel_ms": walk_lp["walk_ms"] / max(1, walk_lp["walk_launches"])},
                  "bounded_walk_variant": {"hits_per_s": world * n_hits / (lean_lms * 1e-3), "ms_per_step": lean_lms,
                                           "walk_kernel_ms": lean_lp["walk_ms"] / max(1, lean_lp["walk_launches"]),
                                           "device_bytes": ix.device_bytes()["lean_sa"],
                                           "position_sampling_distance": ix.lean_sa_ratio(),
                                           "unsampled_array_bytes": ix.device_bytes()["full_sa"]}}
        del d_lq, d_loff, d_hoff

    # ---- CPU baseline + parity + exact algorithmic work (rank 0, N = 1 only)
    cpu_baseline, parity, touches_per_read = None, None, None
    if rank == 0 and world == 1 and not a.no_cpu_baseline:
        from oracle import pyoracle as po
        orc = po.OracleIndex.from_parts(parts.alphabet, parts.ratio, parts.bwt_len, parts.kmer_len, parts.blocks,
                                        parts.prefix_sums, parts.sa_words)
        ns = min(a.cpu_sample, nq)
        sb = d_q[: ns * L].cpu().numpy()
        so = np.arange(ns + 1, dtype=np.uint64) * np.uint64(L)
        cores = po.lib().awo_hw_threads()
        orc.count_batch(sb[: 100_000 * L], so[:100_001])     # warm-up
        t0 = time.perf_counter()
        want, st = orc.count_batch(sb, so)
        dt = time.perf_counter() - t0
        parity = bool(np.array_equal(want, d_cnt[:ns].cpu().numpy().view(np.uint64)))
        touches_per_read = st["seeded_touches"] / ns
        cpu_baseline = {"value": ns / dt, "unit": "reads/s", "cores": cores, "kind": "port",
                        "sample": f"first {ns} reads of the batch ({dt:.1f} s), C port of the reference search path "
                                  f"in the reference block layout, {cores} pthreads (dynamic chunks) for rayon"}
        del orc
    if touches_per_read is None:
        # closed form of SURVEY.md 8(d): L-k seeded steps, ~1.006 distinct blocks per step
        touches_per_read = (L - a.kmer) * 1.006

    # ---- roofline of the dominant kernel (backward search), measured live.  `achieved` is PHYSICAL: the DRAM
    # bytes one launch moves (ncu dram__bytes_read + write of this very command, profiles/) over the kernel's
    # mean launch time in this run; the reference algorithm's bytes (104 B per LF step, SURVEY 8(d)) over the
    # same time are reported beside it -- the pair index does two LF steps per 128-B read, so that figure can
    # exceed the stream peak and is not a fraction of anything.
    peak, peak_src = measured_peak()
    alg_bytes_per_launch = nq * (L + 8 + 16 + ALG_BYTES_PER_BLOCK * touches_per_read)
    search_ms = prof["search_ms"] / max(1, prof["search_launches"])
    std_cfg = nq == 10_000_000 and L == 150 and a.kmer == 13 and a.text_len == 3_100_000_000
    lf_accesses = nq * (((L - a.kmer) + 1) // 2 + 1)          # pair steps (+ odd tail) + seed lookup
    g_reads = g_gbs = None
    gather_err = None
    if rank == 0:
        try:   # the "random-access HBM roofline" of the north star: independent random 128-B reads
            # 4 lanes x LDG.256 per read, 4 in flight per lane group, 16 waves of blocks so the hardware
            # balances the SMs (a static split stops at 37.8 G reads/s: it ends with the slowest SM)
            g_reads, g_gbs = f.bench_random_gather(local_rank, 4 << 30, 128, 3164, 400_000_000, 2)
        except Exception as e:  # noqa: BLE001
            gather_err = str(e)

    def roofline_of(kernel_ms, text_path, share):
        """physical roofline of one flavour of the count kernel: ncu DRAM bytes per launch / its mean launch time"""
        tr = (traffic_from_profiles("search_dna_wave_kernel") if text_path
              else traffic_from_profiles("search_dna_pair_kernel", in_text=False))
        if tr and std_cfg:
            traffic, src = float(tr["dram_bytes_per_launch"]), f"ncu --set full capture of this command ({tr.get('source')})"
        elif text_path:
            traffic, src = float(nq * 940), "estimate: ~7.3 lines of 128 B per read (seed entry, 2-3 pair blocks, SA element, 1-2 lines of text, the read itself)"
        else:
            traffic, src = float(nq * ((((L - a.kmer) + 1) // 2) * 1.006 * 128 + 200)), "estimate: 128 B per block read + ~200 B per read"
        achieved = traffic / (kernel_ms * 1e-3) / 1e9
        lines = traffic / 128 if text_path else float(lf_accesses)
        gather = {"error": gather_err} if g_reads is None else {
            "granule_bytes": 128, "reads_per_s": g_reads, "gb_per_s": g_gbs,
            "kernel_line_reads_per_s": lines / (kernel_ms * 1e-3),
            "line_reads_counted_as": "DRAM bytes / 128" if text_path else "block reads issued: pair steps + seed lookup per read",
            "frac_of_random_gather": lines / (kernel_ms * 1e-3) / g_reads}
        return {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": traffic, "traffic_source": src,
                "traffic_check": "ok" if achieved <= 1.05 * peak else "FAILED: physical traffic above the stream peak",
                "peak_source": peak_src,
                "kernel": ("search_dna_wave_kernel<count, 256, 5> (+ the refilling and the scalar kernel over the queries it hands "
                           "on: none in this batch)" if text_path else "search_dna_pair_kernel<count, 256, 6> (backward search only)"),
                "kernel_ms": kernel_ms, "kernel_share_of_step": share,
                "algorithmic_bytes_per_launch": alg_bytes_per_launch,
                "algorithmic_equivalent_gbs": alg_bytes_per_launch / (kernel_ms * 1e-3) / 1e9,
                "lf_steps_per_s_equivalent": nq * (L - a.kmer) / (kernel_ms * 1e-3), "random_gather_roofline": gather}

    roofline = roofline_of(search_ms, in_text, prof["search_ms"] / ms_total)
    roofline["note"] = (
        "achieved / frac are physical DRAM traffic over the stream peak.  The default count path stops stepping once a read's "
        "interval is one row wide: it reads SA[row] and compares the rest of the read with the text (4 bits per symbol, on the "
        "device) -- ~7 line reads per 150-bp read instead of ~70, identical counts; `lf_only` is the same leg with backward "
        "search to the last symbol (the kernel the north star describes) and carries its own roofline.  "
        "algorithmic_equivalent_gbs counts the reference algorithm's bytes (104 B per LF step, SURVEY 8(d)) over the kernel "
        "time: not a fraction of anything") if in_text else (
        "achieved / frac are physical DRAM traffic over the stream peak; algorithmic_equivalent_gbs counts the reference "
        "algorithm's bytes (104 B per LF step, SURVEY 8(d)) -- two LF steps ride on one 128-B pair-block read, so it may exceed "
        "the peak; frac_of_random_gather compares block reads/s with the random 128-B gather probe of this run")
    if lf_only:
        lf_only["roofline"] = roofline_of(lf_only["kernel_ms"], False, lf_only["kernel_ms"] / lf_only["ms_per_step"])

    # ---- BASELINE cfg4 / cfg5 as secondary legs (one GPU)
    cfg4 = cfg5 = None
    if rank == 0 and world == 1 and not a.no_secondary:
        ix.close()
        ix = None
        del d_q, d_cnt
        torch.cuda.empty_cache()
        from oracle import pyoracle as po
        try:
            cfg4 = secondary_cfg4(a, torch, f, fxg, po, stream, peak)
        except Exception as e:  # noqa: BLE001
            cfg4 = {"error": repr(e)}
        torch.cuda.empty_cache()
        try:
            cfg5 = secondary_cfg5(a, torch, f, fxg, po, stream)
        except Exception as e:  # noqa: BLE001
            cfg5 = {"error": repr(e)}

    # ---- N > 1: ONE call over ONE batch on a handle with N replicas (rank 0), the library's own multi-GPU path
    inproc = None
    if world > 1 and not a.no_inprocess and not a.no_e2e:
        my = torch.tensor([int(d_cnt.sum().item()), int(n_hits)], dtype=torch.int64, device="cuda")
        allv = [torch.zeros_like(my) for _ in range(world)]
        dist.all_gather(allv, my)
        rank_sums = [int(v[0].item()) for v in allv]
        rank_hits = [int(v[1].item()) for v in allv]
        ix.close()
        ix = None
        del d_q, d_cnt
        torch.cuda.empty_cache()
        torch.cuda.synchronize()
        dist.barrier(group=gloo) if gloo is not None else dist.barrier()
        if rank == 0:
            try:
                inproc = inprocess_leg(a, torch, f, fxg, parts, world, rank_sums, rank_hits if not a.no_locate else None)
            except Exception as e:  # noqa: BLE001
                inproc = {"error": repr(e)}
        dist.barrier(group=gloo) if gloo is not None else dist.barrier()   # the other ranks sleep on a socket meanwhile

    if rank == 0:
        e2e_line = e2e
        if inproc and "ascii" in inproc:
            e2e_line = dict(inproc["ascii"])
            e2e_line.update({"host_buffers": "pinned", "host_threads": inproc["host_threads"],
                             "call": f"ONE awry_count_batch per step over {world} x {nq} reads on a handle with {world} replicas "
                                     "(rank 0; the other ranks idle); the batch is range-partitioned by query bytes, one host "
                                     "thread per replica, one shared packer pool"})
        line = {
            "metric": "count queries/s", "value": value, "unit": "reads/s", "n_gpus": world, "steps": a.steps,
            "warmup": max(a.warmup, 3), "ms_per_step": ms_max / a.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "u32", "data": "synthetic",
            "config": config_of(a), "setup": {"setup_s": round(setup_s, 1), "fixture_build_s": phases.get("total"),
                                              "index_device_bytes": dev_bytes},
            "count_path": ("backward search until the interval is one row wide, then SA[row] and a comparison of the rest of "
                           "the read with the text on the device (bit-exact; `lf_only` = backward search to the last symbol)"
                           if in_text else "backward search to the last symbol"),
            "roofline": roofline, "lf_only": lf_only, "cpu_baseline": cpu_baseline, "e2e": e2e_line, "clocks": clocks,
            "gpu_launches": int(prof["launches"]), "parity_vs_oracle_on_sample": parity,
            "e2e_prepacked": (inproc or {}).get("prepacked") or e2e_packed,
            "e2e_per_process": e2e if world > 1 else None,
            "e2e_prepacked_per_process": e2e_packed if world > 1 else None,
            "inprocess_replicas": inproc,
            "locate": locate, "count_with_mismatches": mutated, "cfg4_protein": cfg4, "cfg5_repeat_rich": cfg5,
        }
        print(json.dumps(line), flush=True)
    if ix is not None:
        ix.close()
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
