"""bench.py picks the DRAM-traffic figure of each kernel flavour from the committed ncu summaries (profiles/*_traffic.json):
the lookups must find the captures the roofline blocks are computed from, and tell the two flavours of the pair kernel apart."""
import importlib.util
import os

import numpy as np

from conftest import ROOT


def load_bench():
    spec = importlib.util.spec_from_file_location("bench_module", os.path.join(ROOT, "bench.py"))
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m


def test_traffic_lookup_finds_every_capture():
    b = load_bench()
    wave = b.traffic_from_profiles("search_dna_wave_kernel")
    lf = b.traffic_from_profiles("search_dna_pair_kernel", in_text=False)
    amino = b.traffic_from_profiles("search_amino")
    assert wave and wave["kernel"].startswith("search_dna_wave_kernel") and wave["dram_bytes_per_launch"] > 1e9
    assert lf and lf["kernel"].startswith("search_dna_pair_kernel") and not lf["kernel"].rstrip().endswith(", 1>")
    assert amino and amino["kernel"].startswith("search_amino") and amino["dram_bytes_per_launch"] > 1e9
    # backward search to the last symbol moves an order of magnitude more than the default path
    assert lf["dram_bytes_per_launch"] > 5 * wave["dram_bytes_per_launch"]
    assert b.traffic_from_profiles("no_such_kernel") is None


def test_both_arms_describe_the_same_config():
    b = load_bench()

    class A:
        reads, read_len, text_len, kmer, sa_ratio = 10_000_000, 150, 3_100_000_000, 13, 8
    cfg = b.config_of(A)
    assert "workload" in cfg and "10000000 x 150-bp" in cfg["workload"] and "model" not in cfg


def test_dumped_counts_are_a_fixed_float_sample_under_64_mb(tmp_path):
    """--dump-outputs: float64 counts of the same reads from run to run, the whole batch when it is small"""
    b = load_bench()
    counts = np.arange(10_000_000, dtype=np.uint64) * np.uint64(3)
    for run in ("a", "b"):
        (tmp_path / run).mkdir()
        b.dump_counts(str(tmp_path / run), counts)
    got = {n: [np.load(tmp_path / run / f"{n}.npy") for run in ("a", "b")] for n in ("counts", "count_rows")}
    rows = got["count_rows"][0]
    assert all(x.dtype == np.float64 for v in got.values() for x in v)
    assert np.array_equal(*got["counts"]) and np.array_equal(*got["count_rows"])
    assert len(rows) == b.DUMP_ROWS and len(np.unique(rows)) == len(rows)
    assert np.array_equal(got["counts"][0], counts[rows.astype(np.int64)].astype(np.float64))
    assert sum(os.path.getsize(p) for p in tmp_path.glob("a/*.npy")) <= 64 << 20
    small = tmp_path / "small"
    small.mkdir()
    b.dump_counts(str(small), counts[:1000])
    assert np.array_equal(np.load(small / "count_rows.npy"), np.arange(1000))
