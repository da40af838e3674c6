"""Runs the REFERENCE on the inputs of every test that compares with it and stores what it returned, so that those tests run
without it.  Needs oracle/_ref, built by `make -C oracle ref cli REF=<reference source tree>`:

  reference_results.json   per test module: bin results (the four counters, SHA-256 of payload and LUT), sorted records (SHA-256),
                           counts of the reference CLI, and databases read back by the reference's kmc_tools (SHA-256 of .kmc_pre,
                           .kmc_suf and of the dump it printed for them)
                           "benchmark_bins" holds bench.py's own bins, each with a SHA-256 of its input
  refdb_k*.npz             databases written by the reference CLI: .kmc_pre, .kmc_suf and the four counters of its statistics, made
                           from FASTQs small enough to store

The inputs come from the test modules themselves, so a test and its stored results cannot drift apart.
"""
import json
import os
import sys
import tempfile
import time
from concurrent.futures import ThreadPoolExecutor

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
TESTS = os.path.dirname(HERE)
sys.path[:0] = [os.path.dirname(TESTS), TESTS]

from kmc_testlib import Oracle, Params, Reference, REFERENCE_RESULTS, result_digest, sha256  # noqa: E402
import test_benchmark_bins as tbb  # noqa: E402
import test_db_writer as dbw  # noqa: E402
import test_gpu_parity as gp  # noqa: E402
import test_oracle_vs_reference as ovr  # noqa: E402
import test_reference_cli as cli  # noqa: E402
from test_gpu_kmc_files import KMC_REF, KMC_TOOLS, count, dump_sorted, run, write_fastq  # noqa: E402

REFDB_READS = {31: 400, 28: 40, 55: 40}          # 150 bp reads over a 200 kbp genome: .kmc_suf stays below 50 KB


def oracle_vs_reference(R):
    out = {}
    for case in ovr.BIN_CASES:
        name, p, b = ovr.bin_case(*case)
        out["bin_" + name] = {v: result_digest(R.process_bin(b, p, n_sorters=ns, sort_kind=kind)) for v, (ns, kind) in ovr.BIN_VARIANTS.items()}
    for case in ovr.CUTOFF_CASES:
        name, p, b = ovr.cutoff_case(*case)
        out["cutoff_" + name] = result_digest(R.process_bin(b, p))
    p, bins = ovr.edge_bins()
    out["edge_bins"] = [result_digest(R.process_bin(b, p)) for b in bins]
    p, bins = ovr.several_bins()
    out["several_bins"] = [result_digest(r) for r in R.process_bins(bins, p, n_sorters=ovr.SEVERAL_BINS_SORTERS)[0]]
    for words, key_bytes in ovr.SORT_CASES:
        name, recs = ovr.sort_case(words, key_bytes)
        out["sort_" + name] = sha256(R.sort(recs, key_bytes, n_threads=ovr.SORT_THREADS)[0].tobytes())
    return out


def reference_cli(tmp):
    out = {}
    for k in (15, 13):
        d = os.path.join(tmp, "cli_k%d" % k)
        os.makedirs(d)
        fq = os.path.join(d, "reads.fq")
        write_fastq(fq, cli.FASTQ["seed"], cli.FASTQ["n_reads"], genome_len=cli.FASTQ["genome_len"])
        db, stats = count(KMC_REF, d, "ref", fq, k, cli.CLI_ARGS)
        got = {km: int(c) for km, c in (line.split() for line in dump_sorted(d, db, "ref").splitlines())}
        assert got == {km: min(c, 255) for km, c in cli.brute_force(fq, k).items() if c >= 2}, k
        out["k%d" % k] = {"dump_sha256": cli.counts_sha256(got), "unique_counted_kmers": int(stats["Stats"]["#Unique_counted_k-mers"])}
    return out


def db_writer(tmp, oracle):
    for k, extra in dbw.REFDB_CASES:
        d = os.path.join(tmp, "refdb_k%d" % k)
        os.makedirs(d)
        fq = os.path.join(d, "reads.fq")
        write_fastq(fq, 500 + k, REFDB_READS[k])
        db, stats = count(KMC_REF, d, "ref", fq, k, extra + dbw.REFDB_ARGS)
        pre, suf = dbw.read_db(db)
        dbw.parse_db(pre, suf)
        np.savez_compressed(dbw.refdb_path(k, extra), kmc_pre=np.frombuffer(pre, dtype=np.uint8), kmc_suf=np.frombuffer(suf, dtype=np.uint8),
                            stats=np.array([int(stats["Stats"][key]) for key in dbw.REFDB_STATS], dtype=np.uint64))
    out = {}
    p = dbw.STANDALONE_PARAMS
    res = [oracle.process_bin(b, p) for b in dbw._standalone_bins()]
    for case, results in (("standalone", res), ("standalone_x3", res * 3)):
        db = os.path.join(tmp, case)
        dbw.write_oracle_db(db, results, p, 1 << 20)
        txt = os.path.join(tmp, case + ".txt")
        run([KMC_TOOLS, "transform", db, "dump", txt])
        dump = open(txt, "rb").read()
        assert dump.decode().split("\n")[:-1] == dbw._expected_dump(results, p) and dump.endswith(b"\n"), case
        pre, suf = dbw.read_db(db)
        out[case] = {"kmc_pre_sha256": sha256(pre), "kmc_suf_sha256": sha256(suf), "dump_sha256": sha256(dump)}
    return out


def gpu_parity(R):
    n_sorters = os.cpu_count() or 8
    out = {}
    for k, p_len in gp.BENCHMARK_SCALE_CASES:
        p = Params(k=k, cutoff_min=2, lut_prefix_len=p_len)
        out["bin_2^26_k%d_p%d" % (k, p_len)] = result_digest(R.process_bin(gp.benchmark_scale_bin(k), p, n_sorters=n_sorters))
    p = Params(k=31, cutoff_min=2, lut_prefix_len=7)
    out["bin_117M_k31_p7"] = result_digest(R.process_bin(gp.second_level_bin(), p, n_sorters=n_sorters))
    return out


def benchmark_bins(R):
    """Every bin bench.py times, one at a time (~1.7e9 k-mers in all).  Every result is also checked against the oracle, so that each
    stored digest is backed by two independent implementations (8 cores: ~6 min in all, most of it the single-threaded oracle)."""
    n_sorters = os.cpu_count() or 8
    oracle = Oracle()
    out = {}
    with ThreadPoolExecutor(min(32, n_sorters)) as ex:
        for case in tbb.ALL_CASES:
            t0 = time.perf_counter()
            b = case.make(ex)
            t1 = time.perf_counter()
            r = R.process_bin(b, case.params, n_sorters=n_sorters)
            t2 = time.perf_counter()
            assert oracle.process_bin(b, case.params).same_as(r), case.key
            t3 = time.perf_counter()
            out[case.key] = {"input_sha256": tbb.input_sha256(b), "result": result_digest(r)}
            print("  %s: generated %.1f s, reference %.1f s, oracle %.1f s" % (case.key, t1 - t0, t2 - t1, t3 - t2), flush=True)
            del b, r
    return out


GROUPS = {"oracle_vs_reference": lambda R, tmp: oracle_vs_reference(R), "reference_cli": lambda R, tmp: reference_cli(tmp),
          "db_writer": lambda R, tmp: db_writer(tmp, Oracle()), "gpu_parity": lambda R, tmp: gpu_parity(R),
          "benchmark_bins": lambda R, tmp: benchmark_bins(R)}


def main(groups):
    """Regenerates the named groups (all of them without arguments) and keeps the others as stored."""
    unknown = set(groups) - set(GROUPS)
    if unknown:
        sys.exit("unknown groups %s; known: %s" % (sorted(unknown), sorted(GROUPS)))
    R = Reference()
    results = {}
    if groups and os.path.exists(REFERENCE_RESULTS):
        with open(REFERENCE_RESULTS) as f:
            results = json.load(f)
    with tempfile.TemporaryDirectory() as tmp:
        for name in groups or GROUPS:
            t0 = time.perf_counter()
            results[name] = GROUPS[name](R, tmp)
            print(name, "%.0f s" % (time.perf_counter() - t0), flush=True)
    with open(REFERENCE_RESULTS, "w") as f:
        json.dump(results, f, indent=1, sort_keys=True)
        f.write("\n")
    for group, cases in results.items():
        print(group, len(cases), "cases")


if __name__ == "__main__":
    main(sys.argv[1:])
