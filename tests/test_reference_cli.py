"""BASELINE configs[0] (CPU plumbing, no GPU): a ~1 MB synthetic FASTQ through the UNMODIFIED reference CLI at k = 15 (the regular bin
pipeline: the small-k direct-count path needs k <= 13, SURVEY section 0.2) and k = 13 (small-k path), checked against a brute-force count
of the reads (the reference's own test strategy: tests/kmc_CLI/trivial-k-mer-counter).  What the CLI counted (`kmc -ci2 -cs255`, dumped
by `kmc_tools transform ... dump -s`) is stored in tests/golden/reference_results.json ("reference_cli", made by
tests/golden/make_reference_results.py).  This pins the FASTQ writer the whole-file GPU parity tests rest on."""
import os

import pytest

from kmc_testlib import reference_results, sha256
from test_gpu_kmc_files import write_fastq

FASTQ = dict(seed=15, n_reads=3400, genome_len=200_000)          # 3400 x 150 bp: ~1 MB of FASTQ
CLI_ARGS = ("-ci2", "-cs255")


def brute_force(fastq, k, both=True):
    comp = {"A": "T", "C": "G", "G": "C", "T": "A"}
    cnt = {}
    with open(fastq) as f:
        for i, line in enumerate(f):
            if i % 4 != 1:
                continue
            for piece in line.strip().split("N"):
                for j in range(len(piece) - k + 1):
                    km = piece[j:j + k]
                    if both:
                        rc = "".join(comp[c] for c in reversed(km))
                        km = min(km, rc)
                    cnt[km] = cnt.get(km, 0) + 1
    return cnt


def counts_sha256(counts):
    """SHA-256 of {k-mer: count} as `kmc_tools transform ... dump -s` prints it: one "kmer<TAB>count" line per k-mer, sorted."""
    return sha256("".join("%s\t%d\n" % (km, c) for km, c in sorted(counts.items())).encode())


@pytest.mark.parametrize("k", [15, 13])
def test_reference_cli_on_a_small_fastq(tmp_path, k):
    fq = os.path.join(str(tmp_path), "reads.fq")
    write_fastq(fq, FASTQ["seed"], FASTQ["n_reads"], genome_len=FASTQ["genome_len"])
    assert 0.9e6 < os.path.getsize(fq) < 1.3e6
    exp = {km: min(c, 255) for km, c in brute_force(fq, k).items() if c >= 2}
    ref = reference_results("reference_cli")["k%d" % k]
    assert counts_sha256(exp) == ref["dump_sha256"]
    assert len(exp) == ref["unique_counted_kmers"]
