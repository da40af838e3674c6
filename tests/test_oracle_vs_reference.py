"""CPU: the oracle against the unmodified reference classes (CKmerBinSorter<SIZE>::ProcessBins, RADULS, radix.h).  What the
reference returned for these inputs is stored in tests/golden/reference_results.json ("oracle_vs_reference"); the module-level
case builders are shared with tests/golden/make_reference_results.py, which ran the reference on them."""
import numpy as np
import pytest

from kmc_testlib import Params, synth_bin, pack_superkmers, choose_lut_prefix_len, reference_results, result_digest, sha256

BIN_CASES = [(31, True, 2), (31, False, 1), (28, True, 1), (28, False, 2), (55, True, 2), (55, False, 1),
             (17, True, 1), (32, True, 2), (64, True, 1), (70, True, 2), (33, True, 1), (128, True, 1)]
BIN_VARIANTS = {                       # how the reference processed the bin: (n_sorters, sort_kind)
    "raduls": (1, 0),                  # RADULS, one sorter
    "radix": (1, 1),                   # radix.h + CSmallSort (non-Intel hosts, kmc.h:1556-1560)
    "sorters4": (4, 0),                # in-bin threads: packs with gaps (kxmer_set.h:299-314)
}
CUTOFF_CASES = [(1, 10 ** 9, 255), (3, 9, 4), (2, 300, 65535), (1, 10 ** 9, 1)]
SEVERAL_BINS_SORTERS = 3               # several_bins() went through the reference in one call with this many sorters
SORT_CASES = [(1, 8), (1, 5), (2, 14), (2, 15), (3, 18), (4, 32)]
SORT_THREADS = 2                       # RADULS threads of the reference sort


def bin_case(k, both, cmin):
    p = Params(k=k, both_strands=both, cutoff_min=cmin, lut_prefix_len=choose_lut_prefix_len(k))
    return "k%d_both%d_ci%d" % (k, both, cmin), p, synth_bin(k + cmin, k, 2500, genome_len=3000, err=0.02)


def cutoff_case(cmin, cmax, cntmax):
    p = Params(k=31, cutoff_min=cmin, cutoff_max=cmax, counter_max=cntmax, lut_prefix_len=7)
    return "ci%d_cx%d_cs%d" % (cmin, cmax, cntmax), p, synth_bin(cmin * 7 + cmax % 13, 31, 3000, genome_len=500, err=0.005)


def edge_bins():
    rng = np.random.default_rng(1)
    p = Params(k=31, cutoff_min=1, lut_prefix_len=7)
    return p, [pack_superkmers(31, [rng.integers(0, 4, 31)]),
               pack_superkmers(31, [rng.integers(0, 4, 31 + 255) for _ in range(40)]),
               pack_superkmers(31, [np.zeros(31 + 255, dtype=np.uint8) for _ in range(30)]),
               pack_superkmers(31, [np.tile(np.array([0, 3], dtype=np.uint8), 100)[:31 + 150] for _ in range(20)])]


def several_bins():
    p = Params(k=31, cutoff_min=2, lut_prefix_len=7)
    return p, [synth_bin(50 + i, 31, n, genome_len=max(n, 400)) for i, n in enumerate([400, 0, 2500, 30, 1200])]


def sort_case(words, key_bytes):
    rng = np.random.default_rng(words * 100 + key_bytes)
    n = 20000
    raw = rng.integers(0, 256, size=(n, words * 8), dtype=np.uint8)
    raw[:, key_bytes:] = 0
    raw[n // 2:] = raw[rng.integers(0, n // 2, n - n // 2)]
    return "w%d_kb%d" % (words, key_bytes), raw.view(np.uint64).reshape(n, words)


@pytest.mark.parametrize("k,both,cmin", BIN_CASES)
def test_bin_matches_reference(oracle, k, both, cmin):
    name, p, b = bin_case(k, both, cmin)
    got = result_digest(oracle.process_bin(b, p))
    ref = reference_results("oracle_vs_reference")["bin_" + name]
    for variant in BIN_VARIANTS:
        assert got == ref[variant], variant


def test_cutoffs_and_clamp_match_reference(oracle):
    for case in CUTOFF_CASES:
        name, p, b = cutoff_case(*case)
        assert result_digest(oracle.process_bin(b, p)) == reference_results("oracle_vs_reference")["cutoff_" + name], name


def test_edge_bins_match_reference(oracle):
    p, bins = edge_bins()
    ref = reference_results("oracle_vs_reference")["edge_bins"]
    assert [result_digest(oracle.process_bin(b, p)) for b in bins] == ref


def test_several_bins_many_sorters(oracle):
    p, bins = several_bins()
    ref = reference_results("oracle_vs_reference")["several_bins"]
    assert [result_digest(oracle.process_bin(b, p)) for b in bins] == ref


@pytest.mark.parametrize("words,key_bytes", SORT_CASES)
def test_sort_matches_raduls(oracle, words, key_bytes):
    name, recs = sort_case(words, key_bytes)
    assert sha256(oracle.sort(recs, key_bytes).tobytes()) == reference_results("oracle_vs_reference")["sort_" + name]
