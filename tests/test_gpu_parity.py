"""GPU parity tests: the CUDA path, called through the C ABI, against the oracle (bit-exact)."""
import ctypes as C

import numpy as np
import pytest

from kmc_testlib import Params, Bin, synth_bin, fast_bin, pack_superkmers, choose_lut_prefix_len, bin_from_reads, reference_results, result_digest

pytestmark = pytest.mark.gpu


def _ctx(p: Params, n_slots=1):
    import kmc_b200
    return kmc_b200.Stage2Context(kmc_b200.Stage2Params(p.k, p.both_strands, p.cutoff_min, p.cutoff_max, p.counter_max, p.lut_prefix_len), device=0, n_slots=n_slots)


def _to_skb(b: Bin):
    import kmc_b200
    return kmc_b200.SuperKmerBin(data=b.data, n_rec=b.n_rec, pack_bytes=b.pack_bytes, n_super_kmers=b.n_super_kmers, kmer_len=b.k)


def _check_bin(oracle, b: Bin, p: Params, ctx=None):
    own = ctx is None
    ctx = ctx or _ctx(p)
    r = ctx.process_bin(_to_skb(b))
    e = oracle.process_bin(b, p)
    assert r.stats == e.stats
    assert np.array_equal(r.lut, e.lut)
    assert r.payload.tobytes() == e.payload
    if own:
        ctx.close()


@pytest.mark.parametrize("leaf", ["count", "sort"])
@pytest.mark.parametrize("k,both,cmin", [(31, True, 2), (31, False, 1), (28, True, 1), (17, True, 1), (32, True, 2), (32, False, 1), (15, True, 1), (5, True, 1)])
def test_bin_parity_one_word(oracle, monkeypatch, leaf, k, both, cmin):
    monkeypatch.setenv("KMCB200_LEAF", leaf)
    p = Params(k=k, both_strands=both, cutoff_min=cmin, lut_prefix_len=choose_lut_prefix_len(k))
    _check_bin(oracle, synth_bin(7, k, 20000, genome_len=30000, err=0.02), p)


@pytest.mark.parametrize("p_len,cmin,cmax,cntmax", [(7, 1, 10 ** 9, 255), (11, 2, 10 ** 9, 65535), (15, 1, 40, 3), (3, 3, 10 ** 9, 1)])
def test_leaf_count_cutoffs_and_prefix_lengths(oracle, p_len, cmin, cmax, cntmax):
    """The leaf-count path with LUT prefixes shorter and longer than the partition bits, cutoffs, clamping, 0-byte counters."""
    p = Params(k=31, cutoff_min=cmin, cutoff_max=cmax, counter_max=cntmax, lut_prefix_len=p_len)
    _check_bin(oracle, synth_bin(21, 31, 60000, genome_len=20000, err=0.01), p)


@pytest.mark.parametrize("cmin,cmax,cntmax", [(1, 10 ** 9, 255), (2, 3, 255), (1, 1, 255), (3, 2, 255), (2, 2 ** 32 - 1, 2), (5, 100, 65535)])
@pytest.mark.parametrize("k,both", [(31, True), (32, False), (17, True), (55, True), (96, False)])
def test_leaf_hash_cutoff_instances(oracle, k, both, cmin, cmax, cntmax):
    """leaf_hash_kernel: the SIMPLE instance (cutoff_min >= 2, unreachable cutoff_max) and the general one - cutoff_min = 1 (a claim is already a
    survivor), reachable cutoff_max (second bitmap), cutoff_max < cutoff_min (nothing survives, everything counts as n_cutoff_max)."""
    p = Params(k=k, both_strands=both, cutoff_min=cmin, cutoff_max=cmax, counter_max=cntmax, lut_prefix_len=choose_lut_prefix_len(k))
    _check_bin(oracle, synth_bin(77 + k, k, 30000, genome_len=9000, err=0.01), p)


@pytest.mark.parametrize("env", [{"KMCB200_LEAF_FILL_PCT": "10"}, {"KMCB200_LEAF_RATIO0": "8"}, {"KMCB200_LEAF_RATIO0": "256", "KMCB200_LEAF_FILL_PCT": "85"},
                                 {"KMCB200_L2_BITS": "2"}, {"KMCB200_L2_BITS": "2", "KMCB200_LEAF_RATIO0": "8", "KMCB200_LEAF_SLOT_BITS": "8"},
                                 {"KMCB200_LEAF_KERNEL": "warp"}, {"KMCB200_LEAF_WIDE": "warp"}])
@pytest.mark.parametrize("coverage", ["30x", "distinct"])
@pytest.mark.parametrize("k", [31, 55])
def test_leaf_hash_round_planning(oracle, monkeypatch, env, coverage, k):
    """leaf_hash_kernel plans its table rounds from a running estimate of distinct k-mers per record: rounds planned far too small (many
    predicated rounds over the leaf), far too large (the table fills up: the round is split on the next bit, binary descent), leaves of
    ~10^4 records in 256-slot tables, duplicate-rich and all-distinct k-mers, one-word and two-word records (leaf_hash_wide_kernel); and the
    round-1 kernel (leaf_warp_kernel) stays selectable."""
    for k_, v in env.items():
        monkeypatch.setenv(k_, v)
    p = Params(k=k, cutoff_min=2 if coverage == "30x" else 1, lut_prefix_len=7)
    b = synth_bin(5, k, 26000, genome_len=10000, err=0.01) if coverage == "30x" else synth_bin(6, k, 16000, genome_len=4000000, err=0.0)
    _check_bin(oracle, b, p)


def test_leaf_count_all_T_kmers(oracle):
    """k = 32, -b: TTT...T is the table's EMPTY sentinel and must still be counted (it sorts last)."""
    rng = np.random.default_rng(3)
    p = Params(k=32, both_strands=False, cutoff_min=1, lut_prefix_len=4)
    lists = [np.full(32 + 200, 3, dtype=np.uint8) for _ in range(200)] + [rng.integers(0, 4, 32 + 100) for _ in range(600)]
    _check_bin(oracle, pack_superkmers(32, lists), p)



@pytest.mark.parametrize("k,both,cmin", [(55, True, 2), (55, False, 1), (33, True, 1), (64, True, 2), (70, True, 1), (96, True, 2), (127, False, 1), (128, True, 1)])
def test_bin_parity_multi_word(oracle, k, both, cmin):
    p = Params(k=k, both_strands=both, cutoff_min=cmin, lut_prefix_len=choose_lut_prefix_len(k))
    _check_bin(oracle, synth_bin(11, k, 8000, genome_len=12000, err=0.02), p)


@pytest.mark.parametrize("slot_bits", [8, 9, 10])
@pytest.mark.parametrize("k,both,cmin,p_len", [(31, True, 2, 7), (55, True, 2, 7), (55, False, 1, 3), (33, True, 1, 5), (64, True, 2, 8), (70, True, 1, 6),
                                               (96, False, 2, 8), (128, True, 1, 8), (32, False, 1, 4), (17, True, 1, 5)])
def test_leaf_path_all_widths(oracle, monkeypatch, slot_bits, k, both, cmin, p_len):
    """~170 K k-mers (the hybrid MSD path + warp-counted leaves) for every record width and every table size."""
    monkeypatch.setenv("KMCB200_LEAF_SLOT_BITS", str(slot_bits))
    p = Params(k=k, both_strands=both, cutoff_min=cmin, lut_prefix_len=p_len)
    _check_bin(oracle, synth_bin(31 + k, k, 14000, genome_len=9000, err=0.01), p)


@pytest.mark.parametrize("l2_bits", [3, 9, 10])
@pytest.mark.parametrize("k,both,cmin,p_len", [(31, True, 2, 7), (31, False, 1, 11), (55, True, 2, 7), (70, True, 1, 6), (128, True, 1, 8), (17, True, 1, 5)])
def test_wide_second_partition_level(oracle, monkeypatch, l2_bits, k, both, cmin, p_len):
    """Bins of more than 2^26 k-mers partition their second level on 9-10 bits (512 / 1024 digits: the wide variants of the count and
    scatter kernels, 2^17-2^18 leaves) so that a leaf keeps ~1 K records; forced here on a small bin."""
    monkeypatch.setenv("KMCB200_L2_BITS", str(l2_bits))
    p = Params(k=k, both_strands=both, cutoff_min=cmin, lut_prefix_len=p_len)
    _check_bin(oracle, synth_bin(41 + k, k, 14000, genome_len=9000, err=0.01), p)


@pytest.mark.parametrize("k,p_len", [(31, 7), (55, 7), (100, 8)])
def test_leaf_path_without_duplicates(oracle, k, p_len):
    """Every k-mer distinct (no coverage): the rounds of a leaf overflow their tables and are split on further bits."""
    p = Params(k=k, cutoff_min=1, lut_prefix_len=p_len)
    b = synth_bin(5, k, 20000, genome_len=4_000_000, err=0.0)
    ctx = _ctx(p)
    r = ctx.process_bin(_to_skb(b))
    e = oracle.process_bin(b, p)
    assert r.stats == e.stats and np.array_equal(r.lut, e.lut) and r.payload.tobytes() == e.payload
    ctx.close()


@pytest.mark.parametrize("flow", ["scatter", "filter"])
@pytest.mark.parametrize("k,both,p_len,max_block,max_chunk", [(31, True, 7, 150000, 1 << 18), (55, True, 7, 400000, 1 << 17), (31, False, 3, 1 << 30, 1 << 17), (70, True, 6, 90000, 1 << 18), (31, True, 7, 3000, 1 << 18)])
def test_oversized_bin_in_key_blocks(oracle, monkeypatch, flow, k, both, p_len, max_block, max_chunk):
    """A bin with more k-mers than one sort may take (or too many bytes): expanded chunk by chunk, counted key block by key block
    (limits lowered through the environment so that ~1.3 M k-mers already need ~10-30 blocks and ~6-12 chunks); the result must not change."""
    monkeypatch.setenv("KMCB200_MAX_BLOCK_RECORDS", str(max_block))
    monkeypatch.setenv("KMCB200_MAX_CHUNK_BYTES", str(max_chunk))
    monkeypatch.setenv("KMCB200_KEY_BLOCKS", flow)          # scatter: one expansion into per-block regions; filter: one filtered expansion per block
    p = Params(k=k, both_strands=both, cutoff_min=2, lut_prefix_len=p_len)
    _check_bin(oracle, synth_bin(77 + k, k, 110000, genome_len=60000, err=0.01), p)


def test_expand_matches_oracle(oracle):
    import torch
    for k, both in [(31, True), (31, False), (55, True), (100, True), (9, True)]:
        p = Params(k=k, both_strands=both, lut_prefix_len=choose_lut_prefix_len(k))
        b = synth_bin(3, k, 5000, genome_len=4000, pad_garbage=True)
        ctx = _ctx(p)
        d_bin = torch.zeros(b.size + 64, dtype=torch.uint8, device="cuda")
        d_bin[:b.size] = torch.from_numpy(b.data).cuda()
        d_recs = torch.zeros((b.n_rec + 8) * p.words, dtype=torch.int64, device="cuda")
        d_res = torch.zeros(8, dtype=torch.int64, device="cuda")
        ctx.dev_expand(0, d_bin.data_ptr(), b.size, b.n_rec, b.pack_bytes, d_recs.data_ptr(), d_res.data_ptr(), torch.cuda.current_stream().cuda_stream)
        torch.cuda.synchronize()
        got = d_recs.cpu().numpy().view(np.uint64)[:b.n_rec * p.words].reshape(b.n_rec, p.words)
        exp = oracle.expand(b, p)
        assert int(d_res[6]) == 0
        assert np.array_equal(got, exp), "k=%d both=%s" % (k, both)
        ctx.close()


@pytest.mark.parametrize("mode", ["hybrid", "lsd"])
@pytest.mark.parametrize("words,key_bytes,n", [(1, 8, 100000), (1, 8, 4096), (1, 8, 4097), (1, 5, 33333), (1, 1, 1000), (2, 14, 50001), (2, 16, 2048), (3, 20, 30000), (4, 32, 20000), (1, 8, 1), (1, 8, 3),
                                               (1, 8, 700001), (2, 14, 300000), (3, 23, 150000), (4, 32, 120000)])
def test_sort_records_matches_oracle(oracle, monkeypatch, mode, words, key_bytes, n):
    monkeypatch.setenv("KMCB200_SORT", "lsd" if mode == "lsd" else "msd")
    rng = np.random.default_rng(n + words)
    recs = rng.integers(0, 1 << 63, size=(n, words), dtype=np.uint64)
    # duplicate-rich + masked to the key bytes (bytes above key_bytes are zero in KMC records)
    recs[n // 2:] = recs[rng.integers(0, max(n // 2, 1), n - n // 2)]
    full = np.zeros((n, words * 8), dtype=np.uint8)
    full[:, :key_bytes] = recs.view(np.uint8).reshape(n, words * 8)[:, :key_bytes]
    recs = full.view(np.uint64).reshape(n, words)
    k = {1: 31, 2: 55, 3: 90, 4: 128}[words]
    p = Params(k=k, lut_prefix_len=choose_lut_prefix_len(k))
    ctx = _ctx(p)
    got = ctx.sort_records(recs, key_bytes)
    exp = oracle.sort(recs, key_bytes)
    assert np.array_equal(got, exp)
    ctx.close()


def test_count_matches_oracle_runs_across_tiles(oracle):
    """Runs longer than a tile (giant runs need the backward probe + binary search), cutoffs and clamping."""
    import torch
    rng = np.random.default_rng(5)
    for cmin, cmax, cntmax in [(1, 10 ** 9, 255), (2, 10 ** 9, 255), (3, 50, 7), (1, 20000, 65535), (2, 10 ** 9, 1)]:
        p = Params(k=31, cutoff_min=cmin, cutoff_max=cmax, counter_max=cntmax, lut_prefix_len=7)
        keys = np.sort(rng.integers(0, 1 << 62, 3000, dtype=np.uint64))
        reps = rng.integers(1, 6, keys.size)
        reps[100] = 9000
        reps[101] = 4096
        reps[2000] = 70000
        reps[2999] = 5000
        recs = np.repeat(keys, reps).reshape(-1, 1)
        n = recs.shape[0]
        exp = oracle.compact(recs, p)
        ctx = _ctx(p)
        d = torch.from_numpy(recs.view(np.int64)).cuda()
        cap = ctx.out_capacity(n) + 64
        d_out = torch.zeros(cap, dtype=torch.uint8, device="cuda")
        d_lut = torch.zeros(ctx.lut_entries, dtype=torch.int64, device="cuda")
        d_res = torch.zeros(8, dtype=torch.int64, device="cuda")
        ctx.dev_count(0, d.data_ptr(), n, d_out.data_ptr(), cap, d_lut.data_ptr(), d_res.data_ptr(), torch.cuda.current_stream().cuda_stream)
        torch.cuda.synchronize()
        res = d_res.cpu().numpy()
        assert tuple(int(x) for x in res[:4]) == exp.stats
        nb = int(res[4]) * ctx.out_rec_bytes
        assert d_out[:nb].cpu().numpy().tobytes() == exp.payload
        assert np.array_equal(d_lut.cpu().numpy().view(np.uint64), exp.lut)
        ctx.close()


def test_edge_bins(oracle):
    p = Params(k=31, cutoff_min=1, lut_prefix_len=7)
    ctx = _ctx(p)
    rng = np.random.default_rng(0)
    # empty bin (kb_reader.h:198-205)
    _check_bin(oracle, synth_bin(1, 31, 0), p, ctx)
    # a single k-mer; maximum-length super-k-mers (k+255 symbols); poly-A (one giant run, palindromic ties AT)
    _check_bin(oracle, pack_superkmers(31, [rng.integers(0, 4, 31)]), p, ctx)
    _check_bin(oracle, pack_superkmers(31, [rng.integers(0, 4, 31 + 255) for _ in range(300)]), p, ctx)
    _check_bin(oracle, pack_superkmers(31, [np.zeros(31 + 255, dtype=np.uint8) for _ in range(200)]), p, ctx)
    _check_bin(oracle, pack_superkmers(31, [np.tile(np.array([0, 3], dtype=np.uint8), 100)[:31 + 150] for _ in range(50)]), p, ctx)
    # ragged: many a=0 records
    _check_bin(oracle, pack_superkmers(31, [rng.integers(0, 4, 31) for _ in range(5000)]), p, ctx)
    ctx.close()


def test_reference_kats_through_gpu(oracle):
    """The reference's own CLI known-answers (tests/golden/kats.json, made from .github/workflows/main.yml:35-52)."""
    import json, os
    from kmc_testlib import decode_payload
    kats = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "kats.json")))
    for kat in kats:
        p = Params(k=kat["k"], cutoff_min=kat["cutoff_min"], lut_prefix_len=kat["lut_prefix_len"])
        b = bin_from_reads(kat["k"], kat["reads"])
        ctx = _ctx(p)
        r = ctx.process_bin(_to_skb(b))
        assert r.n_total == kat["n_total"]
        if "dump" in kat:
            assert decode_payload(r.payload.tobytes(), r.lut, p) == [tuple(x) for x in kat["dump"]]
        ctx.close()


def test_pipelined_slots_and_reuse(oracle):
    """Several bins of different sizes through 2 slots (submit/wait), buffers reused and regrown."""
    import kmc_b200
    p = Params(k=31, cutoff_min=2, lut_prefix_len=7)
    ctx = _ctx(p, n_slots=2)
    bins = [synth_bin(100 + i, 31, n, genome_len=max(2000, n), err=0.01) for i, n in enumerate([3000, 50, 12000, 0, 7000, 1])]
    outs = [np.zeros(ctx.out_capacity(b.n_rec) + 64, dtype=np.uint8) for b in bins]
    luts = [np.zeros(ctx.lut_entries, dtype=np.uint64) for _ in bins]
    res = [None] * len(bins)
    for i, b in enumerate(bins):
        slot = i % 2
        if i >= 2:
            res[i - 2] = ctx.wait_bin(slot)
        d = np.ascontiguousarray(b.data)
        ctx.submit_bin(slot, d.ctypes.data, d.size, b.n_rec, np.ascontiguousarray(b.pack_bytes), outs[i].ctypes.data, outs[i].size, luts[i].ctypes.data)
        bins[i].data = d
    for i in range(len(bins) - 2, len(bins)):
        res[i] = ctx.wait_bin(i % 2)
    for i, b in enumerate(bins):
        e = oracle.process_bin(b, p)
        nb, stats = res[i]
        assert stats == e.stats and outs[i][:nb].tobytes() == e.payload and np.array_equal(luts[i], e.lut)
    ctx.close()


def test_bad_packs_are_reported():
    import kmc_b200
    p = Params(k=31, lut_prefix_len=7)
    b = synth_bin(1, 31, 500)
    ctx = _ctx(p)
    skb = _to_skb(b)
    bad = skb.pack_bytes.copy()
    if bad.size == 1:
        bad = np.array([bad[0] - 3, 3], dtype=np.uint64)      # second pack starts in the middle of a record
    skb.pack_bytes = bad
    with pytest.raises(kmc_b200.KmcB200Error) as ei:
        ctx.process_bin(skb)
    assert ei.value.code == kmc_b200.ERR_BIN_FORMAT
    ctx.close()


def test_large_bin_properties_and_parity(oracle):
    """2^22 k-mers (oracle finishes in seconds) bit-exact; then 2^26 (BASELINE config 2) through size-independent
    properties: n_total, sum of LUT == emitted records, emitted records strictly increasing, counters within cutoffs."""
    import kmc_b200
    p = Params(k=31, cutoff_min=2, lut_prefix_len=7)
    ctx = _ctx(p)
    _check_bin(oracle, fast_bin(12345, 31, 1 << 22), p, ctx)
    sk = fast_bin(999, 31, 1 << 26)
    r = ctx.process_bin(sk)
    assert r.n_total == 1 << 26
    n_emit = r.payload.size // ctx.out_rec_bytes
    assert int(r.lut.sum()) == n_emit == r.n_unique - r.n_cutoff_min - r.n_cutoff_max
    rec = r.payload.reshape(n_emit, ctx.out_rec_bytes)
    cnt = rec[:, -1]
    assert cnt.min() >= 2
    # full k-mer = (prefix from the LUT, suffix bytes): strictly increasing
    prefix = np.repeat(np.arange(ctx.lut_entries, dtype=np.uint64), r.lut.astype(np.int64))
    suf = np.zeros(n_emit, dtype=np.uint64)
    for j in range(6):
        suf = (suf << np.uint64(8)) | rec[:, j].astype(np.uint64)
    full = (prefix << np.uint64(48)) | suf
    assert np.all(full[1:] > full[:-1])
    ctx.close()


def test_dropin_inside_reference_pipeline(oracle):
    """The host shim (kmc_b200/host/kb_sorter_b200.h) compiled INSIDE the reference tree: the reference's own reader stand-in,
    CMemoryBins arena, CBinQueue, CSortersManager and CKmerQueue drive CKmerBinSorterB200 instead of CKmerBinSorter
    (oracle/ref/ref_harness.cpp, sort_kind=2); what the completer stand-in pops must equal the CPU reference's output."""
    import os
    from kmc_testlib import Reference, REF_B200_SO
    if not os.path.exists(REF_B200_SO):
        pytest.skip("oracle/_ref/libkmc_ref_b200.so not built")
    Rg = Reference(with_b200=True)
    for k, both, cmin in [(31, True, 2), (55, True, 1), (28, False, 1)]:
        p = Params(k=k, both_strands=both, cutoff_min=cmin, lut_prefix_len=choose_lut_prefix_len(k))
        bins = [synth_bin(300 + i, k, n, genome_len=max(n, 500)) for i, n in enumerate([4000, 0, 900, 15000, 1])]
        got, _ = Rg.process_bins(bins, p, n_sorters=2, sort_kind=Reference.B200_DROPIN)
        cpu, _ = Rg.process_bins(bins, p, n_sorters=2, sort_kind=Reference.RADULS)
        for b, g, c in zip(bins, got, cpu):
            assert g.same_as(c)
            assert g.same_as(oracle.process_bin(b, p))


@pytest.mark.parametrize("kind", ["one_leaf", "heavy_key", "two_level_skew"])
def test_skewed_keys_fall_back_to_lsd(oracle, kind):
    """Leaves that do not fit on chip raise the device flag; the LSD passes queued behind the hybrid path then sort the bin."""
    rng = np.random.default_rng(9)
    n = 300000
    if kind == "one_leaf":            # all keys share their top 16 bits
        recs = (rng.integers(0, 1 << 40, n, dtype=np.uint64) | (np.uint64(0x2A5B) << np.uint64(46))).reshape(-1, 1)
    elif kind == "heavy_key":         # one key holds a third of the bin, the rest is uniform
        recs = rng.integers(0, 1 << 62, n, dtype=np.uint64)
        recs[: n // 3] = recs[0]
        recs = rng.permutation(recs).reshape(-1, 1)
    else:                             # uniform first digit, second digit constant
        recs = (rng.integers(0, 1 << 62, n, dtype=np.uint64) & ~(np.uint64(0xFF) << np.uint64(46))).reshape(-1, 1)
    p = Params(k=31, lut_prefix_len=7)
    ctx = _ctx(p)
    got = ctx.sort_records(recs, 8)
    assert np.array_equal(got, oracle.sort(recs, 8))
    ctx.close()


def test_leaf_count_crowded_leaf_and_heavy_kmer(oracle):
    """A leaf with far more distinct k-mers than one round of the leaf table holds (counted in several rounds), plus a k-mer
    that occurs 50 000 times, inside a bin large enough for the hybrid MSD path."""
    rng = np.random.default_rng(12)
    k = 31
    head = np.array([0, 1, 2, 3, 0, 1, 2, 3], dtype=np.uint8)                     # same first 8 symbols = same leaf (-b mode: no canonicalisation)
    crowded = [np.concatenate([head, rng.integers(0, 4, k - 8)]) for _ in range(9000)]
    heavy_one = np.concatenate([head[::-1], rng.integers(0, 4, k - 8)])
    heavy = [heavy_one.copy() for _ in range(50000)]
    rest = [rng.integers(0, 4, k + 40) for _ in range(3000)]
    p = Params(k=k, both_strands=False, cutoff_min=1, lut_prefix_len=7)
    _check_bin(oracle, pack_superkmers(k, crowded + heavy + rest), p)


# ----------------------------------------------------------------------------------------------------------------------
# Round 2: parity at benchmark scale, against the reference itself: what the unmodified CKmerBinSorter<SIZE>::ProcessBins + RADULS
# returned for these bins is stored in tests/golden/reference_results.json ("gpu_parity", made by tests/golden/make_reference_results.py)
BENCHMARK_SCALE_CASES = [(31, 7), (55, 7)]


def benchmark_scale_bin(k):
    return fast_bin(2600 + k, k, 1 << 26)


def second_level_bin():
    return fast_bin(117, 31, 117_000_000)


@pytest.mark.parametrize("k,p_len", BENCHMARK_SCALE_CASES)
def test_benchmark_scale_bit_exact_vs_reference(k, p_len):
    """One bin of 2^26 k-mers (BASELINE configs[1] / the benchmark's bin size): payload, LUT and statistics byte for byte
    against the unmodified CKmerBinSorter<SIZE>::ProcessBins + RADULS (k=55: against the reference's (k,x)-mer path)."""
    p = Params(k=k, cutoff_min=2, lut_prefix_len=p_len)
    ctx = _ctx(p)
    r = ctx.process_bin(benchmark_scale_bin(k))
    assert result_digest(r) == reference_results("gpu_parity")["bin_2^26_k%d_p%d" % (k, p_len)], "k=%d" % k
    assert r.n_total == 1 << 26
    ctx.close()


def test_large_second_level_bit_exact_vs_reference():
    """A bin of the target workload's size (1.2e8 k-mers: 9-bit second partition level, 2^17 leaves) against the reference."""
    p = Params(k=31, cutoff_min=2, lut_prefix_len=7)
    ctx = _ctx(p)
    r = ctx.process_bin(second_level_bin())
    assert result_digest(r) == reference_results("gpu_parity")["bin_117M_k31_p7"]
    ctx.close()


def _golden():
    import glob, os
    return sorted(glob.glob(os.path.join(os.path.dirname(__file__), "golden", "bins_*.npz")))


@pytest.mark.parametrize("path", _golden(), ids=[__import__("os").path.basename(p)[5:-4] for p in _golden()])
def test_golden_fixtures_through_gpu(path):
    """The committed reference-generated vectors (tests/golden/make_golden.py), expected bytes straight from the fixture."""
    from test_oracle_golden import load_golden
    prm, b, payload, lut, stats = load_golden(path)
    ctx = _ctx(prm)
    r = ctx.process_bin(b)
    assert r.stats == stats and np.array_equal(r.lut, lut) and r.payload.tobytes() == payload
    ctx.close()


@pytest.mark.parametrize("kind", ["all_distinct", "coverage_2x", "coverage_2x_ci1"])
def test_low_coverage_bins_2_24(oracle, kind):
    """2^24 k-mers with (nearly) no duplicates / coverage 2: the rounds of the leaf tables overflow and are split, nothing or
    half of the k-mers survive the cutoff - the opposite regime of the 30x benchmark bins."""
    n = 1 << 24
    if kind == "all_distinct":
        b, p = fast_bin(51, 31, n, genome_len=4 * n, err_ppm=0), Params(k=31, cutoff_min=1, lut_prefix_len=7)
    elif kind == "coverage_2x":
        b, p = fast_bin(52, 31, n, genome_len=n // 2), Params(k=31, cutoff_min=2, lut_prefix_len=7)
    else:
        b, p = fast_bin(53, 31, n, genome_len=n // 2), Params(k=31, cutoff_min=1, lut_prefix_len=11)
    _check_bin(oracle, b, p)


def test_key_blocks_equal_one_shot_2_27(monkeypatch):
    """2^27 k-mers: the oversized-bin path (key blocks of <= 2^24 k-mers, 16 MiB chunks) must give the bytes of the one-shot path."""
    p = Params(k=31, cutoff_min=2, lut_prefix_len=7)
    b = fast_bin(4711, 31, 1 << 27)
    ctx = _ctx(p)
    a = ctx.process_bin(b)
    ctx.close()
    monkeypatch.setenv("KMCB200_MAX_BLOCK_RECORDS", str(1 << 24))
    monkeypatch.setenv("KMCB200_MAX_CHUNK_BYTES", str(1 << 24))
    for flow in ("scatter", "filter"):
        monkeypatch.setenv("KMCB200_KEY_BLOCKS", flow)
        ctx = _ctx(p)
        c = ctx.process_bin(b)
        ctx.close()
        assert a.n_total == 1 << 27 and a.stats == c.stats and np.array_equal(a.lut, c.lut) and a.payload.tobytes() == c.payload.tobytes(), flow


def test_wrong_n_rec_is_fatal_on_the_device(oracle):
    """ADVICE r1: a bin that holds MORE k-mers than n_rec says (buffers are sized from n_rec) must stop on the device - no kernel
    behind the index may touch the records - and the context must stay usable."""
    import kmc_b200
    p = Params(k=31, cutoff_min=1, lut_prefix_len=7)
    ctx = _ctx(p, n_slots=2)
    good = synth_bin(5, 31, 9000, genome_len=20000)
    for n_true, n_claimed in [(300000, 100000), (300000, 299999), (100000, 300000), (2_000_000, 70000)]:
        b = fast_bin(77, 31, n_true)
        lie = kmc_b200.SuperKmerBin(data=b.data, n_rec=n_claimed, pack_bytes=b.pack_bytes, n_super_kmers=b.n_super_kmers, kmer_len=31)
        with pytest.raises(kmc_b200.KmcB200Error) as ei:
            ctx.process_bin(lie)
        assert ei.value.code == kmc_b200.ERR_BIN_FORMAT
        _check_bin(oracle, good, p, ctx)                 # neighbouring allocations were not scribbled on
    # a pack boundary in the middle of a record, in a bin large enough for the hybrid path
    b = fast_bin(78, 31, 400000)
    bad = b.pack_bytes.copy()
    bad[0] -= 3
    bad[1] += 3
    with pytest.raises(kmc_b200.KmcB200Error) as ei:
        ctx.process_bin(kmc_b200.SuperKmerBin(data=b.data, n_rec=b.n_rec, pack_bytes=bad, kmer_len=31))
    assert ei.value.code == kmc_b200.ERR_BIN_FORMAT
    _check_bin(oracle, good, p, ctx)
    _check_bin(oracle, b, p, ctx)
    ctx.close()


def test_one_byte_records(oracle):
    """ADVICE r1: k - p = 4 with counter_max = 1 -> emitted records of ONE byte (no counter); leaves that emit many records."""
    p = Params(k=13, cutoff_min=1, counter_max=1, lut_prefix_len=9)
    assert p.out_rec_bytes == 1
    _check_bin(oracle, fast_bin(13, 13, 300000, genome_len=100000), p)
    p = Params(k=17, both_strands=False, cutoff_min=1, counter_max=1, lut_prefix_len=13)
    _check_bin(oracle, fast_bin(17, 17, 200000, genome_len=150000), p)


@pytest.mark.parametrize("k,p_len", [(31, 7), (55, 7)])
def test_lsd_fallback_is_one_cooperative_launch(oracle, monkeypatch, k, p_len):
    """The device-flagged fallback (a leaf that cannot be counted on chip) through the whole-bin path: same bytes as the oracle.
    k = 31: 70000 copies of one k-mer are handled inside the leaf kernel since round 2 (dominant-k-mer path); k = 55 (wide records: the entry
    holds a 16-bit record index) still takes the fallback."""
    rng = np.random.default_rng(4)
    heavy_one = rng.integers(0, 4, k)
    heavy = [heavy_one.copy() for _ in range(70000)]               # one k-mer 70000 times: beyond a warp-counted leaf
    rest = [rng.integers(0, 4, k + 60) for _ in range(4000)]
    p = Params(k=k, both_strands=False, cutoff_min=1, lut_prefix_len=p_len)
    b = pack_superkmers(k, heavy + rest)
    ctx = _ctx(p)
    r = ctx.process_bin(_to_skb(b))
    e = oracle.process_bin(b, p)
    assert r.stats == e.stats and np.array_equal(r.lut, e.lut) and r.payload.tobytes() == e.payload
    ctx.close()
    monkeypatch.setenv("KMCB200_SORT", "lsd")                      # and the plain LSD sort (the same cooperative kernel, always on)
    _check_bin(oracle, fast_bin(9, 31, 250000), Params(k=31, cutoff_min=2, lut_prefix_len=7))


@pytest.mark.parametrize("k,both,cmin,p_len,n", [(31, True, 2, 7, 300000), (31, False, 1, 11, 200000), (55, True, 2, 7, 150000), (70, True, 1, 6, 90000), (128, True, 1, 8, 60000),
                                                 (17, True, 1, 5, 250000), (9, True, 1, 5, 120000), (31, True, 2, 7, 3_000_000)])
def test_fused_expansion_option(oracle, monkeypatch, k, both, cmin, p_len, n):
    """KMCB200_EXPAND=fused: walk, look-back and rolling expansion in one kernel per pack (expand_fused.cuh), aligned level-1 cells."""
    monkeypatch.setenv("KMCB200_EXPAND", "fused")
    p = Params(k=k, both_strands=both, cutoff_min=cmin, lut_prefix_len=p_len)
    _check_bin(oracle, fast_bin(900 + k, k, n), p)
    ctx = _ctx(p)                                   # malformed bins are stopped on the device in this path too
    import kmc_b200
    b = fast_bin(901, k, 200000)
    with pytest.raises(kmc_b200.KmcB200Error) as ei:
        ctx.process_bin(kmc_b200.SuperKmerBin(data=b.data, n_rec=150000, pack_bytes=b.pack_bytes, kmer_len=k))
    assert ei.value.code == kmc_b200.ERR_BIN_FORMAT
    _check_bin(oracle, synth_bin(5, k, 5000, genome_len=20000), p, ctx)
    ctx.close()


@pytest.mark.parametrize("k,p_len,n,n_ctx", [(31, 7, 3_000_000, 2), (31, 7, 1_500_000, 3), (55, 7, 1_200_000, 2), (17, 5, 900_000, 4)])
def test_one_bin_split_over_several_gpus(oracle, monkeypatch, k, p_len, n, n_ctx):
    """kmcb200_process_bin_multi (SURVEY 8f N2): contiguous key ranges per GPU, the bin bytes travel by peer copies, outputs concatenated in
    key order - byte-identical to one GPU.  Distinct devices when the box has them, otherwise several contexts on device 0; the block limit
    is lowered so that every GPU's range itself needs several key blocks."""
    import torch
    import kmc_b200
    monkeypatch.setenv("KMCB200_MAX_BLOCK_RECORDS", str(max(n // 7, 1024)))
    p = Params(k=k, cutoff_min=2, lut_prefix_len=p_len)
    n_dev = torch.cuda.device_count()
    sp = kmc_b200.Stage2Params(p.k, p.both_strands, p.cutoff_min, p.cutoff_max, p.counter_max, p.lut_prefix_len)
    ctxs = [kmc_b200.Stage2Context(sp, device=(g % n_dev), n_slots=1) for g in range(n_ctx)]
    b = fast_bin(600 + k, k, n)
    r = kmc_b200.Stage2Context.process_bin_multi(ctxs, b)
    e = oracle.process_bin(b, p)
    assert r.stats == e.stats and np.array_equal(r.lut, e.lut) and r.payload.tobytes() == e.payload
    # a malformed bin is reported, and the contexts stay usable
    with pytest.raises(kmc_b200.KmcB200Error):
        kmc_b200.Stage2Context.process_bin_multi(ctxs, kmc_b200.SuperKmerBin(data=b.data, n_rec=b.n_rec - 5, pack_bytes=b.pack_bytes, kmer_len=k))
    r2 = ctxs[-1].process_bin(b)
    assert r2.payload.tobytes() == e.payload
    for c in ctxs:
        c.close()


@pytest.mark.parametrize("k,both,cmin,p_len,n", [(31, True, 2, 7, 400000), (55, True, 1, 7, 150000), (17, False, 1, 5, 200000), (128, True, 1, 8, 50000)])
def test_indexed_submit_needs_no_walk(oracle, k, both, cmin, p_len, n):
    """kmcb200_submit_bin_indexed (SURVEY 8f N4): stage 1 hands over the length bytes as a separate array; the index is two prefix sums per
    pack.  Same bytes as the walk; an array that disagrees with the stream is a bin-format error."""
    import kmc_b200
    from kmc_testlib import bin_extras
    p = Params(k=k, both_strands=both, cutoff_min=cmin, lut_prefix_len=p_len)
    b = fast_bin(700 + k, k, n)
    extras, psk = bin_extras(b)
    ctx = _ctx(p, n_slots=2)
    e = oracle.process_bin(b, p)
    cap = ctx.out_capacity(b.n_rec) + 64
    out = np.zeros(cap, dtype=np.uint8)
    lut = np.zeros(ctx.lut_entries, dtype=np.uint64)
    data = np.ascontiguousarray(b.data)
    l0 = ctx.kernel_launches()
    ctx.submit_bin_indexed(0, data.ctypes.data, data.size, b.n_rec, np.ascontiguousarray(b.pack_bytes), extras, psk, out.ctypes.data, cap, lut.ctypes.data)
    nbytes, stats = ctx.wait_bin(0)
    assert stats == e.stats and out[:nbytes].tobytes() == e.payload and np.array_equal(lut, e.lut)
    # wrong arrays: a length byte off by one / a record moved to the neighbouring pack
    bad = extras.copy()
    bad[len(bad) // 2] ^= 1
    for ex, ps in [(bad, psk)] + ([(extras, psk + np.array([1, -1] + [0] * (psk.size - 2)).astype(np.uint32))] if psk.size >= 2 else []):
        ctx.submit_bin_indexed(1, data.ctypes.data, data.size, b.n_rec, np.ascontiguousarray(b.pack_bytes), ex, ps, out.ctypes.data, cap, lut.ctypes.data)
        with pytest.raises(kmc_b200.KmcB200Error) as ei:
            ctx.wait_bin(1)
        assert ei.value.code == kmc_b200.ERR_BIN_FORMAT
    _check_bin(oracle, b, p, ctx)                  # and the walk path on the same context still works
    ctx.close()


@pytest.mark.parametrize("cmin,cmax,cntmax", [(2, 10 ** 9, 255), (1, 100000, 65535), (3, 10 ** 9, 10 ** 6)])
def test_dominant_kmers_are_counted_inside_the_leaf_kernel(oracle, cmin, cmax, cntmax):
    """Real genomes: poly-A / satellite k-mers with 10^5..10^6 copies.  One-word records: the copies of the dominant k-mer of a large leaf are
    counted by comparison and enter the table once; the bin must NOT take the LSD fallback (result[7] = 0) unless the rest of the leaf is too
    large as well.  Cases: a 300 000-copy k-mer with a 40 000-copy neighbour in the same leaf; a dominant k-mer that is not the first record
    of its leaf; cutoffs / counter clamps that the big counts cross."""
    import torch
    rng = np.random.default_rng(8)
    k = 31
    head = np.array([0, 1, 2, 3, 0, 1, 2, 3, 1], dtype=np.uint8)                     # same first 9 symbols = same leaf (-b mode)
    big = np.concatenate([head, rng.integers(0, 4, k - 9)])
    second = np.concatenate([head, rng.integers(0, 4, k - 9)])
    other_head = np.array([3, 2, 1, 0, 3, 2, 1, 0, 2], dtype=np.uint8)
    late = np.concatenate([other_head, rng.integers(0, 4, k - 9)])
    # every record is one super-k-mer of exactly k symbols; order inside the bin is what the leaf sees (the partition is not stable, but
    # "not the first record" holds with overwhelming probability when 3000 other k-mers of the leaf come first)
    lists = ([np.concatenate([other_head, rng.integers(0, 4, k - 9)]) for _ in range(3000)] + [late.copy() for _ in range(120000)]
             + [big.copy() for _ in range(300000)] + [second.copy() for _ in range(40000)]
             + [np.concatenate([head, rng.integers(0, 4, k - 9)]) for _ in range(5000)] + [rng.integers(0, 4, k + 40) for _ in range(20000)])
    p = Params(k=k, both_strands=False, cutoff_min=cmin, cutoff_max=cmax, counter_max=cntmax, lut_prefix_len=7)
    b = pack_superkmers(k, lists)
    ctx = _ctx(p)
    e = oracle.process_bin(b, p)
    r = ctx.process_bin(_to_skb(b))
    assert r.stats == e.stats and np.array_equal(r.lut, e.lut) and r.payload.tobytes() == e.payload
    # the device-level call exposes result[7]: no fallback for this bin
    d_bin = torch.zeros(b.size + 64, dtype=torch.uint8, device="cuda"); d_bin[:b.size] = torch.from_numpy(b.data).cuda()
    cap = ctx.out_capacity(b.n_rec) + 64
    d_out = torch.zeros(cap, dtype=torch.uint8, device="cuda"); d_lut = torch.zeros(ctx.lut_entries, dtype=torch.int64, device="cuda"); d_res = torch.zeros(8, dtype=torch.int64, device="cuda")
    ctx.dev_process_bin(0, d_bin.data_ptr(), b.size, b.n_rec, b.pack_bytes, d_out.data_ptr(), cap, d_lut.data_ptr(), d_res.data_ptr(), torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    res = d_res.cpu().numpy()
    assert tuple(int(x) for x in res[:4]) == e.stats
    ctx.close()
