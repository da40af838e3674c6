"""The bins bench.py times, compared with the reference byte for byte through every entry point the benchmark uses.

bench.py checks its timed steps only against its own warm-up run (the eight counters of the result row, and on the host-buffer path the
k-mer count and output size).  Here every one of its bins - the eight pool bins of the k=31 workload and the bins of its secondary block -
is compared with what the unmodified reference (CKmerBinSorter<SIZE>::ProcessBins + RADULS) returned for it: payload, LUT and statistics,
stored in tests/golden/reference_results.json ("benchmark_bins", made by tests/golden/make_reference_results.py, which also checks every
k=31 result against the oracle).  The inputs are generated here from the same seeds; each entry also stores a SHA-256 of its input, so
that a generator that draws differently on another machine is reported as a different input, not as a wrong result.
"""
import os
from concurrent.futures import ThreadPoolExecutor
from dataclasses import dataclass

import hashlib
import numpy as np
import pytest

import bench
from kmc_testlib import Oracle, Params, fast_bin, reference_results, result_digest

GROUP = "benchmark_bins"
POOL_SEED = 4000                 # bench.make_pool: pool bin j is gen_bin(4000 + j, K, pool_sizes(scale)[j])
N26, N28 = 1 << 26, 1 << 28      # bench.secondary_block at scale 1


def bench_params(k=bench.K, cutoff_min=bench.CUTOFF_MIN):
    return Params(k=k, cutoff_min=cutoff_min, cutoff_max=bench.CUTOFF_MAX, counter_max=bench.COUNTER_MAX, lut_prefix_len=bench.LUT_P)


@dataclass(frozen=True)
class Case:
    gen: str                     # "gen_bin" (bench.gen_bin: independent 2^24-k-mer pieces) or "fast_bin" (one piece)
    seed: int
    k: int
    n: int
    cutoff_min: int = bench.CUTOFF_MIN
    gen_kw: tuple = ()           # extra fast_bin arguments, as (name, value) pairs

    @property
    def params(self):
        return bench_params(self.k, self.cutoff_min)

    @property
    def key(self):
        p = self.params
        args = ",".join(["%d" % x for x in (self.seed, self.k, self.n)] + ["%s=%d" % kv for kv in self.gen_kw])
        return "%s(%s) %s ci=%d cx=%d cs=%d p=%d" % (self.gen, args, "canonical" if p.both_strands else "-b", p.cutoff_min, p.cutoff_max,
                                                    p.counter_max, p.lut_prefix_len)

    def make(self, pool=None):
        if self.gen == "gen_bin":
            return bench.gen_bin(self.seed, self.k, self.n, pool)
        return fast_bin(self.seed, self.k, self.n, **dict(self.gen_kw))


POOL = [Case("gen_bin", POOL_SEED + j, bench.K, n) for j, n in enumerate(bench.pool_sizes(1))]
# bench.secondary_block (bench.py:373-378): two configs[1] bins, two all-distinct bins (also one at ci=1: every k-mer is emitted), configs[3]
DISTINCT_KW = (("genome_len", 2 * N26 + 1000), ("err_ppm", 0))
SECONDARY = [Case("gen_bin", 1000, 31, N26), Case("gen_bin", 1017, 31, N26),
             Case("fast_bin", 2000, 31, N26, gen_kw=DISTINCT_KW), Case("fast_bin", 2001, 31, N26, gen_kw=DISTINCT_KW),
             Case("fast_bin", 2000, 31, N26, cutoff_min=1, gen_kw=DISTINCT_KW),
             Case("gen_bin", 3000, 55, N28)]
K55 = SECONDARY[-1]
ALL_CASES = POOL + SECONDARY


def input_sha256(b):
    """SHA-256 of what a bin is as input: its bytes, then its pack sizes (little-endian uint64)."""
    h = hashlib.sha256(np.ascontiguousarray(b.data))
    h.update(np.ascontiguousarray(b.pack_bytes, dtype="<u8"))
    return h.hexdigest()


def stored(case):
    return reference_results(GROUP)[case.key]


def check_input(case, b):
    assert b.n_rec == case.n
    assert input_sha256(b) == stored(case)["input_sha256"], (
        "%s: the input differs from the bin the reference was run on (the synthetic generator draws differently here); "
        "this says nothing about the kernels" % case.key)


def check_result(case, r):
    assert result_digest(r) == stored(case)["result"], case.key


# ---------------------------------------------------------------------------------------------------------------- CPU
def test_every_benchmark_bin_has_a_stored_reference_result():
    """A change to bench.py's pool or to these cases that did not regenerate reference_results.json fails here, not on the GPU."""
    sizes = bench.pool_sizes(1)
    assert [c.n for c in POOL] == sizes and [c.n >> 20 for c in POOL] == bench.POOL_MI
    group = reference_results(GROUP)
    for c in ALL_CASES:
        assert c.key in group, c.key
        e = group[c.key]
        assert len(e["input_sha256"]) == 64 and e["result"]["stats"][3] == c.n, c.key
    assert set(group) == {c.key for c in ALL_CASES}


def test_pool_seeds_are_the_benchmarks():
    """POOL_SEED restates a literal of bench.make_pool: at a tiny scale the benchmark's own pool is gen_bin(POOL_SEED + j, ...)."""
    scale = 1 << 13
    ours = [bench.gen_bin(POOL_SEED + j, bench.K, n) for j, n in enumerate(bench.pool_sizes(scale))]
    for a, b in zip(bench.make_pool(scale, threads=2), ours):
        assert a.n_rec == b.n_rec and input_sha256(a) == input_sha256(b)


def test_smallest_pool_bins_generate_identically_and_oracle_agrees():
    """The generator gives the stored inputs on this machine, and the oracle's result for the 32 Mi pool bin is the reference's."""
    small = sorted(POOL, key=lambda c: c.n)[:2]
    with ThreadPoolExecutor(min(16, os.cpu_count() or 4)) as ex:
        bins = [c.make(ex) for c in small]
    for c, b in zip(small, bins):
        check_input(c, b)
    check_result(small[0], Oracle().process_bin(bins[0], small[0].params))


# ---------------------------------------------------------------------------------------------------------------- GPU
class BinCache:
    """Every bin generated once per module (pieces on a thread pool, as bench.make_pool does), its input checked before first use."""

    def __init__(self):
        self.ex = ThreadPoolExecutor(max(1, min(32, os.cpu_count() or 8)))
        self.bins = {}

    def __call__(self, case):
        if case not in self.bins:
            b = case.make(self.ex)
            check_input(case, b)
            self.bins[case] = b
        return self.bins[case]


@pytest.fixture(scope="module")
def bins():
    c = BinCache()
    yield c
    c.ex.shutdown()


def _ctx(p, n_slots=1):
    import kmc_b200
    return kmc_b200.Stage2Context(kmc_b200.Stage2Params(p.k, p.both_strands, p.cutoff_min, p.cutoff_max, p.counter_max, p.lut_prefix_len),
                                  device=0, n_slots=n_slots)


def _as_result(payload, lut, stats):
    import kmc_b200
    return kmc_b200.BinResult(payload, lut, *[int(x) for x in stats])


def pool_order():
    """The pool largest-first (bench.py's LPT order on one GPU), then the first 16 bins of the workload: sizes go down, then up and down."""
    from kmc_b200.sharding import assign_bins
    return assign_bins([c.n for c in POOL], 1)[0] + bench.workload_bins()[:16]


@pytest.mark.gpu
def test_resident_path_as_the_benchmark_runs_it(bins):
    """kmcb200_dev_process_bin on a non-default stream, one 3-slot context for every bin (bench.py's `value`), output, LUT and result
    row overwritten with garbage before every call."""
    import torch
    dev = torch.device("cuda", 0)
    ctx = _ctx(bench_params(), n_slots=bench.E2E_SLOTS)
    tstream = torch.cuda.Stream(device=dev)
    assert tstream.cuda_stream != 0
    d_pool = {}
    d_out = torch.empty(ctx.out_capacity(max(c.n for c in POOL)) + 64, dtype=torch.uint8, device=dev)
    d_lut = torch.empty(ctx.lut_entries, dtype=torch.int64, device=dev)
    d_res = torch.empty(8, dtype=torch.int64, device=dev)
    garbage = torch.tensor([0x5A5A5A5A5A5A5A5A, -1, 7, 1 << 40, 123456789, 1, 2, 3], dtype=torch.int64, device=dev)
    for j in pool_order():
        case = POOL[j]
        b = bins(case)
        with torch.cuda.stream(tstream):
            if j not in d_pool:
                t = torch.zeros(b.size + 64, dtype=torch.uint8, device=dev)
                t[:b.size] = torch.from_numpy(b.data).to(dev)
                d_pool[j] = t
            d_out.fill_(0xFF)
            d_lut.fill_(-1)
            d_res.copy_(garbage)
        ctx.dev_process_bin(0, d_pool[j].data_ptr(), b.size, b.n_rec, b.pack_bytes, d_out.data_ptr(), ctx.out_capacity(b.n_rec) + 64,
                            d_lut.data_ptr(), d_res.data_ptr(), tstream.cuda_stream)
        tstream.synchronize()
        res = d_res.cpu().numpy()
        assert res[3] == b.n_rec and res[5] == 0 and res[6] == 0, "pool bin %d: %s" % (j, res)
        payload = d_out[:int(res[4]) * ctx.out_rec_bytes].cpu().numpy()
        check_result(case, _as_result(payload, d_lut.cpu().numpy().view(np.uint64), res[:4]))
    ctx.close()


@pytest.mark.gpu
@pytest.mark.parametrize("overlap_walk", ["1", "0"])
def test_host_buffer_pipeline_as_the_benchmark_runs_it(bins, monkeypatch, overlap_walk):
    """kmcb200_submit_bin / kmcb200_wait_bin with three bins in flight and pinned host buffers (bench.py's `e2e`), slot buffers regrown
    as sizes go up and down; the index kernels of the next bin on the copy stream (KMCB200_OVERLAP_WALK=1, the default) or on the compute
    stream.  Every third bin is collected with kmcb200_wait_bin_scanned: its LUT arrives as the exclusive prefix sum plus a base."""
    import torch
    monkeypatch.setenv("KMCB200_OVERLAP_WALK", overlap_walk)
    n_slots = bench.E2E_SLOTS
    ctx = _ctx(bench_params(), n_slots=n_slots)
    cap = ctx.out_capacity(max(c.n for c in POOL)) + 64
    pin_pool = {}
    pin_out = [torch.empty(cap, dtype=torch.uint8).pin_memory() for _ in range(n_slots)]
    pin_lut = [torch.empty(ctx.lut_entries, dtype=torch.int64).pin_memory() for _ in range(n_slots)]
    seq = pool_order()
    base = 12345                             # records before this bin in the database, as the completer's running total would be

    def collect(i):
        nonlocal base
        s, case = i % n_slots, POOL[seq[i]]
        scanned = i % 3 == (i // 3) % n_slots            # every third bin, over all slots in turn
        nb, stats = ctx.wait_bin_scanned(s, base) if scanned else ctx.wait_bin(s)
        assert nb % ctx.out_rec_bytes == 0
        n_emit = nb // ctx.out_rec_bytes
        lut = pin_lut[s].numpy().view(np.uint64).copy()
        if scanned:
            assert lut[0] == base and np.all(lut[1:] >= lut[:-1]) and lut[-1] <= base + n_emit, "bin %d: not an exclusive scan from %d" % (i, base)
            lut = np.diff(np.append(lut, np.uint64(base + n_emit)))
        base += n_emit
        check_result(case, _as_result(pin_out[s][:nb].numpy(), lut, stats))

    for i, j in enumerate(seq):
        s = i % n_slots
        if i >= n_slots:
            collect(i - n_slots)
        b = bins(POOL[j])
        if j not in pin_pool:
            pin_pool[j] = torch.from_numpy(b.data.copy()).pin_memory()
        pin_out[s].fill_(0xFF)
        pin_lut[s].fill_(-1)
        ctx.submit_bin(s, pin_pool[j].data_ptr(), b.size, b.n_rec, b.pack_bytes, pin_out[s].data_ptr(), ctx.out_capacity(b.n_rec) + 64,
                       pin_lut[s].data_ptr())
    for i in range(max(len(seq) - n_slots, 0), len(seq)):
        collect(i)
    ctx.close()


@pytest.mark.gpu
@pytest.mark.parametrize("case", SECONDARY, ids=[c.key.split(" ")[0] + "_ci%d" % c.cutoff_min for c in SECONDARY])
def test_secondary_bins(bins, case):
    """bench.py's secondary block: configs[1] (2^26, 30x), all-distinct 2^26 (nothing survives ci=2; everything survives ci=1) and configs[3]
    (k=55, 2^28 k-mers: two-word records, >= 4 GiB of them, the 1024-digit second level and leaf_hash_wide_kernel on 2^18 leaves)."""
    ctx = _ctx(case.params)
    check_result(case, ctx.process_bin(bins(case)))
    ctx.close()


MAX_BLOCK = 1 << 28                           # the 256 Mi pool bin has exactly this many k-mers: one over the oversized threshold, and at it
KNOBS_K31 = [{}, {"KMCB200_LEAF_KERNEL": "warp"}, {"KMCB200_LEAF": "sort"}, {"KMCB200_LEAF_MAX_B2": "8"}, {"KMCB200_LEAF_MAX_B2": "10"},
             {"KMCB200_EXPAND": "fused"}, {"KMCB200_SORT": "lsd"},
             {"KMCB200_MAX_BLOCK_RECORDS": str(MAX_BLOCK - 1), "KMCB200_KEY_BLOCKS": "scatter"},
             {"KMCB200_MAX_BLOCK_RECORDS": str(MAX_BLOCK - 1), "KMCB200_KEY_BLOCKS": "filter"},
             {"KMCB200_MAX_BLOCK_RECORDS": str(MAX_BLOCK)}]
KNOBS_K55 = [{}, {"KMCB200_LEAF_WIDE": "warp"}, {"KMCB200_L2_BITS": "9"}]
_knob_id = lambda env: ",".join("%s=%s" % (k[8:], v) for k, v in env.items()) or "default"


@pytest.mark.gpu
@pytest.mark.parametrize("case,env", [(POOL[0], e) for e in KNOBS_K31] + [(K55, e) for e in KNOBS_K55],
                         ids=["k31_256Mi-" + _knob_id(e) for e in KNOBS_K31] + ["k55_2^28-" + _knob_id(e) for e in KNOBS_K55])
def test_knobs_at_full_size(bins, monkeypatch, case, env):
    """Every kernel choice and limit the library exposes gives the reference's bytes on the largest bins the benchmark times."""
    assert POOL[0].n == MAX_BLOCK
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    ctx = _ctx(case.params)
    check_result(case, ctx.process_bin(bins(case)))
    ctx.close()
