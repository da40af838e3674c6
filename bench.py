#!/usr/bin/env python
"""bench.py — stage-2 k-mers/s (k=31) of the B200 path on BASELINE.json's target workload, next to the reference's CPU stage 2.

Workload (BASELINE configs[2], SURVEY 8d "config 3"): 512 bins of a 30x human-like run, ~6.1e10 k-mers in total, k=31 canonical,
ci=2 cx=1e9 cs=255 p=7.  The 512 bins are drawn from a pool of 8 distinct synthetic bins (kb_collector format, ~12 k-mers per
super-k-mer, 30x duplicate-rich, 1 % substitutions) whose sizes are spread Zipf-like over 2^25 .. 2^28 k-mers (mean 1.2e8, so the
9-bit second partition level is the common case).  A "step" = all 512 bins once.  STRONG scaling: the bins are sharded over the
ranks in the reference's order - descending size, each to the least-loaded rank (kmc_b200.sharding.assign_bins = LPT, what N sorter
objects pulling from one CBinQueue in get_sorted_req_sizes order converge to; kmc_core/kmc.h:1564-1600, queues.h:499-558) - and no
collective touches the data path.

  value     : total k-mers of the step / device time of the slowest rank, bins resident in HBM (CUDA events on the launching stream)
  e2e       : the same through the host-buffer C ABI (kmcb200_submit_bin / kmcb200_wait_bin, three bins in flight), pinned host
              buffers, H2D of every bin and D2H of its database records + LUT + counters inside the timed region
  roofline  : the stage with the largest share of the step (CUDA-event intervals of every pool bin, weighted by the workload),
              algorithmic bytes / interval; `passes` holds the same for every radix (MSD partition) pass - the metric's second half
  secondary : BASELINE configs[1] (one 2^26 bin), all-distinct keys, configs[3] (k=55, 2^28 k-mers per bin) and the seam-1 sort of
              2^26 uniform keys against RADULS alone - N=1 only
  cpu_baseline / --impl reference : the UNMODIFIED reference classes (oracle/_ref: CKmerBinSorter<1>::ProcessBins + RADULS) on the
              host cores over a bounded, size-stratified sample of the SAME 512 bins; the warm-up steps sweep the reference's
              concurrency (arena size = bins in flight, sorter threads) and the timed steps use the best setting

Usage: python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--scale S] [--no-cpu] [--no-secondary] [--dump-outputs DIR]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time
from concurrent.futures import ThreadPoolExecutor

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

K = 31
LUT_P = 7
CUTOFF_MIN, CUTOFF_MAX, COUNTER_MAX = 2, 10 ** 9, 255
METRIC = "stage-2 k-mers/s (k=31)"
UNIT = "k-mers/s"
REC_BYTES = 8
KEY_BYTES = 8
OUT_REC_BYTES = 7                      # (31 - 7) / 4 suffix bytes + 1 counter byte
E2E_SLOTS = int(os.environ.get("KMCB200_E2E_SLOTS", "3"))
MI = 1 << 20
POOL_MI = [256, 192, 160, 128, 112, 96, 64, 32]        # k-mers per pool bin, in Mi
POOL_COUNT = [24, 40, 56, 72, 96, 96, 80, 48]          # how often each occurs among the 512 bins (Zipf-like: few large, many small)
N_BINS = sum(POOL_COUNT)
GEN_CHUNK = 1 << 24


def hbm_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


# ------------------------------------------------------------------------------------------------ workload
def pool_sizes(scale):
    return [max(m * MI // scale, 4096) for m in POOL_MI]


def workload_bins():
    """pool index of each of the 512 bins (bin ids interleave the sizes, as signatures do in a real run)."""
    left = list(POOL_COUNT)
    out = []
    while len(out) < N_BINS:
        for j in range(len(left)):
            if left[j]:
                left[j] -= 1
                out.append(j)
    return out


def gen_bin(seed, k, n_rec, pool=None):
    """One bin of exactly n_rec k-mers, generated in independent 2^24-k-mer pieces (each its own 30x genome; packs never straddle pieces)."""
    import numpy as np
    from kmc_testlib import fast_bin, Bin
    pieces = []
    left, i = n_rec, 0
    while left > 0:
        c = min(left, GEN_CHUNK)
        pieces.append((seed * 1000 + i, c))
        left -= c
        i += 1
    fn = lambda sc: fast_bin(sc[0], k, sc[1])
    parts = list(pool.map(fn, pieces)) if pool is not None else [fn(p) for p in pieces]
    if len(parts) == 1:
        return parts[0]
    return Bin(data=np.concatenate([p.data for p in parts]), n_rec=n_rec, n_super_kmers=sum(p.n_super_kmers for p in parts),
               pack_bytes=np.concatenate([p.pack_bytes for p in parts]), pack_recs=np.concatenate([p.pack_recs for p in parts]), k=k)


def make_pool(scale, threads=None):
    threads = threads or max(1, min(32, (os.cpu_count() or 8) // max(1, int(os.environ.get("LOCAL_WORLD_SIZE", "1")))))
    with ThreadPoolExecutor(threads) as ex:
        return [gen_bin(4000 + j, K, n, ex) for j, n in enumerate(pool_sizes(scale))]


def workload_config(scale, n_gpus, sizes):
    total = sum(sizes[j] * c for j, c in enumerate(POOL_COUNT))
    return {
        "workload": "BASELINE configs[2]: k=31 canonical, %d bins (~30x human), %.3g k-mers per step, ci=2 cx=1e9 cs=255 p=7" % (N_BINS, total),
        "n_bins": N_BINS, "kmers_per_step": total, "record_bytes": REC_BYTES, "key_bytes": KEY_BYTES,
        "bin_pool_kmers": sizes, "bin_pool_count": POOL_COUNT, "scale_divisor": scale,
        "bin": "synthetic super-k-mers (kb_collector format), ~12 k-mers/super-k-mer, 30x duplicate-rich, 1% substitutions",
        "sharding": "LPT over descending bin size (kmc_b200.sharding.assign_bins), %d rank(s), no collective on the data path" % n_gpus,
        "l2": "every bin's working set (2 record buffers of 8 B x 3e7..2.7e8 records) >> 126 MB L2; consecutive bins differ",
    }


class ClockSampler:
    """nvidia-smi clocks/throttle reasons DURING the timed region."""
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.index = index
        self.lines = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons, pw = [], [], set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for l in self.lines:
            f = [x.strip() for x in l.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1])); pw.append(float(f[2]))
            except ValueError:
                continue
            for n, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_min_mhz": min(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "power_w_median": statistics.median(pw) if pw else None,
                "samples": len(sm), "reasons": sorted(reasons)}


# ------------------------------------------------------------------------------------------------ reference arm
def reference_lib():
    from kmc_testlib import Reference, reference_available, ensure_reference_built
    if not (reference_available() or ensure_reference_built()):
        return None
    return Reference()


def mem_available_gb():
    try:
        for l in open("/proc/meminfo"):
            if l.startswith("MemAvailable"):
                return int(l.split()[1]) / 1e6
    except Exception:
        pass
    return 64.0


def ref_params():
    from kmc_testlib import Params
    return Params(k=K, cutoff_min=CUTOFF_MIN, cutoff_max=CUTOFF_MAX, counter_max=COUNTER_MAX, lut_prefix_len=LUT_P)


def stratified_sample(bin_pool_idx, sizes, n_sample):
    """n_sample of the 512 bins, evenly spaced over the size-sorted list: the sample keeps the workload's size distribution."""
    order = sorted(range(len(bin_pool_idx)), key=lambda b: (-sizes[bin_pool_idx[b]], b))
    n_sample = max(1, min(n_sample, len(order)))
    return [order[(2 * i + 1) * len(order) // (2 * n_sample)] for i in range(n_sample)]


def cpu_plan(R, prm, pool, sizes, seconds_per_step, cores):
    """How many of the 512 bins one reference step takes: a probe gives the rate, the time budget gives the k-mers, RAM caps the arena."""
    bins_idx = workload_bins()
    probe = [pool[-1]] * max(1, min(cores // 8, 16))                      # the smallest pool bin, as many as get ~8 threads each
    arena_gb = max(8.0, 0.6 * mem_available_gb())
    os.environ["KMCREF_ARENA_GB"] = "%d" % int(arena_gb)
    R.process_bins(probe, prm, n_sorters=cores)                           # faults the arena in
    t0 = time.perf_counter()
    R.process_bins(probe, prm, n_sorters=cores)
    rate = sum(b.n_rec for b in probe) / (time.perf_counter() - t0)
    mean = sum(sizes[j] for j in bins_idx) / len(bins_idx)
    n_sample = int(rate * seconds_per_step / mean)
    n_sample = max(4, min(n_sample, N_BINS))
    # ~18 bytes of arena per k-mer (2 record arrays + bin bytes + output): keep the whole sample in flight when RAM allows
    while n_sample > 4 and n_sample * mean * 18 / 1e9 > arena_gb:
        n_sample -= 1
    ids = stratified_sample(bins_idx, sizes, n_sample)
    return ids, [pool[bins_idx[b]] for b in ids], arena_gb, rate


def run_reference(R, prm, bins, cores, steps, warmup, arena_gb, sweep=True):
    """A sweep over the reference's concurrency (arena size = how many bins it holds at once, like kmc's -m; sorter threads) picks
    the best setting; then `warmup` untimed and `steps` timed steps with it.  Every setting runs twice and the second run counts:
    a new arena is page-faulted in by its first user."""
    total = sum(b.n_rec for b in bins)
    settings = [(1.0, cores), (0.5, cores), (1.0, max(cores // 2, 1)), (1.0, cores * 2)] if sweep else [(1.0, cores)]
    tried = []
    for frac, ns in settings:
        agb = max(4, int(arena_gb * frac))
        os.environ["KMCREF_ARENA_GB"] = "%d" % agb
        for rep in range(2 if sweep else 0):
            _, (wall, _) = R.process_bins(bins, prm, n_sorters=ns)
        if sweep:
            tried.append({"arena_gb": agb, "n_sorters": ns, "k-mers/s": total / wall})
    if tried:
        b = max(tried, key=lambda t: t["k-mers/s"])
        agb, ns = b["arena_gb"], b["n_sorters"]
    else:
        agb, ns = max(4, int(arena_gb)), cores
    os.environ["KMCREF_ARENA_GB"] = "%d" % agb
    for i in range(max(warmup, 1)):
        R.process_bins(bins, prm, n_sorters=ns)
    times = []
    for i in range(steps):
        _, (wall, _) = R.process_bins(bins, prm, n_sorters=ns)
        times.append(wall)
    return total, times, tried, {"arena_gb": agb, "n_sorters": ns}


def cpu_baseline_block(pool, sizes, seconds=14.0):
    """Reported beside the GPU number (rank 0, N=1): the unmodified reference on the box's host cores, bounded sample of the same bins."""
    R = reference_lib()
    cores = os.cpu_count() or 1
    if R is None:
        return {"value": None, "unit": UNIT, "cores": cores, "kind": "reference", "sample": "oracle/_ref not available on this box"}
    prm = ref_params()
    ids, bins, arena_gb, _ = cpu_plan(R, prm, pool, sizes, seconds / 2, cores)
    total, times, _, best = run_reference(R, prm, bins, cores, 1, 1, arena_gb, sweep=False)
    return {"value": total / times[0], "unit": UNIT, "cores": cores, "kind": "reference",
            "sample": "%d of the %d bins (size-stratified, %.3g k-mers) through the unmodified CKmerBinSorter<1>::ProcessBins + RADULS AVX2 (oracle/_ref), n_sorters=%d, arena %d GB, wall %.2f s"
                      % (len(bins), N_BINS, total, best["n_sorters"], best["arena_gb"], times[0])}


def main_reference(args, rank, world):
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    sizes = pool_sizes(args.scale)
    base = {"impl": "reference", "metric": METRIC, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "u64", "data": "synthetic",
            "config": workload_config(args.scale, args.gpus, sizes)}
    R = reference_lib()
    if R is None:
        base["unavailable"] = "oracle/_ref/libkmc_ref.so was not built (needs /root/reference at build time)"
        print(json.dumps(base))
        return
    pool = make_pool(args.scale)
    prm = ref_params()
    budget = 170.0 / (args.steps + max(args.warmup, 1) + 8)          # 8 = the sweep: 4 settings, twice each
    ids, bins, arena_gb, probe_rate = cpu_plan(R, prm, pool, sizes, budget, cores)
    total, times, tried, best = run_reference(R, prm, bins, cores, args.steps, args.warmup, arena_gb)
    t = sum(times)
    value = total * args.steps / t
    sample = ("per step %d of the %d bins (size-stratified: every %d-th of the size-sorted list, %.3g k-mers), unmodified CKmerBinSorter<1>::ProcessBins + "
              "RADULS AVX2 (oracle/_ref), best setting of the sweep: n_sorters=%d, arena %d GB" % (len(bins), N_BINS, max(N_BINS // len(bins), 1), total, best["n_sorters"], best["arena_gb"]))
    base.update({"value": value, "ms_per_step": 1e3 * t / args.steps,
                 "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "reference", "sample": sample},
                 "cpu_sweep": tried, "cpu_best": best,
                 "step_spread": {"min_s": min(times), "median_s": statistics.median(times), "max_s": max(times)},
                 "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                 "gpu_launches": 0})
    print(json.dumps(base))


# ------------------------------------------------------------------------------------------------ our arm
STAGE_BYTES = {      # algorithmic bytes of a stage for a bin of N k-mers, S bin bytes, U emitted records (SURVEY 8d; DESIGN section 3)
    "expand": lambda N, S, U, W: S + N * W,
    "msd_scan_L1": lambda N, S, U, W: 0,
    "msd_partition_L1": lambda N, S, U, W: 2 * N * W,
    "msd_count_L2": lambda N, S, U, W: N * W,
    "msd_partition_L2": lambda N, S, U, W: 2 * N * W,
    "leaf_count": lambda N, S, U, W: N * W + U * (OUT_REC_BYTES if W == 8 else 13),
    "lsd_fallback(all passes)": lambda N, S, U, W: 0,
}


def stage_profile(ctx, torch, dev, stream, run_one, pool_bins, weights, W):
    """CUDA-event intervals (recorded by the library on the launching stream) of one pass over every pool bin."""
    acc, alg = {}, {}
    for j, b in enumerate(pool_bins):
        res = run_one(j)
        torch.cuda.synchronize()
        st = ctx.stage_times(0)
        U = int(res[4])
        iv = {"expand": st["expand_ms"]}
        for nm, x in zip(st["pass_names"], st["pass_ms"]):
            iv[nm] = iv.get(nm, 0.0) + x
        known = sum(iv.values())
        iv["other"] = max(st["expand_ms"] + st["sort_ms"] + st["count_ms"] - known, 0.0)
        for nm, x in iv.items():
            acc[nm] = acc.get(nm, 0.0) + weights[j] * x
            f = STAGE_BYTES.get(nm)
            alg[nm] = alg.get(nm, 0.0) + weights[j] * (f(b.n_rec, b.size, U, W) if f else 0)
    return acc, alg


def secondary_block(kmc_b200, torch, dev, tstream, args, peak):
    """N=1 only: BASELINE configs[1], all-distinct keys, configs[3] (k=55), seam-1 sort vs RADULS alone."""
    import numpy as np
    out = {}
    stream = tstream.cuda_stream
    n26 = max((1 << 26) // args.scale, 4096)
    n28 = max((1 << 28) // args.scale, 4096)

    def one(k, p, bins, label, W, reps=5):
        ctx = kmc_b200.Stage2Context(kmc_b200.Stage2Params(k, True, CUTOFF_MIN, CUTOFF_MAX, COUNTER_MAX, p), device=dev.index, n_slots=1)
        n_rec = bins[0].n_rec
        cap = ctx.out_capacity(n_rec) + 64
        d_bins = []
        for b in bins:
            t = torch.zeros(b.size + 64, dtype=torch.uint8, device=dev)
            t[:b.size] = torch.from_numpy(b.data).to(dev)
            d_bins.append(t)
        d_out = torch.zeros(cap, dtype=torch.uint8, device=dev)
        d_lut = torch.zeros(ctx.lut_entries, dtype=torch.int64, device=dev)
        d_res = torch.zeros(8, dtype=torch.int64, device=dev)
        run = lambda i: ctx.dev_process_bin(0, d_bins[i % len(bins)].data_ptr(), bins[i % len(bins)].size, n_rec, bins[i % len(bins)].pack_bytes,
                                            d_out.data_ptr(), cap, d_lut.data_ptr(), d_res.data_ptr(), stream)
        for i in range(3):
            run(i)
        torch.cuda.synchronize()
        r = d_res.cpu().numpy()
        assert int(r[3]) == n_rec and int(r[5]) == 0 and int(r[6]) == 0, "%s: %s" % (label, r)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(reps):
            run(3 + i)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / reps
        st = ctx.stage_times(0)
        iv = {}
        for nm, x in zip(st["pass_names"], st["pass_ms"]):
            iv[nm] = iv.get(nm, 0.0) + x
        passes = {nm: {"ms": x, "GB/s": 2.0 * n_rec * W / (x * 1e-3) / 1e9, "frac_of_peak": 2.0 * n_rec * W / (x * 1e-3) / 1e9 / peak}
                  for nm, x in iv.items() if nm.startswith("msd_partition") and x > 0}
        res = {"workload": label, "value": n_rec / (ms * 1e-3), "unit": UNIT, "ms_per_bin": ms, "n_rec": n_rec, "record_bytes": W,
               "emitted_records": int(r[4]), "lsd_fallback_taken": int(r[7]),
               "stage_ms": {"expand": st["expand_ms"], "sort": st["sort_ms"], "count": st["count_ms"]}, "sort_intervals_ms": iv, "radix_passes": passes}
        ctx.close()
        del d_bins, d_out
        torch.cuda.empty_cache()
        return res

    from kmc_testlib import fast_bin
    with ThreadPoolExecutor(min(16, os.cpu_count() or 8)) as ex:
        out["config1_k31_one_bin_2^26"] = one(31, 7, [gen_bin(1000, 31, n26, ex), gen_bin(1017, 31, n26, ex)],
                                              "BASELINE configs[1]: k=31, one bin of %d k-mers, 30x duplicate-rich" % n26, 8)
        distinct = [fast_bin(2000 + j, 31, n26, genome_len=2 * n26 + 1000, err_ppm=0) for j in range(2)]
        out["k31_all_distinct_2^26"] = one(31, 7, distinct, "k=31, one bin of %d k-mers, every k-mer (nearly) distinct: coverage 1, nothing survives ci=2" % n26, 8)
        del distinct
        out["config3_k55_2^28"] = one(55, 7, [gen_bin(3000, 55, n28, ex)], "BASELINE configs[3]: k=55 (two-word records, expanded to plain k-mers), one bin of %d k-mers" % n28, 16, reps=3)
    # seam #1: the sort alone on 2^26 uniform 64-bit keys (configs[1] literally: "2^26 packed 64-bit k-mers" = k = 32) - device-resident and
    # through the host-buffer call - vs RADULS alone.  (Keys that leave the top bits of their key bytes unused make the first MSD level
    # coarser: seam #1 takes the significant bits from key_bytes, not from k.)
    ctx = kmc_b200.Stage2Context(kmc_b200.Stage2Params(32, True, CUTOFF_MIN, CUTOFF_MAX, COUNTER_MAX, 8), device=dev.index, n_slots=1)
    rng = np.random.default_rng(12345)
    keys = (rng.integers(0, 1 << 63, size=n26, dtype=np.uint64) * np.uint64(2) + rng.integers(0, 2, size=n26, dtype=np.uint64)).reshape(-1, 1)
    d_a = torch.from_numpy(keys.view(np.int64)).to(dev)
    d_in = torch.empty_like(d_a); d_tmp = torch.empty_like(d_a)
    ms_l = []
    for i in range(5):
        d_in.copy_(d_a)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        where = ctx.dev_sort(0, d_in.data_ptr(), d_tmp.data_ptr(), n26, 8, False, stream)
        e1.record()
        torch.cuda.synchronize()
        ms_l.append(e0.elapsed_time(e1))
    got = (d_tmp if where == 1 else d_in).cpu().numpy().view(np.uint64).reshape(-1)
    assert bool(np.all(got[1:] >= got[:-1])) and int(got.sum(dtype=np.uint64)) == int(keys.sum(dtype=np.uint64)), "seam-1 sort is wrong"
    t0 = time.perf_counter()
    ctx.sort_records(keys, 8)
    t_host = time.perf_counter() - t0
    sort = {"workload": "kmcb200_dev_sort / kmcb200_sort_records, %d uniform 64-bit keys (k = 32: 8-byte records, 8 key bytes)" % n26,
            "dev_ms": min(ms_l[1:]), "dev_keys_per_s": n26 / (min(ms_l[1:]) * 1e-3), "host_call_s": t_host, "host_call_keys_per_s": n26 / t_host}
    R = reference_lib()
    if R is not None and not args.no_cpu:
        cores = os.cpu_count() or 1
        best = None
        for thr in sorted({cores, max(cores // 2, 1), max(cores // 4, 1), min(16, cores)}):
            _, sec = R.sort(keys, 8, n_threads=thr)
            if best is None or sec < best[1]:
                best = (thr, sec)
        sort["raduls_avx2_s"] = best[1]
        sort["raduls_avx2_threads"] = best[0]
        sort["raduls_avx2_keys_per_s"] = n26 / best[1]
        sort["dev_vs_raduls"] = best[1] / (min(ms_l[1:]) * 1e-3)
    out["seam1_sort_2^26_uniform"] = sort
    ctx.close()
    return out


DUMP_RECORDS = 1 << 17          # sampled records per pool bin: 8 bins x 2^17 x 4 float64 = 32 MiB of the 64 MiB a dump may take


def dump_outputs(out_dir, torch, dev, out_rec_bytes, my, bin_pool_idx, last_rows, d_outs, d_luts):
    """--dump-outputs: what kmcb200_dev_process_bin returned in the last timed step, as float64 .npy files, so that two builds can be
    compared output for output (the inputs depend only on the arguments).
      bin_results.npy   one row per bin of the step in processing order: bin id, pool bin, then the 8 values of d_result
                        (n_unique, n_cutoff_min, n_cutoff_max, n_total, emitted records, capacity error, format error bits, LSD fallback)
      lut_<j>.npy       LUT of pool bin j: emitted records per k-mer prefix of LUT_P symbols
      records_<j>.npy   emitted records of pool bin j, a fixed sample (seed j) of at most DUMP_RECORDS: record index, prefix (from the
                        LUT), suffix ((K - LUT_P) / 4 bytes, big-endian) and counter (little-endian)
    Every occurrence of pool bin j in the step writes the same buffers, so the last one's output is pool bin j's output."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    save = lambda name, a: np.save(os.path.join(out_dir, name + ".npy"), np.asarray(a, dtype=np.float64))
    save("bin_results", [[bid, bin_pool_idx[bid]] + [int(x) for x in r] for bid, r in zip(my, last_rows)])
    suffix_bytes = (K - LUT_P) // 4
    for j in sorted({bin_pool_idx[bid] for bid in my}):
        n = int(next(r[4] for bid, r in zip(my, last_rows) if bin_pool_idx[bid] == j))
        lut = d_luts[j].cpu().numpy()
        assert int(lut.sum()) == n, "pool bin %d: LUT holds %d records, the result row %d" % (j, int(lut.sum()), n)
        idx = np.sort(np.random.default_rng(j).choice(n, size=min(n, DUMP_RECORDS), replace=False))
        recs = d_outs[j][:n * out_rec_bytes].view(n, out_rec_bytes)[torch.from_numpy(idx).to(dev)].cpu().numpy().astype(np.uint64)
        suffix = np.zeros(idx.size, dtype=np.uint64)
        for c in range(suffix_bytes):
            suffix = (suffix << np.uint64(8)) | recs[:, c]
        counter = np.zeros(idx.size, dtype=np.uint64)
        for c in range(out_rec_bytes - 1, suffix_bytes - 1, -1):
            counter = (counter << np.uint64(8)) | recs[:, c]
        prefix = np.searchsorted(np.cumsum(lut), idx, side="right")
        save("lut_%d" % j, lut)
        save("records_%d" % j, np.stack([idx, prefix, suffix, counter], axis=1))


_ORIG_AFFINITY = None


def unbind():
    """Back to all the host cores (the CPU legs of the bench must not inherit the GPU arm's binding)."""
    if _ORIG_AFFINITY:
        os.sched_setaffinity(0, _ORIG_AFFINITY)


def bind_to_gpu_numa_node(local_rank):
    """Run this rank (and therefore allocate its pinned host buffers) on the CPUs next to its GPU: with 8 ranks feeding 8 PCIe links the
    host-to-device copies otherwise cross the socket interconnect (measured at N=8: 0.71 s per 3 steps on the lucky ranks, 0.86 s on the others)."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(local_rank)
        words = (os.cpu_count() + 63) // 64
        mask = pynvml.nvmlDeviceGetCpuAffinity(h, words)
        cpus = {64 * i + b for i, w in enumerate(mask) for b in range(64) if (int(w) >> b) & 1}
        global _ORIG_AFFINITY
        _ORIG_AFFINITY = set(os.sched_getaffinity(0))
        cpus &= _ORIG_AFFINITY
        if cpus:
            os.sched_setaffinity(0, cpus)
            return sorted(cpus)[0], len(cpus)
    except Exception:
        pass
    return None


def main_ours(args, rank, world, local_rank):
    import numpy as np
    import torch
    import kmc_b200
    from kmc_b200.sharding import assign_bins
    numa = bind_to_gpu_numa_node(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)

    sizes = pool_sizes(args.scale)
    pool = make_pool(args.scale)
    bin_pool_idx = workload_bins()
    costs = [sizes[j] for j in bin_pool_idx]
    shards = assign_bins(costs, world)                       # every rank computes the same assignment: no communication
    my = shards[rank]                                        # bin ids in processing order (largest first)
    my_kmers = sum(costs[b] for b in my)
    total_kmers = sum(costs)
    loads = [sum(costs[b] for b in s) for s in shards]

    ctx = kmc_b200.Stage2Context(kmc_b200.Stage2Params(K, True, CUTOFF_MIN, CUTOFF_MAX, COUNTER_MAX, LUT_P), device=local_rank, n_slots=E2E_SLOTS)
    cap = ctx.out_capacity(max(sizes)) + 64

    # ---- value: the pool resident in HBM; every bin of the shard is one kmcb200_dev_process_bin call with its own result row.
    # Each pool bin has its own output and LUT buffers, so after a step they hold what that step returned for every distinct bin.
    d_pool = []
    for b in pool:
        t = torch.zeros(b.size + 64, dtype=torch.uint8, device=dev)
        t[:b.size] = torch.from_numpy(b.data).to(dev)
        d_pool.append(t)
    d_outs = [torch.zeros(ctx.out_capacity(b.n_rec) + 64, dtype=torch.uint8, device=dev) for b in pool]
    d_luts = [torch.zeros(ctx.lut_entries, dtype=torch.int64, device=dev) for _ in pool]
    n_my = max(len(my), 1)
    d_res = torch.zeros((args.steps + 1) * n_my, 8, dtype=torch.int64, device=dev)
    tstream = torch.cuda.Stream(device=dev)          # a real (non-default) stream: the library enqueues on it, torch events time it
    torch.cuda.set_stream(tstream)
    stream = tstream.cuda_stream
    assert stream != 0

    def run_dev(j, row):
        b = pool[j]
        ctx.dev_process_bin(0, d_pool[j].data_ptr(), b.size, b.n_rec, b.pack_bytes, d_outs[j].data_ptr(), d_outs[j].numel(), d_luts[j].data_ptr(),
                            d_res[row].data_ptr(), stream)

    def step_dev(s):
        for i, bid in enumerate(my):
            run_dev(bin_pool_idx[bid], s * n_my + i)

    def barrier():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    # expected result of every pool bin (one untimed pass; also sizes every workspace)
    expect = []
    for j in range(len(pool)):
        run_dev(j, args.steps * n_my)
        torch.cuda.synchronize()
        r = d_res[args.steps * n_my].cpu().numpy().copy()
        assert int(r[3]) == pool[j].n_rec and int(r[5]) == 0 and int(r[6]) == 0, "pool bin %d failed: %s" % (j, r)
        expect.append(r)
    for s in range(args.warmup):
        step_dev(args.steps)
    barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    launches0 = ctx.kernel_launches()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for s in range(args.steps):
        step_dev(s)
    e1.record()
    barrier()
    dev_ms = e0.elapsed_time(e1)
    launches = ctx.kernel_launches() - launches0
    # every bin of every timed step is checked (not only the warm-up): statistics, emitted records, no error / fallback flag
    res_all = d_res.cpu().numpy()
    fallbacks = 0
    for s in range(args.steps):
        for i, bid in enumerate(my):
            r, e = res_all[s * n_my + i], expect[bin_pool_idx[bid]]
            assert np.array_equal(r[:7], e[:7]), "step %d bin %d: %s != %s" % (s, bid, r, e)
            fallbacks += int(r[7])
    if args.dump_outputs and rank == 0:
        last = args.steps - 1
        dump_outputs(args.dump_outputs, torch, dev, ctx.out_rec_bytes, my, bin_pool_idx, res_all[last * n_my:last * n_my + len(my)], d_outs, d_luts)
    t_dev = torch.tensor([dev_ms], dtype=torch.float64, device=dev)
    if dist is not None:
        all_ms = [torch.zeros_like(t_dev) for _ in range(world)]
        dist.all_gather(all_ms, t_dev)
        rank_ms = [float(x.item()) for x in all_ms]
    else:
        rank_ms = [dev_ms]
    dev_ms = max(rank_ms)
    value = total_kmers * args.steps / (dev_ms * 1e-3)

    # ---- per-stage CUDA-event intervals over the pool, weighted by this workload (rank 0's view is the same on every rank)
    weights = [float(c) for c in POOL_COUNT]
    acc, alg = stage_profile(ctx, torch, dev, stream, lambda j: (run_dev(j, args.steps * n_my), torch.cuda.synchronize(), d_res[args.steps * n_my].cpu().numpy())[2],
                             pool, weights, REC_BYTES)

    # ---- e2e: host buffers through submit/wait, E2E_SLOTS bins in flight, pinned memory
    pin_pool = [torch.from_numpy(b.data.copy()).pin_memory() for b in pool]
    pin_out = [torch.zeros(cap, dtype=torch.uint8).pin_memory() for _ in range(E2E_SLOTS)]
    pin_lut = [torch.zeros(ctx.lut_entries, dtype=torch.int64).pin_memory() for _ in range(E2E_SLOTS)]

    def e2e_run(n_steps):
        moved_in = moved_out = 0
        seq = [bin_pool_idx[bid] for _ in range(n_steps) for bid in my]
        for i, j in enumerate(seq):
            s = i % E2E_SLOTS
            if i >= E2E_SLOTS:
                nb, stats = ctx.wait_bin(s)
                jj = seq[i - E2E_SLOTS]
                assert stats[3] == pool[jj].n_rec and nb == int(expect[jj][4]) * ctx.out_rec_bytes, "e2e bin differs from the resident run"
                moved_out += nb
            b = pool[j]
            ctx.submit_bin(s, pin_pool[j].data_ptr(), b.size, b.n_rec, b.pack_bytes, pin_out[s].data_ptr(), cap, pin_lut[s].data_ptr())
            moved_in += b.size + 8 * (b.pack_bytes.size + 1)
        for i in range(max(len(seq) - E2E_SLOTS, 0), len(seq)):
            nb, stats = ctx.wait_bin(i % E2E_SLOTS)
            assert stats[3] == pool[seq[i]].n_rec
            moved_out += nb
        return moved_in, moved_out + len(seq) * (8 * ctx.lut_entries + 64)

    e2e_run(min(args.warmup, 2))
    barrier()
    t0 = time.perf_counter()
    h2d, d2h = e2e_run(args.steps)
    torch.cuda.synchronize()
    t_e2e = time.perf_counter() - t0
    t_e = torch.tensor([t_e2e], dtype=torch.float64, device=dev)
    if dist is not None:
        all_e = [torch.zeros_like(t_e) for _ in range(world)]
        dist.all_gather(all_e, t_e)
        rank_e2e = [float(x.item()) for x in all_e]
        io = torch.tensor([h2d, d2h], dtype=torch.int64, device=dev)
        dist.all_reduce(io)
        h2d, d2h = int(io[0]), int(io[1])
    else:
        rank_e2e = [t_e2e]
    t_e2e = max(rank_e2e)
    e2e_value = total_kmers * args.steps / t_e2e
    clocks = sampler.stop() if rank == 0 else None          # sampled across both timed regions (device-resident and end-to-end)
    unbind()

    if rank == 0:
        peak, peak_src = hbm_peak()
        tot_ms = sum(acc.values())
        share = {nm: x / tot_ms for nm, x in acc.items()}
        dom = max((nm for nm in acc if nm != "other"), key=lambda nm: acc[nm])
        gbs = lambda nm: alg[nm] / (acc[nm] * 1e-3) / 1e9 if acc.get(nm, 0) > 0 else None
        kernel_names = {"expand": "walk_packs_parallel_kernel + scan_packs_kernel + tile_desc_kernel + expand_kernel<1> (index + expansion of a bin)",
                        "msd_partition_L1": "msd_partition_kernel<1> (level-1 8-bit MSD partition pass)",
                        "msd_partition_L2": "msd_partition_kernel<1,256|1024> (level-2 MSD partition pass, 8-9 bits)",
                        "msd_count_L2": "msd_count_kernel<1> + cell scan (level-2 digit counts)",
                        "leaf_count": "leaf_hash_kernel<10> + leaf_scan/gather (count the leaves, emit the database records)"}
        traffic, traffic_src = None, None
        tp = os.path.join(ROOT, "profiles", "dominant_kernel_traffic.json")
        if os.path.exists(tp):
            try:
                tj = json.load(open(tp))
                if dom in tj.get("stages", {}):
                    traffic = tj["stages"][dom]["dram_bytes_per_launch"]
                    traffic_src = "%s; kernel %s" % (tj.get("source"), tj["stages"][dom].get("kernel"))
            except Exception:
                pass
        n_w = sum(weights)
        passes = {nm: {"ms_per_mean_bin": acc[nm] / n_w, "algorithmic_bytes_per_mean_bin": alg[nm] / n_w, "GB/s": gbs(nm), "frac": gbs(nm) / peak}
                  for nm in acc if nm.startswith("msd_partition") and acc[nm] > 0}
        out = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": dev_ms / args.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "u64", "data": "synthetic", "config": workload_config(args.scale, world, sizes),
            "roofline": {"bound": "hbm", "kernel": kernel_names.get(dom, dom), "stage": dom, "share_of_step": share[dom],
                         "achieved": gbs(dom), "peak": peak, "unit": "GB/s", "frac": gbs(dom) / peak, "traffic": traffic, "traffic_source": traffic_src,
                         "peak_source": peak_src, "algorithmic_bytes_per_launch": alg[dom] / n_w, "avg_launch_ms": acc[dom] / n_w,
                         "how": "CUDA events recorded by the library around every stage of each of the 8 pool bins (after the timed region), weighted by how often the bin occurs among the 512",
                         "passes": passes,
                         "stages": {nm: {"share": share[nm], "ms_per_mean_bin": acc[nm] / n_w, "GB/s": gbs(nm), "frac": (gbs(nm) / peak if gbs(nm) else None)} for nm in acc}},
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d // args.steps, "d2h_bytes_per_step": d2h // args.steps,
                    "ms_per_step": 1e3 * t_e2e / args.steps, "api": "kmcb200_submit_bin/kmcb200_wait_bin, %d slots, pinned host buffers" % E2E_SLOTS,
                    "rank_seconds": rank_e2e, "cpu_binding": ("first cpu %d, %d cpus (GPU's NUMA node)" % numa) if numa else "none"},
            "gpu_launches": launches * world if world > 1 else launches, "gpu_launches_per_bin": launches / max(args.steps * len(my), 1),
            "lsd_fallbacks_taken": fallbacks, "clocks": clocks,
            "ranks": {"bins": [len(s) for s in shards], "kmers": loads, "device_ms": rank_ms,
                      "straggler": "rank %d (%.4g k-mers, %.1f ms); largest bin = %.3g k-mers = %.2f %% of a rank's share"
                                   % (rank_ms.index(max(rank_ms)), loads[rank_ms.index(max(rank_ms))], max(rank_ms), max(sizes), 100.0 * max(sizes) / max(loads))},
            "timed_region_s": {"value": dev_ms * 1e-3, "e2e": t_e2e},
        }
        del d_pool, d_outs
        torch.cuda.empty_cache()
        if world == 1 and not args.no_secondary:
            ctx.close()
            ctx = None
            out["secondary"] = secondary_block(kmc_b200, torch, dev, tstream, args, peak)
        if world == 1 and not args.no_cpu:
            out["cpu_baseline"] = cpu_baseline_block(pool, sizes)
        else:
            out["cpu_baseline"] = {"value": None, "unit": UNIT, "cores": os.cpu_count(), "kind": "reference", "sample": "only measured at N=1"}
        print(json.dumps(out))
    if ctx is not None:
        ctx.close()
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--scale", type=int, default=int(os.environ.get("KMCB200_BENCH_SCALE", "1")), help="divide every bin size by this (development runs)")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg (profiling runs)")
    ap.add_argument("--no-secondary", action="store_true", help="skip the secondary workloads (profiling runs)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step returned to DIR/<name>.npy (see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        main_reference(args, rank, world)
    else:
        main_ours(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
