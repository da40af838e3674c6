"""Shared helpers for the test-suite (TEST INFRASTRUCTURE).

* synthetic bins in KMC's stage-1 output format (kmc_core/kb_collector.cpp:34-90):
  records `[u8 a][ceil((k+a)/4) bytes, 2 bits per symbol, first symbol in bits 7-6]`
* ctypes wrappers for the two checkers:
    - `Oracle`     : oracle/_build/libkmc_oracle.so  (our plain-C restatement)
    - `Reference`  : oracle/_ref/libkmc_ref.so       (the unmodified reference classes, when built)
* what the reference returned for the tests' inputs (tests/golden/reference_results.json, made by
  tests/golden/make_reference_results.py), so that the comparisons with it run without the reference
"""
import ctypes as C
import functools
import hashlib
import json
import os
import subprocess
from dataclasses import dataclass, field

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ORACLE_DIR = os.path.join(ROOT, "oracle")
ORACLE_SO = os.path.join(ORACLE_DIR, "_build", "libkmc_oracle.so")
REF_SO = os.path.join(ORACLE_DIR, "_ref", "libkmc_ref.so")
REF_B200_SO = os.path.join(ORACLE_DIR, "_ref", "libkmc_ref_b200.so")    # same harness, CKmerBinSorterB200 in place of CKmerBinSorter
PACK_BYTES = 1 << 16          # bin_part_size, kmc_core/kmc.h:151
GOLDEN_DIR = os.path.join(ROOT, "tests", "golden")
REFERENCE_RESULTS = os.path.join(GOLDEN_DIR, "reference_results.json")


# ----------------------------------------------------------------------------- parameters
@dataclass
class Params:
    k: int = 31
    both_strands: bool = True
    cutoff_min: int = 2
    cutoff_max: int = 1_000_000_000
    counter_max: int = 255
    lut_prefix_len: int = 7

    def __post_init__(self):
        assert (self.k - self.lut_prefix_len) % 4 == 0, "(k-p) % 4 must be 0 (kmc.h:1434-1469)"

    @property
    def words(self):
        return (self.k + 31) // 32

    @property
    def counter_bytes(self):
        if self.counter_max == 1:
            return 0
        bl = lambda x: 1 if x < 1 << 8 else 2 if x < 1 << 16 else 3 if x < 1 << 24 else 4
        return min(bl(self.cutoff_max), bl(self.counter_max))

    @property
    def out_rec_bytes(self):
        return (self.k - self.lut_prefix_len) // 4 + self.counter_bytes

    @property
    def lut_entries(self):
        return 1 << (2 * self.lut_prefix_len)

    def out_capacity(self, n_rec):
        # kb_reader.h:141-150
        return ((n_rec + 1) // max(self.cutoff_min, 1)) * self.out_rec_bytes


def choose_lut_prefix_len(k, default=7):
    """A legal p for tests: (k-p) % 4 == 0, 2 <= p <= 15 where possible (kmc.h:1452-1466)."""
    for p in (default, 3, 11, 15, 4, 5, 6, 2, 8, 9, 10, 12, 13, 14, 1):
        if p < k and (k - p) % 4 == 0:
            return p
    raise ValueError(k)


# ----------------------------------------------------------------------------- synthetic bins
@dataclass
class Bin:
    data: np.ndarray                 # uint8 bin byte stream
    n_rec: int                       # sum(a+1)
    n_super_kmers: int
    pack_bytes: np.ndarray           # uint64, one per <=64 KiB collector flush
    pack_recs: np.ndarray            # uint64, safe upper bound of (k+x)-mers per pack (= k-mers per pack)
    k: int = 31
    extras: np.ndarray = None        # int64 `a` of every super-k-mer
    pack_first: np.ndarray = None    # index of the first super-k-mer of every pack (+ sentinel)

    @property
    def size(self):
        return int(self.data.size)

    def kx_counts(self, both_strands):
        """(n_plus_x_recs, pack_recs) as stage 1 would report them for the (k,x)-mer path.
        Canonical: a+1 per super-k-mer is a safe upper bound, surplus slots are removed by the expander
        (kb_sorter.h:605-633).  Non-canonical: must be exact, 1 + a/(max_x+1) (kb_collector.cpp:78, kb_sorter.h:640-724)."""
        max_x = 0 if self.k % 32 == 0 else min(31 - self.k % 32, 3)
        if both_strands or max_x == 0 or self.extras is None or self.extras.size == 0:
            return int(self.n_rec), self.pack_recs
        per = 1 + self.extras // (max_x + 1)
        c = np.concatenate([[0], np.cumsum(per)])
        pr = (c[self.pack_first[1:]] - c[self.pack_first[:-1]]).astype(np.uint64)
        return int(per.sum()), pr


def pack_superkmers(k, symbol_lists, pad_garbage_rng=None):
    """symbol_lists: iterable of 1-D integer arrays (values 0..3, length k..k+255) -> Bin."""
    chunks = []
    n_rec = 0
    rec_sizes = []
    for s in symbol_lists:
        s = np.asarray(s, dtype=np.uint8)
        n = s.size
        assert k <= n <= k + 255
        nb = (n + 3) // 4
        pad = np.zeros(nb * 4, dtype=np.uint8)
        if pad_garbage_rng is not None:
            pad[n:] = pad_garbage_rng.integers(0, 4, nb * 4 - n)
        pad[:n] = s
        q = pad.reshape(-1, 4)
        b = (q[:, 0] << 6) | (q[:, 1] << 4) | (q[:, 2] << 2) | q[:, 3]
        chunks.append(np.concatenate([np.array([n - k], dtype=np.uint8), b.astype(np.uint8)]))
        n_rec += n - k + 1
        rec_sizes.append((1 + nb, n - k + 1))
    data = np.concatenate(chunks) if chunks else np.zeros(0, dtype=np.uint8)
    pb, pr, pf = _make_packs(np.array([r[0] for r in rec_sizes], dtype=np.int64), np.array([r[1] for r in rec_sizes], dtype=np.int64))
    return Bin(data=data, n_rec=n_rec, n_super_kmers=len(rec_sizes), pack_bytes=pb, pack_recs=pr, k=k,
               extras=np.array([r[1] - 1 for r in rec_sizes], dtype=np.int64), pack_first=pf)


def _make_packs(rec_bytes, rec_kmers):
    """Group whole records into packs of <= PACK_BYTES bytes (kb_collector.cpp:34-106)."""
    if rec_bytes.size == 0:
        return np.zeros(0, dtype=np.uint64), np.zeros(0, dtype=np.uint64), np.zeros(1, dtype=np.int64)
    ends = np.cumsum(rec_bytes)
    kc = np.cumsum(rec_kmers)
    pb, pr, pf = [], [], [0]
    start_b, start_k, i, n = 0, 0, 0, rec_bytes.size
    while i < n:
        j = int(np.searchsorted(ends, start_b + PACK_BYTES, side="right"))
        j = max(j, i + 1)
        pb.append(int(ends[j - 1]) - start_b)
        pr.append(int(kc[j - 1]) - start_k)
        start_b, start_k, i = int(ends[j - 1]), int(kc[j - 1]), j
        pf.append(j)
    return np.array(pb, dtype=np.uint64), np.array(pr, dtype=np.uint64), np.array(pf, dtype=np.int64)


def synth_bin(seed, k, n_super_kmers, genome_len=None, mean_extra=11.0, err=0.01, max_extra=255,
              both_strand_reads=True, pad_garbage=False):
    """Vectorised synthetic bin: super-k-mers are noisy substrings of a random genome (duplicate-rich when
    n_super_kmers * mean_extra >> genome_len), random strand, `err` substitution rate."""
    rng = np.random.default_rng(seed)
    if n_super_kmers == 0:
        return Bin(np.zeros(0, np.uint8), 0, 0, np.zeros(0, np.uint64), np.zeros(0, np.uint64), k, np.zeros(0, np.int64), np.zeros(1, np.int64))
    if genome_len is None:
        genome_len = max(k + max_extra + 1, int(n_super_kmers * (mean_extra + 1) / 8))
    genome_len = max(genome_len, k + max_extra + 1)
    genome = rng.integers(0, 4, genome_len, dtype=np.uint8)
    a = np.minimum(rng.geometric(1.0 / (mean_extra + 1.0), n_super_kmers) - 1, max_extra).astype(np.int64)
    n = a + k
    pos = rng.integers(0, genome_len - n + 1)
    rc = rng.integers(0, 2, n_super_kmers).astype(bool) if both_strand_reads else np.zeros(n_super_kmers, bool)
    starts = np.concatenate([[0], np.cumsum(n)[:-1]])
    T = int(n.sum())
    rec = np.repeat(np.arange(n_super_kmers), n)
    off = np.arange(T) - starts[rec]
    gi = np.where(rc[rec], pos[rec] + n[rec] - 1 - off, pos[rec] + off)
    sym = genome[gi]
    sym = np.where(rc[rec], 3 - sym, sym).astype(np.uint8)
    if err > 0:
        m = rng.random(T) < err
        sym = ((sym + m * rng.integers(1, 4, T)) % 4).astype(np.uint8)
    nb = (n + 3) // 4
    bstarts = np.concatenate([[0], np.cumsum(nb)[:-1]])
    padded = np.zeros(int(nb.sum()) * 4, dtype=np.uint8)
    if pad_garbage:
        padded[:] = rng.integers(0, 4, padded.size)
    padded[4 * bstarts[rec] + off] = sym
    q = padded.reshape(-1, 4)
    payload = ((q[:, 0] << 6) | (q[:, 1] << 4) | (q[:, 2] << 2) | q[:, 3]).astype(np.uint8)
    total = int(nb.sum()) + n_super_kmers
    data = np.zeros(total, dtype=np.uint8)
    brec = np.repeat(np.arange(n_super_kmers), nb)
    data[np.arange(payload.size) + brec + 1] = payload
    data[bstarts + np.arange(n_super_kmers)] = a.astype(np.uint8)
    pb, pr, pf = _make_packs(1 + nb, a + 1)
    return Bin(data=data, n_rec=int((a + 1).sum()), n_super_kmers=n_super_kmers, pack_bytes=pb, pack_recs=pr, k=k, extras=a, pack_first=pf)


SYNTH_DIR = os.path.join(ROOT, "tests", "synth")
SYNTH_SO = os.path.join(SYNTH_DIR, "libkmc_synth.so")
_synth = None


def _synth_lib():
    """tests/synth/libkmc_synth.so: the C generator (test infrastructure; the product library does not contain it)."""
    global _synth
    if _synth is None:
        src = os.path.join(SYNTH_DIR, "synth_bin.cpp")
        if (not os.path.exists(SYNTH_SO)) or os.path.getmtime(SYNTH_SO) < os.path.getmtime(src):
            subprocess.check_call(["make", "-C", SYNTH_DIR], stdout=subprocess.DEVNULL)
        L = C.CDLL(SYNTH_SO)
        L.kmcsynth_bin.argtypes = [C.c_uint64, C.c_uint32, C.c_uint64, C.c_uint64, C.c_double, C.c_uint32, C.c_void_p, C.c_uint64,
                                   C.POINTER(C.c_uint64), C.c_void_p, C.c_void_p, C.c_uint32, C.POINTER(C.c_uint32), C.POINTER(C.c_uint64)]
        _synth = L
    return _synth


def fast_bin(seed, k, n_rec, genome_len=None, mean_extra=11.0, err_ppm=10000) -> Bin:
    """A bin of exactly n_rec k-mers from the C generator (seconds for 2^28 k-mers): 30x duplicate-rich by default
    (genome_len = n_rec / 30), all-distinct with genome_len >= n_rec."""
    L = _synth_lib()
    if genome_len is None:
        genome_len = max(n_rec // 30, k + 256)
    size, n_packs, n_sk = C.c_uint64(0), C.c_uint32(0), C.c_uint64(0)
    # one pass into a generous buffer (a k-mer costs ~1 byte at ~12 k-mers per super-k-mer); the sizing call only when that was too small
    guess = int(n_rec * (1.0 + (1 + (k + 3) // 4) / (mean_extra + 1.0)) * 0.25 * 1.15) + (1 << 16) if mean_extra >= 1 else 0
    data = np.empty(guess + 64, dtype=np.uint8)
    packs = np.zeros(guess // 32768 + 64, dtype=np.uint64)
    precs = np.zeros(packs.size, dtype=np.uint64)
    rc = L.kmcsynth_bin(seed, k, n_rec, genome_len, mean_extra, err_ppm, data.ctypes.data, guess, C.byref(size),
                        packs.ctypes.data, precs.ctypes.data, packs.size, C.byref(n_packs), C.byref(n_sk)) if guess else -5
    if rc == -5:
        rc = L.kmcsynth_bin(seed, k, n_rec, genome_len, mean_extra, err_ppm, None, 0, C.byref(size), None, None, 0, C.byref(n_packs), C.byref(n_sk))
        assert rc == 0, rc
        data = np.zeros(size.value + 64, dtype=np.uint8)
        packs = np.zeros(max(n_packs.value, 1), dtype=np.uint64)
        precs = np.zeros(packs.size, dtype=np.uint64)
        rc = L.kmcsynth_bin(seed, k, n_rec, genome_len, mean_extra, err_ppm, data.ctypes.data, data.size, C.byref(size),
                            packs.ctypes.data, precs.ctypes.data, packs.size, C.byref(n_packs), C.byref(n_sk))
    assert rc == 0, rc
    data[size.value:size.value + 64] = 0
    # pack_recs = k-mers per pack: a safe upper bound of its (k+x)-mers in canonical mode (kb_sorter.h:605-633); -b mode needs Bin.extras
    return Bin(data=data[:size.value], n_rec=n_rec, n_super_kmers=int(n_sk.value), pack_bytes=packs[:n_packs.value], pack_recs=precs[:n_packs.value], k=k)


def bin_extras(b: "Bin"):
    """(extras u8 [n_super_kmers], pack_superkmers u32 [n_packs]): what a stage 1 with the N4 patch would hand over (kmcb200_submit_bin_indexed)."""
    d, k = b.data, b.k
    ex, per_pack = [], []
    pos = 0
    for pb in [int(x) for x in b.pack_bytes]:
        end, n = pos + pb, 0
        while pos < end:
            a = int(d[pos])
            ex.append(a)
            pos += 1 + (a + k + 3) // 4
            n += 1
        assert pos == end
        per_pack.append(n)
    return np.array(ex, dtype=np.uint8), np.array(per_pack, dtype=np.uint32)


def to_skb(b: "Bin"):
    """Bin -> the package's SuperKmerBin (what Stage2Context.process_bin takes)."""
    import kmc_b200
    return kmc_b200.SuperKmerBin(data=b.data, n_rec=b.n_rec, pack_bytes=b.pack_bytes, n_super_kmers=b.n_super_kmers, kmer_len=b.k)


def bin_from_reads(k, reads):
    """Put whole reads (strings over ACGT) into one bin as super-k-mers of <= k+255 symbols overlapping by k-1.
    (Stage 1 would cut by minimizer, splitter.cpp:557-677; for stage 2 only the multiset of k-mers matters.)"""
    lut = {"A": 0, "C": 1, "G": 2, "T": 3}
    lists = []
    for r in reads:
        s = np.array([lut[c] for c in r.upper()], dtype=np.uint8)
        i = 0
        while s.size - i >= k:
            n = min(s.size - i, k + 255)
            lists.append(s[i:i + n])
            i += n - k + 1
    return pack_superkmers(k, lists)


# ----------------------------------------------------------------------------- brute force (pure python, tiny cases)
def brute_force_counts(bin_, p: Params):
    """dict canonical-kmer-int -> count, straight from the definition (tests/kmc_CLI/trivial-k-mer-counter/main.cpp:161-166)."""
    k = bin_.k
    d = bin_.data
    pos = 0
    cnt = {}
    mask = (1 << (2 * k)) - 1
    while pos < d.size:
        a = int(d[pos]); pos += 1
        n = k + a
        syms = [(int(d[pos + (i >> 2)]) >> (6 - 2 * (i & 3))) & 3 for i in range(n)]
        pos += (n + 3) // 4
        for i in range(a + 1):
            f = 0
            r = 0
            for j in range(k):
                f = (f << 2) | syms[i + j]
                r |= (3 - syms[i + j]) << (2 * j)
            c = min(f, r) if p.both_strands else f
            cnt[c & mask] = cnt.get(c & mask, 0) + 1
    return cnt


def expected_from_counts(cnt, p: Params):
    """(payload bytes, lut, stats) from a dict of counts, following kb_sorter.h:1168-1267."""
    out = bytearray()
    lut = np.zeros(p.lut_entries, dtype=np.uint64)
    kb = (p.k - p.lut_prefix_len) // 4
    n_unique = n_min = n_max = n_total = 0
    for km in sorted(cnt):
        c = cnt[km]
        n_total += c
        n_unique += 1
        if c < p.cutoff_min:
            n_min += 1
        elif c > p.cutoff_max:
            n_max += 1
        else:
            c = min(c, p.counter_max)
            out += (km & ((1 << (8 * kb)) - 1)).to_bytes(kb, "big") if kb else b""
            out += c.to_bytes(8, "little")[:p.counter_bytes]
            lut[km >> (2 * (p.k - p.lut_prefix_len))] += 1
    return bytes(out), lut, (n_unique, n_min, n_max, n_total)


def decode_payload(payload, lut, p: Params):
    """Inverse of the emit format: list of (kmer string, count) in file order (kmc_api/kmc_file.cpp reader logic)."""
    kb = (p.k - p.lut_prefix_len) // 4
    rb = p.out_rec_bytes
    res = []
    i = 0
    for prefix in range(p.lut_entries):
        for _ in range(int(lut[prefix])):
            suf = int.from_bytes(payload[i * rb:i * rb + kb], "big")
            c = int.from_bytes(payload[i * rb + kb:(i + 1) * rb], "little") if p.counter_bytes else 1
            km = (prefix << (8 * kb)) | suf
            s = "".join("ACGT"[(km >> (2 * (p.k - 1 - j))) & 3] for j in range(p.k))
            res.append((s, c))
            i += 1
    return res


# ----------------------------------------------------------------------------- stored reference results
def sha256(data):
    return hashlib.sha256(bytes(data)).hexdigest()


def result_digest(r):
    """A bin result (this module's BinResult or kmc_b200's) as reference_results.json stores it: the four counters in
    the clear, payload and LUT (uint64) by SHA-256."""
    payload = r.payload if isinstance(r.payload, bytes) else r.payload.tobytes()
    return {"stats": [int(x) for x in r.stats], "payload_sha256": sha256(payload),
            "lut_sha256": sha256(np.ascontiguousarray(r.lut, dtype=np.uint64).tobytes())}


@functools.lru_cache(maxsize=None)
def _reference_results():
    with open(REFERENCE_RESULTS) as f:
        return json.load(f)


def reference_results(group):
    """What the reference returned for one test module's inputs (a dict keyed by case)."""
    return _reference_results()[group]


# ----------------------------------------------------------------------------- build helpers
def ensure_oracle_built():
    src = os.path.join(ORACLE_DIR, "stage2_oracle.c")
    if (not os.path.exists(ORACLE_SO)) or os.path.getmtime(ORACLE_SO) < os.path.getmtime(src):
        subprocess.check_call(["make", "-C", ORACLE_DIR, "oracle"], stdout=subprocess.DEVNULL)
    return ORACLE_SO


def reference_available():
    return os.path.exists(REF_SO)


def ensure_reference_built():
    """Build oracle/_ref from /root/reference when it is there (dev container); on the GPU box the prebuilt .so travels."""
    if not os.path.exists(REF_SO) and os.path.exists("/root/reference/kmc_core/kb_sorter.h"):
        subprocess.check_call(["make", "-C", ORACLE_DIR, "ref"], stdout=subprocess.DEVNULL)
    return os.path.exists(REF_SO)


def _u8p(a):
    return a.ctypes.data_as(C.POINTER(C.c_uint8))


def _u64p(a):
    return a.ctypes.data_as(C.POINTER(C.c_uint64))


@dataclass
class BinResult:
    payload: bytes
    lut: np.ndarray
    stats: tuple      # n_unique, n_cutoff_min, n_cutoff_max, n_total

    def same_as(self, o):
        return self.payload == o.payload and np.array_equal(self.lut, o.lut) and tuple(self.stats) == tuple(o.stats)


class _KmcoParams(C.Structure):
    _fields_ = [("kmer_len", C.c_uint32), ("both_strands", C.c_uint32), ("cutoff_min", C.c_uint32),
                ("cutoff_max", C.c_uint32), ("counter_max", C.c_uint32), ("lut_prefix_len", C.c_uint32)]


class Oracle:
    def __init__(self):
        self.lib = C.CDLL(ensure_oracle_built())
        L = self.lib
        L.kmco_process_bin.restype = C.c_uint64
        L.kmco_process_bin.argtypes = [C.POINTER(_KmcoParams), C.c_void_p, C.c_uint64, C.c_uint64, C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p]
        L.kmco_expand.restype = C.c_uint64
        L.kmco_expand.argtypes = [C.POINTER(_KmcoParams), C.c_void_p, C.c_uint64, C.c_void_p]
        L.kmco_sort.restype = None
        L.kmco_sort.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint32, C.c_uint32]
        L.kmco_compact.restype = C.c_uint64
        L.kmco_compact.argtypes = [C.POINTER(_KmcoParams), C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p]
        L.kmco_walk_bin.restype = C.c_uint64
        L.kmco_walk_bin.argtypes = [C.c_void_p, C.c_uint64, C.c_uint32, C.c_void_p]

    @staticmethod
    def _p(p: Params):
        return _KmcoParams(p.k, int(p.both_strands), p.cutoff_min, min(p.cutoff_max, 0xFFFFFFFF), min(p.counter_max, 0xFFFFFFFF), p.lut_prefix_len)

    def walk(self, bin_: Bin):
        n = C.c_uint64(0)
        d = np.ascontiguousarray(bin_.data)
        r = self.lib.kmco_walk_bin(d.ctypes.data, d.size, bin_.k, C.byref(n))
        return int(r), int(n.value)

    def expand(self, bin_: Bin, p: Params):
        recs = np.zeros((bin_.n_rec + 1) * p.words, dtype=np.uint64)
        d = np.ascontiguousarray(bin_.data)
        n = self.lib.kmco_expand(C.byref(self._p(p)), d.ctypes.data, d.size, recs.ctypes.data)
        assert n == bin_.n_rec
        return recs[:n * p.words].reshape(n, p.words)

    def sort(self, recs, key_bytes):
        recs = np.ascontiguousarray(recs, dtype=np.uint64).copy()
        n, w = recs.shape
        tmp = np.empty_like(recs)
        self.lib.kmco_sort(recs.ctypes.data, tmp.ctypes.data, n, w, key_bytes)
        return recs

    def compact(self, sorted_recs, p: Params):
        sorted_recs = np.ascontiguousarray(sorted_recs, dtype=np.uint64)
        n = sorted_recs.shape[0]
        cap = max(p.out_capacity(n), p.out_rec_bytes) + 64
        out = np.zeros(cap, dtype=np.uint8)
        lut = np.zeros(p.lut_entries, dtype=np.uint64)
        stats = np.zeros(4, dtype=np.uint64)
        r = self.lib.kmco_compact(C.byref(self._p(p)), sorted_recs.ctypes.data, n, out.ctypes.data, cap, lut.ctypes.data, stats.ctypes.data)
        assert r != 0xFFFFFFFFFFFFFFFF
        return BinResult(out[:r].tobytes(), lut, tuple(int(x) for x in stats))

    def process_bin(self, bin_: Bin, p: Params) -> BinResult:
        cap = max(p.out_capacity(bin_.n_rec), p.out_rec_bytes) + 64
        out = np.zeros(cap, dtype=np.uint8)
        lut = np.zeros(p.lut_entries, dtype=np.uint64)
        stats = np.zeros(4, dtype=np.uint64)
        d = np.ascontiguousarray(bin_.data)
        r = self.lib.kmco_process_bin(C.byref(self._p(p)), d.ctypes.data, d.size, bin_.n_rec, out.ctypes.data, cap, lut.ctypes.data, stats.ctypes.data)
        assert r < 0xFFFFFFFFFFFFFFF0, "oracle failed (%d)" % (r - (1 << 64))
        return BinResult(out[:r].tobytes(), lut, tuple(int(x) for x in stats))


class Reference:
    """The unmodified reference stage 2 (oracle/ref/ref_harness.cpp)."""
    RADULS, RADIX_H, B200_DROPIN = 0, 1, 2

    def __init__(self, with_b200=False):
        if not ensure_reference_built():
            raise RuntimeError("oracle/_ref/libkmc_ref.so is not built and /root/reference is absent")
        if with_b200 and not os.path.exists(REF_B200_SO):
            raise RuntimeError("oracle/_ref/libkmc_ref_b200.so is not built")
        self.lib = C.CDLL(REF_B200_SO if with_b200 else REF_SO)
        self.lib.kmcref_process_bins.restype = C.c_int
        self.lib.kmcref_sort.restype = C.c_int
        self.lib.kmcref_sort.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint32, C.c_uint32, C.c_int, C.c_int, C.POINTER(C.c_double)]

    def process_bins(self, bins, p: Params, n_sorters=1, sort_kind=0):
        nb = len(bins)
        datas = [np.ascontiguousarray(b.data) for b in bins]
        caps = [max(p.out_capacity(b.n_rec), p.out_rec_bytes) + 64 for b in bins]
        outs = [np.zeros(c, dtype=np.uint8) for c in caps]
        luts = [np.zeros(p.lut_entries, dtype=np.uint64) for _ in bins]
        pbs = [np.ascontiguousarray(b.pack_bytes, dtype=np.uint64) for b in bins]
        kx = [b.kx_counts(p.both_strands) for b in bins]
        prs = [np.ascontiguousarray(c[1], dtype=np.uint64) for c in kx]
        PP = C.c_void_p * nb
        U64 = C.c_uint64 * nb
        U32 = C.c_uint32 * nb
        out_bytes = U64()
        stats = (C.c_uint64 * (4 * nb))()
        times = (C.c_double * 2)()
        rc = self.lib.kmcref_process_bins(
            C.c_int(p.k), C.c_int(int(p.both_strands)), C.c_uint32(p.cutoff_min), C.c_uint32(min(p.cutoff_max, 0xFFFFFFFF)),
            C.c_uint32(min(p.counter_max, 0xFFFFFFFF)), C.c_uint32(p.lut_prefix_len), C.c_int(n_sorters), C.c_int(sort_kind), C.c_int(nb),
            PP(*[d.ctypes.data for d in datas]), U64(*[d.size for d in datas]), U64(*[b.n_rec for b in bins]),
            U64(*[c[0] for c in kx]),
            PP(*[a.ctypes.data for a in pbs]), PP(*[a.ctypes.data for a in prs]), U32(*[a.size for a in pbs]),
            PP(*[o.ctypes.data for o in outs]), U64(*caps), out_bytes, PP(*[l.ctypes.data for l in luts]), stats, times)
        assert rc == 0, "reference harness rc=%d" % rc
        res = [BinResult(outs[i][:out_bytes[i]].tobytes(), luts[i], tuple(int(stats[4 * i + j]) for j in range(4))) for i in range(nb)]
        return res, (times[0], times[1])

    def process_bin(self, bin_, p: Params, n_sorters=1, sort_kind=0) -> BinResult:
        return self.process_bins([bin_], p, n_sorters, sort_kind)[0][0]

    def sort(self, recs, key_bytes, n_threads=1, sort_kind=0):
        recs = np.ascontiguousarray(recs, dtype=np.uint64).copy()
        n, w = recs.shape
        # RADULS wants 256-byte aligned buffers (arena alignment, defs.h:119)
        def aligned(nbytes):
            raw = np.empty(nbytes + 256, dtype=np.uint8)
            off = (-raw.ctypes.data) % 256
            return raw[off:off + nbytes]
        a = aligned(recs.nbytes + 64); a[:recs.nbytes] = recs.view(np.uint8).reshape(-1)
        t = aligned(recs.nbytes + 64)
        sec = C.c_double(0)
        where = self.lib.kmcref_sort(a.ctypes.data, t.ctypes.data, n, w, key_bytes, n_threads, sort_kind, C.byref(sec))
        assert where in (0, 1)
        src = t if where == 1 else a
        return src[:recs.nbytes].view(np.uint64).reshape(n, w).copy(), sec.value
