"""The database writer of SURVEY 8f N3 (kmcb200_db_*: pinned staging ring, writer thread, footer) against files written by the REFERENCE:
a database made by the unmodified reference CLI (one stage-2 sorter so that the bin order is deterministic) is taken apart into its bins
(payload and LUT of every bin, signature map, header fields) and replayed through the writer; .kmc_pre and .kmc_suf must come out byte
for byte.  Host-only: runs without a GPU (the staging ring is then plain memory).

The reference's databases are stored in tests/golden/refdb_*.npz, and the SHA-256 of the files the reference's kmc_tools read back
(with the dump it printed) in tests/golden/reference_results.json ("db_writer"); tests/golden/make_reference_results.py made both."""
import os
import struct

import numpy as np
import pytest

from kmc_testlib import GOLDEN_DIR, Params, reference_results, sha256

REFDB_CASES = [(31, ("-ci2",)), (28, ("-ci1", "-cs65535")), (55, ("-ci1", "-b"))]
REFDB_ARGS = ("-sr1", "-n64")          # one stage-2 sorter, 64 bins
REFDB_STATS = ("#Unique_k-mers", "#k-mers_below_min_threshold", "#k-mers_above_max_threshold", "#Total no. of k-mers")
STANDALONE_PARAMS = Params(k=31, cutoff_min=2, lut_prefix_len=7)
STANDALONE_SIG_LEN = 9


def refdb_path(k, extra):
    return os.path.join(GOLDEN_DIR, "refdb_k%d%s.npz" % (k, "".join(extra)))


def read_db(prefix):
    return open(prefix + ".kmc_pre", "rb").read(), open(prefix + ".kmc_suf", "rb").read()


def parse_db(pre, suf):
    assert pre[:4] == b"KMCP" and pre[-4:] == b"KMCP" and suf[:4] == b"KMCS" and suf[-4:] == b"KMCS"
    header_offset = struct.unpack("<I", pre[-8:-4])[0]
    h = len(pre) - 8 - header_offset
    k, mode, counter_size, p, sig_len, cmin, cmax = struct.unpack("<7I", pre[h:h + 28])
    n_counted, = struct.unpack("<Q", pre[h + 28:h + 36])
    both = pre[h + 36] == 0
    map_entries = (1 << (2 * sig_len)) + 1
    m0 = h - 4 * map_entries
    sig_map = np.frombuffer(pre[m0:h], dtype=np.uint32)
    n_recs, = struct.unpack("<Q", pre[m0 - 8:m0])
    lut_all = np.frombuffer(pre[4:m0 - 8], dtype=np.uint64)
    n_lut = 1 << (2 * p)
    assert lut_all.size % n_lut == 0
    luts = lut_all.reshape(-1, n_lut)
    rec = (k - p) // 4 + counter_size
    starts = np.append(luts[:, 0], np.uint64(n_recs)).astype(np.int64)
    payloads = [suf[4 + int(starts[b]) * rec:4 + int(starts[b + 1]) * rec] for b in range(luts.shape[0])]
    assert 4 + n_recs * rec + 4 == len(suf)
    return dict(k=k, counter_size=counter_size, p=p, sig_len=sig_len, cmin=cmin, cmax=cmax, both=both, n_counted=n_counted,
                sig_map=sig_map, luts=luts, payloads=payloads, n_recs=n_recs)


@pytest.mark.parametrize("k,extra", REFDB_CASES)
@pytest.mark.parametrize("raw_lut", [False, True])
def test_writer_reproduces_reference_files(tmp_path, k, extra, raw_lut):
    import ctypes as C
    import kmc_b200
    tmp = str(tmp_path)
    z = np.load(refdb_path(k, extra))
    ref_pre, ref_suf = z["kmc_pre"].tobytes(), z["kmc_suf"].tobytes()
    d = parse_db(ref_pre, ref_suf)
    assert d["k"] == k
    st = dict(zip(REFDB_STATS, z["stats"]))
    out = os.path.join(tmp, "replay")
    w = kmc_b200.DbWriter(out, d["k"], d["counter_size"], d["p"], d["sig_len"], d["cmin"], d["cmax"], d["both"], staging_bytes=1 << 20)   # a small ring: it wraps and blocks
    n_bins = d["luts"].shape[0]
    for b in range(n_bins):
        pay = d["payloads"][b]
        # every region is 64 KiB larger than its payload (as when a GPU caller reserves the bin's output capacity): the 64 bins pass
        # through the 1 MiB ring several times
        ptr = w.reserve(len(pay) + (1 << 16))
        C.memmove(ptr, pay, len(pay))
        lut = d["luts"][b]
        if raw_lut:
            nxt = np.append(lut[1:], np.uint64(w.records + len(pay) // max((d["k"] - d["p"]) // 4 + d["counter_size"], 1)))
            lut = nxt - lut
        # the statistics only enter the file as n_unique - n_cutoff_min - n_cutoff_max: give them all to the first bin
        bin_stats = (int(st["#Unique_k-mers"]), int(st["#k-mers_below_min_threshold"]), int(st["#k-mers_above_max_threshold"]), int(st["#Total no. of k-mers"])) if b == 0 else (0, 0, 0, 0)
        sigs = np.nonzero(d["sig_map"] == b)[0]
        w.commit_bin(len(pay), lut, bin_stats, sigs, raw_lut=raw_lut)
    tot = w.close()
    assert tot[0] - tot[1] - tot[2] == d["n_counted"]
    assert open(out + ".kmc_suf", "rb").read() == ref_suf
    assert open(out + ".kmc_pre", "rb").read() == ref_pre


def _standalone_bins():
    from kmc_testlib import synth_bin
    sizes = [4000, 0, 900, 15000, 1, 7000]
    return [synth_bin(40 + i, 31, n, genome_len=max(n, 500)) for i, n in enumerate(sizes)]


def _expected_dump(results, p):
    from kmc_testlib import decode_payload
    lines = []
    for r in results:
        lines += ["%s\t%d" % (s, c) for s, c in decode_payload(r.payload if isinstance(r.payload, bytes) else r.payload.tobytes(), r.lut, p)]
    return lines


def dump_sha256(results, p):
    """SHA-256 of what `kmc_tools transform <db> dump` prints for a database of these bin results (one line per record, in file order)."""
    return sha256("".join(line + "\n" for line in _expected_dump(results, p)).encode())


def write_oracle_db(out, results, p, staging_bytes):
    """A database of bin results through the writer (bin i under signature i, LUTs scanned by the writer)."""
    import ctypes as C
    import kmc_b200
    w = kmc_b200.DbWriter(out, p.k, p.counter_bytes, p.lut_prefix_len, STANDALONE_SIG_LEN, p.cutoff_min, p.cutoff_max, p.both_strands,
                          staging_bytes=staging_bytes)
    for i, r in enumerate(results):
        ptr = w.reserve(len(r.payload))
        C.memmove(ptr, r.payload, len(r.payload))
        w.commit_bin(len(r.payload), r.lut, r.stats, [i], raw_lut=True)
    return w.close()


def check_against_reference_tools(out, results, p, case):
    """The files must be those the reference's kmc_tools read back, and what it printed must be the dump of the bin results."""
    ref = reference_results("db_writer")[case]
    pre, suf = read_db(out)
    assert sha256(pre) == ref["kmc_pre_sha256"] and sha256(suf) == ref["kmc_suf_sha256"]
    assert dump_sha256(results, p) == ref["dump_sha256"]


def test_standalone_database_is_readable_by_the_reference_tools(tmp_path, oracle):
    """Bins -> (oracle results) -> writer -> files; the reference's kmc_tools must read the database back bin after bin."""
    p = STANDALONE_PARAMS
    res = [oracle.process_bin(b, p) for b in _standalone_bins()]
    out = os.path.join(str(tmp_path), "standalone")
    tot = write_oracle_db(out, res, p, 1 << 20)
    assert tot == tuple(sum(r.stats[j] for r in res) for j in range(4))
    check_against_reference_tools(out, res, p, "standalone")


@pytest.mark.gpu
def test_gpu_bins_straight_into_the_database(tmp_path, oracle):
    """The standalone stage 2: bins -> kmcb200_submit_bin with the writer's pinned ring as D2H target -> kmcb200_wait_bin_scanned (LUT prefix
    sum on the GPU, base = records so far) -> commit; two bins in flight while the writer thread appends the earlier ones."""
    import kmc_b200
    p = STANDALONE_PARAMS
    bins = _standalone_bins() * 3
    res = [oracle.process_bin(b, p) for b in bins]
    out = os.path.join(str(tmp_path), "gpu_db")
    ctx = kmc_b200.Stage2Context(kmc_b200.Stage2Params(31, True, 2, 10 ** 9, 255, 7), device=0, n_slots=2)
    w = kmc_b200.DbWriter(out, 31, p.counter_bytes, 7, STANDALONE_SIG_LEN, p.cutoff_min, p.cutoff_max, True, staging_bytes=1 << 18)
    luts = [np.zeros(ctx.lut_entries, dtype=np.uint64) for _ in range(2)]
    datas = [np.ascontiguousarray(b.data) for b in bins]

    def finish(i):
        nbytes, stats = ctx.wait_bin_scanned(i % 2, w.records)
        assert stats == res[i].stats and nbytes == len(res[i].payload)
        w.commit_bin(nbytes, luts[i % 2], stats, [i])

    # one region is open at a time (commit order = file order), so the pipeline is: reserve i, submit i, (GPU works), wait i, commit i -
    # the overlap is between the GPU / the copies of bin i and the writer thread's fwrite of bins < i
    for i, b in enumerate(bins):
        cap = ctx.out_capacity(b.n_rec) + 64
        ptr = w.reserve(cap)
        ctx.submit_bin(i % 2, datas[i].ctypes.data, datas[i].size, b.n_rec, np.ascontiguousarray(b.pack_bytes), ptr, cap, luts[i % 2].ctypes.data)
        finish(i)
    tot = w.close()
    ctx.close()
    assert tot == tuple(sum(r.stats[j] for r in res) for j in range(4))
    check_against_reference_tools(out, res, p, "standalone_x3")
