"""TEST INFRASTRUCTURE: the depth sweep over several devices (fastf_bam2db_run_sharded_sweep) against the single-job sweep
(fastf_bam2db_finish_sweep), single-rate sharded runs and the CPU oracle on the same input.  Runs on whatever FASTF_GPU_LIB names (the
emulator build with FASTF_EMU_DEVICES "devices" on CPU; libfastf_gpu.so on a B200 box).

    sharded_sweep_worker.py driver <n_devices> <n_reads> <seed>     seeded synthetic BAM, unsorted rates with the threshold edge cases
    sharded_sweep_worker.py chunks                                  shards that stream several chunks each; empty shards
    sharded_sweep_worker.py golden <case> <n_devices> <tmp>         Python host, bam2db_sweep(gpus=n) against the goldens / one GPU
    sharded_sweep_worker.py refusals <tmp>                          inputs the driver refuses, each with a message"""
import ctypes as C
import gzip
import json
import os
import shutil
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from fastf_b200 import _lib, bam2db_host as B   # noqa: E402

GOLD = os.path.join(ROOT, "tests", "golden")
KEYS = ("total", "cb_valid", "sampled", "valid", "nnz")
COO = ("m_gene", "m_cell", "m_count")
# unsorted; 0 and -1 share a threshold, as do 1e-12 and 2e-12; NaN and inf as -r takes them
EDGE_RATES = [0.5, float("nan"), 0.0, 1.0, -1.0, 0.2, float("inf"), 1e-12, 0.8, 2e-12, 0.35]


def thresholds(lib, rates):
    return np.array([lib.fastf_keep_threshold(C.c_float(r)) for r in rates], dtype=np.uint64)


def raw_sweep(lib, call, rates):
    """call(thr, res) fills a Bam2dbSweepResult; returns (per-rate [(stats, arrays)], row_keys, row_rate)"""
    thr = thresholds(lib, rates)
    res = _lib.Bam2dbSweepResult()
    try:
        call(thr, res)
        rows = np.ctypeslib.as_array(res.row_keys, (res.n_rows,)).copy() if res.n_rows else np.zeros(0, np.uint64)
        rr = np.ctypeslib.as_array(res.row_rate, (res.n_rows,)).copy() if res.n_rows else np.zeros(0, np.uint8)
        return B._sweep_to_python(res, thr, True), rows, rr
    finally:
        lib.fastf_bam2db_sweep_result_free(C.byref(res))


def single_job(ctx, bam, inputs, rates, seed, **kw):
    lib = ctx.lib

    def call(thr, res):
        with B.Bam2dbJob(ctx, inputs, 0.0, seed, want_rows=True, **kw) as job:
            job.feed(bam.ctypes.data, bam.size)
            ctx.check(lib.fastf_bam2db_finish_sweep(job.job, len(thr), thr.ctypes.data_as(_lib.c_u64p), C.byref(res)), "finish_sweep")
    return raw_sweep(lib, call, rates)


def sharded(lib, bam, inputs, rates, seed, g, **kw):
    p, keep = B.make_params(lib, inputs, 0.0, seed, True, **kw)

    def call(thr, res):
        if lib.fastf_bam2db_run_sharded_sweep(g, None, C.byref(p), C.c_void_p(bam.ctypes.data), bam.size, len(thr), thr.ctypes.data_as(_lib.c_u64p), C.byref(res)) != 0:
            raise _lib.FastfError(lib.fastf_sharded_last_error().decode())
    return raw_sweep(lib, call, rates)


def assert_same(a, b, what):
    (ra, rows_a, rr_a), (rb, rows_b, rr_b) = a, b
    assert np.array_equal(rows_a, rows_b), (what, "row_keys")
    assert np.array_equal(rr_a, rr_b), (what, "row_rate")
    for i, ((sa, xa), (sb, xb)) in enumerate(zip(ra, rb)):
        assert [sa[k] for k in KEYS] == [sb[k] for k in KEYS], (what, i, [sa[k] for k in KEYS], [sb[k] for k in KEYS])
        assert sa["bits_cell"] == sb["bits_cell"] and sa["bits_gene"] == sb["bits_gene"] and sa["bits_umi"] == sb["bits_umi"], (what, i)
        for k in COO + ("row_keys",):
            assert np.array_equal(xa[k], xb[k]), (what, i, k)


def far_copies_with_other_rates(rows, rr):
    """some key has two copies at least half the file apart whose rate indices differ: the cross-shard minimum is exercised"""
    order = np.argsort(rows, kind="stable")
    k, r, pos = rows[order], rr[order], order
    same = k[1:] == k[:-1]
    # per run of equal keys: the first and the last copy in file order
    heads = np.flatnonzero(np.concatenate(([True], ~same)))
    ends = np.concatenate((heads[1:], [len(k)])) - 1
    for h, e in zip(heads, ends):
        if e > h and pos[e] - pos[h] > len(rows) // 2 and len(set(r[h:e + 1].tolist())) > 1:
            return True
    return False


def worker_driver(G, n_reads, seed):
    import oracle_binding
    import synth_binding
    O, S = oracle_binding.load(), synth_binding.load()
    lib = _lib.load()
    rc = 0.7
    with tempfile.TemporaryDirectory() as d:
        # few molecules for the reads: every key has many copies spread over the file
        paths, _ = S.write_bam_set(d, n_reads=n_reads, n_cells=max(20, n_reads // 300), n_genes=max(30, n_reads // 150), seed=seed, p_umi_n=0.01, n_molecules=max(50, n_reads // 12))
        inputs = B.Bam2dbInputs(lib, paths["barcodes"], paths["features"], rc, seed)
        bam = np.fromfile(paths["bam"], dtype=np.uint8)
        with _lib.Context(0) as ctx:
            one = single_job(ctx, bam, inputs, EDGE_RATES, seed)
        assert far_copies_with_other_rates(one[1], one[2]), "the input has no key with far-apart copies of different rate indices"
        for g in sorted({1, G}):
            got = sharded(lib, bam, inputs, EDGE_RATES, seed, g)
            assert_same(got, one, ("driver", g))
            x = int(lib.fastf_sharded_exchanged())
            assert g == 1 or x > 0, x
            # the Python host: the same result, and without rows the same COO
            py = B.run_sharded_sweep(lib, bam, inputs, EDGE_RATES, seed, g)
            nr = B.run_sharded_sweep(lib, bam, inputs, EDGE_RATES, seed, g, want_rows=False)
            for i, ((s1, a1), (s2, a2), (s3, a3)) in enumerate(zip(one[0], py, nr)):
                assert [s1[k] for k in KEYS] == [s2[k] for k in KEYS] == [s3[k] for k in KEYS], (g, i)
                assert s2["exchanged_keys"] == x and s3["n_rows"] == 0 and a3["row_keys"].size == 0, (g, i)
                for k in COO:
                    assert np.array_equal(a1[k], a2[k]) and np.array_equal(a1[k], a3[k]), (g, i, k)
                assert np.array_equal(a1["row_keys"], a2["row_keys"]), (g, i)
        # three rates: the single-rate sharded driver and the oracle
        for r in (0.2, 0.5, 1.0):
            i = EDGE_RATES.index(r)
            st, arr = B.run_sharded(lib, bam, inputs, r, seed, G, want_rows=True)
            o = O.bam2db(paths["bam"], paths["barcodes"], paths["features"], rc, r, seed)
            s1, a1 = one[0][i]
            assert [s1[k] for k in KEYS] == [st[k] for k in KEYS] == [o[k] for k in KEYS], r
            for k in COO:
                assert np.array_equal(a1[k], arr[k]) and np.array_equal(a1[k], o[k]), (r, k)
            assert np.array_equal(a1["row_keys"], arr["row_keys"]), r
    print("ok sharded sweep driver: %d devices, %d reads, %d rows, exchanged %d keys" % (G, n_reads, one[1].size, x))


def worker_chunks():
    """shards that stream several chunks each, and a BAM of fewer blocks than devices (empty shards)"""
    import synth_binding
    S = synth_binding.load()
    lib = _lib.load()
    rates = [0.9, 0.1, 0.5, 0.0, 1.0]
    with tempfile.TemporaryDirectory() as d:
        for n_reads, G, chunk in ((12000, 2, 1 << 20), (40, 5, 0)):
            paths, _ = S.write_bam_set(d, n_reads=n_reads, n_cells=20, n_genes=30, seed=7, p_umi_n=0.01, n_molecules=max(10, n_reads // 4))
            inputs = B.Bam2dbInputs(lib, paths["barcodes"], paths["features"], 0.8, 926)
            bam = np.fromfile(paths["bam"], dtype=np.uint8)
            with _lib.Context(0) as ctx:
                one = single_job(ctx, bam, inputs, rates, 926)
            got = sharded(lib, bam, inputs, rates, 926, G, chunk_inflated_bytes=chunk)
            st = got[0][0][0]
            assert (st["n_chunks"] >= 2 * G) if chunk else (st["n_blocks"] < G), (n_reads, G, st["n_chunks"], st["n_blocks"])
            assert_same(got, one, ("chunks", n_reads, G))
    print("ok chunks")


def worker_golden(case_name, G, tmp):
    import fastf_b200
    from dbdigest import db_digest
    c = {c["name"]: c for c in json.load(open(os.path.join(GOLD, "manifest.json")))["cases"]}[case_name]
    d = os.path.join(GOLD, c["dir"])
    rd, umi = c["rate_depth"], bool(c.get("umicopies"))
    others = [r for r in (0.7, 0.0, 1.0, 0.25) if r != rd]
    rates = [others[0], rd] + others[1:3]
    files = ["matrix.mtx.gz", "barcodes.tsv.gz", "features.tsv.gz"] + (["umi.tsv.gz"] if umi else [])
    B._umi_copies_flag = 1 if umi else 0
    os.chdir(d)   # the matrix header records the BAM path as passed: the golden run used "in.bam"
    multi, one = os.path.join(tmp, "multi"), os.path.join(tmp, "one")
    args = ("in.bam", "x.db")
    rest = ("barcodes.tsv.gz", "features.tsv.gz", c["rate_cell"], rates, c["seed"])
    assert fastf_b200.bam2db_sweep(args[0], args[1], multi, *rest, gpus=G) == 0
    assert fastf_b200.bam2db_sweep(args[0], args[1], one, *rest) == 0

    def same(a, b):
        return all(gzip.open(os.path.join(a, f), "rb").read() == gzip.open(os.path.join(b, f), "rb").read() for f in files)
    for r in rates:
        got = os.path.join(multi, "depth_%s" % r)
        want = os.path.join(d, c["expect"]) if r == rd else os.path.join(one, "depth_%s" % r)
        assert same(got, want), (case_name, r)
        wd = json.load(open(os.path.join(want, "db_digest.json"))) if r == rd else db_digest(os.path.join(want, "x.db"))
        assert db_digest(os.path.join(got, "x.db")) == wd, (case_name, r)
    print("ok golden", case_name, G)


def worker_refusals(tmp):
    import bamgen
    lib = _lib.load()
    g = os.path.join(GOLD, "synth4k")
    inputs = B.Bam2dbInputs(lib, os.path.join(g, "barcodes.tsv.gz"), os.path.join(g, "features.tsv.gz"), 1.0, 926)
    bam = np.fromfile(os.path.join(g, "in.bam"), dtype=np.uint8)

    def refused(needle, bam_, rates=None, thr=None, G=3):
        p, keep = B.make_params(lib, inputs, 0.0, 926, True)
        t = thresholds(lib, rates) if thr is None else np.asarray(thr, dtype=np.uint64)
        res = _lib.Bam2dbSweepResult()
        rc = lib.fastf_bam2db_run_sharded_sweep(G, None, C.byref(p), C.c_void_p(bam_.ctypes.data), bam_.size, len(t), t.ctypes.data_as(_lib.c_u64p) if t.size else None, C.byref(res))
        msg = lib.fastf_sharded_last_error().decode()
        lib.fastf_bam2db_sweep_result_free(C.byref(res))
        assert rc != 0 and needle in msg, (needle, rc, msg)
        return msg
    bad = bam.copy()
    bad[bad.size // 2: bad.size // 2 + 4096] = 7
    refused("malformed input", bad, [0.1, 0.5])
    refused("1..32 keep thresholds", bam, thr=[])
    refused("1..32 keep thresholds", bam, [0.01 * (i + 1) for i in range(33)])
    refused("keep_thresholds[1] > 2^32", bam, thr=[1 << 31, (1 << 32) + 1])
    # records that straddle BGZF blocks (a writer other than htslib): single-GPU only
    whole = gzip.decompress(open(os.path.join(g, "in.bam"), "rb").read())
    cut = np.frombuffer(bamgen.bgzf_file([whole[i:i + 30011] for i in range(0, len(whole), 30011)]), dtype=np.uint8)
    refused("record-straddles-bgzf-block", cut, [0.1, 0.5])
    # the Python host retries in the straddle mode, which needs the whole file in one job: a clear failure, no output
    w = os.path.join(tmp, "cut")
    os.makedirs(w)
    open(os.path.join(w, "in.bam"), "wb").write(cut.tobytes())
    for f in ("barcodes.tsv.gz", "features.tsv.gz"):
        shutil.copy(os.path.join(g, f), w)
    os.chdir(w)
    import fastf_b200
    assert fastf_b200.bam2db_sweep("in.bam", "x.db", os.path.join(w, "out"), "barcodes.tsv.gz", "features.tsv.gz", 1.0, [0.1, 0.5], 926, gpus=2) == 1
    assert not os.path.exists(os.path.join(w, "out", "depth_0.1", "matrix.mtx.gz"))
    print("ok refusals")


if __name__ == "__main__":
    if sys.argv[1] == "driver":
        worker_driver(int(sys.argv[2]), int(sys.argv[3]), int(sys.argv[4]))
    elif sys.argv[1] == "chunks":
        worker_chunks()
    elif sys.argv[1] == "golden":
        worker_golden(sys.argv[2], int(sys.argv[3]), sys.argv[4])
    elif sys.argv[1] == "refusals":
        worker_refusals(sys.argv[2])
