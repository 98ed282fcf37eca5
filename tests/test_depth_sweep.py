"""The depth sweep (`fastF bam2db --depths`, fastf_b200.bam2db_sweep, fastf_bam2db_finish_sweep): one pass over the BAM, the exact
output set of every depth rate.  On the CPU through the SIMT-emulator build (this file, run as a script, is the worker the tests
start with FASTF_GPU_LIB pointing at it); on the B200 against single-rate jobs on the same context."""
import gzip
import json
import os
import shutil
import subprocess
import sys

import numpy as np
import pytest

from bam2db_harness import FILES, GOLD, KEYS, ROOT, bam2db_cases, bam_4m, cli_refusal, emu_cli, emu_lib, same_files, single_run, spawn  # noqa: F401 (fixtures)


def _sweep_rates(rd):
    """the golden rate among others, unsorted, golden rate second"""
    others = [r for r in (0.7, 0.0, 1.0, 0.25) if r != rd]
    return [others[0], rd] + others[1:3]


# ------------------------------------------------------------------------------------------------------------------------------
# worker (runs under the emulator build)
# ------------------------------------------------------------------------------------------------------------------------------
def _worker_golden(case_name, use_cli, tmp):
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import fastf_b200
    from fastf_b200 import _lib, bam2db_host as B
    from dbdigest import db_digest
    import oracle_binding
    c = {c["name"]: c for c in bam2db_cases()}[case_name]
    d = os.path.join(GOLD, c["dir"])
    rc_, rd, seed, umi = c["rate_cell"], c["rate_depth"], c["seed"], bool(c.get("umicopies"))
    rates = _sweep_rates(rd)
    files = FILES + (["umi.tsv.gz"] if umi else [])
    cli = os.environ.get("FASTF_EMU_CLI") if use_cli else None
    B._umi_copies_flag = 1 if umi else 0
    os.chdir(d)   # the matrix header records the BAM path as passed: the golden run used "in.bam"

    out = os.path.join(tmp, "sweep")
    if cli:
        cmd = [cli, "bam2db", "-b", "in.bam", "-f", "features.tsv.gz", "-a", "barcodes.tsv.gz", "-d", "x.db", "-c", str(rc_), "--depths", ",".join(str(r) for r in rates), "-o", out, "-s", str(seed)]
        os.makedirs(out)
        r = subprocess.run(cmd + (["-u"] if umi else []), stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True)
        assert r.returncode == 0, r.stderr
    else:
        assert fastf_b200.bam2db_sweep("in.bam", "x.db", out, "barcodes.tsv.gz", "features.tsv.gz", rc_, rates, seed) == 0
    O = oracle_binding.load()
    ctx = _lib.Context(0)
    inputs = B.Bam2dbInputs(ctx.lib, "barcodes.tsv.gz", "features.tsv.gz", rc_, seed)
    api = B.run_device_sweep(ctx, np.fromfile("in.bam", dtype=np.uint8), inputs, rates, seed)
    for k, rate in enumerate(rates):
        got = os.path.join(out, "depth_" + str(rate))
        if rate == rd:
            want = os.path.join(d, c["expect"])
            assert same_files(got, want, files), (case_name, rate)
            assert db_digest(os.path.join(got, "x.db")) == json.load(open(os.path.join(want, "db_digest.json"))), (case_name, rate)
        else:
            want = os.path.join(tmp, "single_%d" % k)
            single_run(cli, rc_, rate, seed, umi, want)
            assert same_files(got, want, files), (case_name, rate)
            assert db_digest(os.path.join(got, "x.db")) == db_digest(os.path.join(want, "x.db")), (case_name, rate)
            o = O.bam2db(os.path.join(d, "in.bam"), os.path.join(d, "barcodes.tsv.gz"), os.path.join(d, "features.tsv.gz"), rc_, rate, seed)
            st, arr = api[k]
            assert [st[x] for x in KEYS] == [o[x] for x in KEYS], (case_name, rate)
            for x in ("m_gene", "m_cell", "m_count"):
                assert np.array_equal(arr[x], o[x]), (case_name, rate, x)
    ctx.close()
    print("ok", case_name, "cli" if cli else "python")


def _worker_streaming(tmp):
    """the same sweep from many streamed chunks and odd feed pieces, and on a BAM whose records straddle BGZF blocks"""
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import fastf_b200
    import bamgen
    from fastf_b200 import _lib, bam2db_host as B
    from dbdigest import db_digest
    ctx = _lib.Context(0)
    rates = [0.9, 0.1, 0.5, 0.0, 1.0]
    for d, rc_ in (("edge", 0.8), ("synth4k", 0.5)):
        g = os.path.join(GOLD, d)
        inputs = B.Bam2dbInputs(ctx.lib, os.path.join(g, "barcodes.tsv.gz"), os.path.join(g, "features.tsv.gz"), rc_, 926)
        bam = np.fromfile(os.path.join(g, "in.bam"), dtype=np.uint8)
        ref = None
        for chunk, piece in ((0, 0), (1 << 20, 777), (1 << 20, 50001)):
            res = B.run_device_sweep(ctx, bam, inputs, rates, 926, chunk_inflated_bytes=chunk, feed_piece=piece)
            key = [(tuple(st[x] for x in KEYS), tuple(a[x].tobytes() for x in ("m_gene", "m_cell", "m_count", "row_keys"))) for st, a in res]
            assert res[0][0]["n_chunks"] > 1 or chunk == 0 or d == "edge", (d, chunk, res[0][0]["n_chunks"])
            if ref is None:
                ref = key
            assert key == ref, (d, chunk, piece)
        # re-cut into blocks of odd sizes: records cross block boundaries, the host retries in the straddle mode
        w = os.path.join(tmp, d)
        os.makedirs(w)
        whole = gzip.decompress(open(os.path.join(g, "in.bam"), "rb").read())
        cut = 997 if d == "edge" else 30011
        open(os.path.join(w, "in.bam"), "wb").write(bamgen.bgzf_file([whole[i:i + cut] for i in range(0, len(whole), cut)]))
        for f in ("barcodes.tsv.gz", "features.tsv.gz"):
            shutil.copy(os.path.join(g, f), w)
        os.chdir(w)
        B._umi_copies_flag = 1
        assert fastf_b200.bam2db_sweep("in.bam", "x.db", os.path.join(w, "cut"), "barcodes.tsv.gz", "features.tsv.gz", rc_, rates, 926, ctx=ctx) == 0
        os.chdir(g)
        assert fastf_b200.bam2db_sweep("in.bam", "x.db", os.path.join(w, "orig"), "barcodes.tsv.gz", "features.tsv.gz", rc_, rates, 926, ctx=ctx) == 0
        for r in rates:
            a, b = os.path.join(w, "cut", "depth_%s" % r), os.path.join(w, "orig", "depth_%s" % r)
            assert same_files(a, b, ["barcodes.tsv.gz", "features.tsv.gz", "umi.tsv.gz"]), (d, r)
            # the matrix header names the BAM as passed ("in.bam" both times): identical too
            assert same_files(a, b, ["matrix.mtx.gz"]), (d, r)
            assert db_digest(os.path.join(a, "x.db")) == db_digest(os.path.join(b, "x.db")), (d, r)
        print("ok", d)
    ctx.close()


def _skewed_vs_single(ctx, d, n_reads, rates):
    """a sweep over a BAM whose (cell, gene) groups hold thousands of UMIs equals single-rate jobs; returns the largest group"""
    import synth_binding
    from fastf_b200 import bam2db_host as B
    paths, _ = synth_binding.load().write_bam_set(d, n_reads=n_reads, n_molecules=n_reads, n_cells=2, n_genes=2, seed=5, p_umi_n=0.01)
    inputs = B.Bam2dbInputs(ctx.lib, paths["barcodes"], paths["features"], 1.0, 926)
    bam = np.fromfile(paths["bam"], dtype=np.uint8)
    sweep = B.run_device_sweep(ctx, bam, inputs, rates, 926)
    for r, (st, arr) in zip(rates, sweep):
        st1, arr1 = B.run_device(ctx, bam, inputs, r, 926)
        assert [st[k] for k in KEYS] == [st1[k] for k in KEYS], (r, st, st1)
        for k in ("m_gene", "m_cell", "m_count", "row_keys"):
            assert np.array_equal(arr[k], arr1[k]), (r, k)
    return int(sweep[-1][1]["m_count"].max())


def _worker_skewed():
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import tempfile
    from fastf_b200 import _lib
    ctx = _lib.Context(0)
    with tempfile.TemporaryDirectory() as d:
        biggest = _skewed_vs_single(ctx, d, 12000, [0.5, 0.05, 1.0])
    assert biggest > 1000, biggest
    ctx.close()
    print("ok skewed", biggest)


# ------------------------------------------------------------------------------------------------------------------------------
# CPU tests (emulator build)
# ------------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("case", [c["name"] for c in bam2db_cases()])
def test_emu_sweep_reproduces_golden_python(emu_lib, case, tmp_path):
    """every golden bam2db case as one rate of an unsorted sweep (Python host): that rate equals the reference's recorded files and
    tables, every other rate equals the single-rate run (files, tables) and the oracle (counters, COO)"""
    spawn(__file__, emu_lib, ["golden", case, "python", str(tmp_path)])


@pytest.mark.parametrize("case", [c["name"] for c in bam2db_cases()])
def test_emu_sweep_reproduces_golden_cli(emu_lib, emu_cli, case, tmp_path):
    """the same through `fastF bam2db --depths` (C host), -u where the golden case has it"""
    spawn(__file__, emu_lib, ["golden", case, "cli", str(tmp_path)], cli=emu_cli)


def test_emu_sweep_streamed_and_straddling(emu_lib, tmp_path):
    spawn(__file__, emu_lib, ["streaming", str(tmp_path)])


def test_emu_sweep_long_groups(emu_lib):
    """two cells x two genes: (cell, gene) groups of thousands of UMIs, read by fastf_group_rate_kernel in many warp steps"""
    spawn(__file__, emu_lib, ["skewed"])


@pytest.mark.parametrize("extra,needle", [
    (["-r", "0.5", "--depths", "0.1,0.2"], "exclude each other"),
    (["--depths", "0.1,0.5,0.1"], "twice"),
    (["--depths", ",".join("%.2f" % (0.01 * (i + 1)) for i in range(33))], "at most 32"),
    (["--depths", "0.1,0.2", "--gpus", "2"], "one GPU"),
    (["--depths", "0.1,0.2"], "already exists"),
    (["--depths", "0.1,0.2", "--gpus", "1", "FASTF_GPUS=2"], "one GPU"),
    (["-c", "1.5", "--depths", "0.1,0.2"], "Sample size must be smaller"),
])
def test_emu_cli_sweep_refusals(emu_cli, tmp_path, extra, needle):
    """refused before any work (no device job, no database written, no output directory made)"""
    os.makedirs(tmp_path / "out" / "depth_0.2")
    if needle == "already exists":
        open(tmp_path / "out" / "depth_0.2" / "x.db", "wb").close()
    cli_refusal(emu_cli, tmp_path, ["-c", "1.0"] + extra, needle, tmp_path / "out" / "depth_0.1")


# ------------------------------------------------------------------------------------------------------------------------------
# B200
# ------------------------------------------------------------------------------------------------------------------------------
def _single_and_sweep(ctx, bam, inputs, rates, seed):
    from fastf_b200 import bam2db_host as B
    sweep = B.run_device_sweep(ctx, bam, inputs, rates, seed)
    for r, (st, arr) in zip(rates, sweep):
        st1, arr1 = B.run_device(ctx, bam, inputs, r, seed)
        assert [st[k] for k in KEYS] == [st1[k] for k in KEYS], (r, st, st1)
        assert st["status"] == 0 and st["bits_umi"] == st1["bits_umi"] and st["bits_gene"] == st1["bits_gene"]
        for k in ("m_gene", "m_cell", "m_count", "row_keys"):
            assert np.array_equal(arr[k], arr1[k]), (r, k)
    return sweep


@pytest.mark.gpu
def test_gpu_sweep_equals_single_rate_jobs(gpu_ctx, bam_4m, oracle):
    """about 4 M reads, -c 0.5, rates 0.1 .. 1.0 (unsorted): per rate the counters, COO, rows and umi.tsv equal a single-rate job's;
    the oracle agrees at three rates"""
    from fastf_b200 import bam2db_host as B
    rates = [0.5, 0.1, 1.0, 0.3, 0.8, 0.2, 0.9, 0.4, 0.7, 0.6]
    inputs = B.Bam2dbInputs(gpu_ctx.lib, bam_4m["barcodes"], bam_4m["features"], 0.5, 926)
    bam = np.fromfile(bam_4m["bam"], dtype=np.uint8)
    sweep = _single_and_sweep(gpu_ctx, bam, inputs, rates, 926)
    st0 = sweep[0][0]
    assert st0["total"] == 4_000_000 and st0["n_chunks"] >= 1
    for r, (st, arr) in zip(rates, sweep):
        if r in (0.1, 0.5, 1.0):
            o = oracle.bam2db(bam_4m["bam"], bam_4m["barcodes"], bam_4m["features"], 0.5, r, 926)
            assert [st[k] for k in KEYS] == [o[k] for k in KEYS], r
            for k in ("m_gene", "m_cell", "m_count"):
                assert np.array_equal(arr[k], o[k]), (r, k)
        # umi.tsv / numi: the copies of every distinct key among the rate's rows
        u, c = B.unique_counts(gpu_ctx, arr["row_keys"], st["bits_cell"] + st["bits_gene"] + st["bits_umi"])
        wu, wc = np.unique(arr["row_keys"], return_counts=True)
        assert np.array_equal(u, wu) and np.array_equal(c.astype(np.int64), wc), r
    # the subset property the sweep rests on
    for (r1, (s1, _)), (r2, (s2, _)) in zip(sorted(zip(rates, sweep))[:-1], sorted(zip(rates, sweep))[1:]):
        assert s1["sampled"] <= s2["sampled"] and s1["valid"] <= s2["valid"], (r1, r2)


@pytest.mark.gpu
def test_gpu_sweep_threshold_edge_cases(gpu_ctx, bam_4m):
    """NaN, -1, 0, 1.0, inf; (-1, 0) and (1e-12, 2e-12) share a threshold: each equals its single-rate run"""
    from fastf_b200 import bam2db_host as B
    rates = [float("nan"), -1.0, 0.0, 1.0, float("inf"), 1e-12, 2e-12, 0.37]
    lib = gpu_ctx.lib
    import ctypes as C
    thr = [lib.fastf_keep_threshold(C.c_float(r)) for r in rates]
    assert thr[1] == thr[2] and thr[5] == thr[6]
    inputs = B.Bam2dbInputs(lib, bam_4m["barcodes"], bam_4m["features"], 0.5, 926)
    _single_and_sweep(gpu_ctx, np.fromfile(bam_4m["bam"], dtype=np.uint8), inputs, rates, 926)


@pytest.mark.gpu
def test_gpu_sweep_long_groups(gpu_ctx, tmp_path):
    """2 cells x 2 genes, 2 M reads: (cell, gene) groups of hundreds of thousands of UMIs"""
    assert _skewed_vs_single(gpu_ctx, str(tmp_path), 2_000_000, [0.3, 0.01, 1.0, 0.7]) > 100_000


@pytest.mark.gpu
def test_gpu_sweep_one_rate_equals_finish(gpu_ctx, bam_4m):
    from fastf_b200 import bam2db_host as B
    inputs = B.Bam2dbInputs(gpu_ctx.lib, bam_4m["barcodes"], bam_4m["features"], 0.5, 926)
    _single_and_sweep(gpu_ctx, np.fromfile(bam_4m["bam"], dtype=np.uint8), inputs, [0.42], 926)


if __name__ == "__main__":
    assert "libfastf_emu" in os.environ.get("FASTF_GPU_LIB", ""), "this worker is for the emulator build only"
    if sys.argv[1] == "golden":
        _worker_golden(sys.argv[2], sys.argv[3] == "cli", sys.argv[4])
    elif sys.argv[1] == "streaming":
        _worker_streaming(sys.argv[2])
    elif sys.argv[1] == "skewed":
        _worker_skewed()
