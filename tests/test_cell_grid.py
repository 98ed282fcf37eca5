"""The cell-rate grid (`fastF bam2db --cells`, fastf_b200.bam2db_grid, fastf_bam2db_finish_grid): one pass over the BAM, the exact
output set of every (cell rate, depth rate).  On the CPU through the SIMT-emulator build (this file, run as a script, is the worker the
tests start with FASTF_GPU_LIB pointing at it); on the B200 against single-rate jobs on the same context."""
import ctypes as C
import gzip
import json
import os
import shutil
import subprocess
import sys

import numpy as np
import pytest

from bam2db_harness import FILES, GOLD, KEYS, ROOT, bam2db_cases, bam_4m, cli_refusal, dup_barcodes, emu_cli, emu_lib, same_files, single_run, spawn  # noqa: F401 (fixtures)

ARRAYS = ("m_gene", "m_cell", "m_count", "row_keys")


def _grid_cells(rc):
    """the golden cell rate among 1.0 (d0 = 0) and a smaller rate, unsorted"""
    out = []
    for c in (round(rc / 2, 3), 1.0, rc):
        if c not in out:
            out.append(c)
    return out


def _grid_depths(rd):
    return [r for r in (0.7, 0.25) if r != rd][:1] + [rd]


# ------------------------------------------------------------------------------------------------------------------------------
# worker (runs under the emulator build)
# ------------------------------------------------------------------------------------------------------------------------------
def _imports():
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))


def _grid(cli, cells, depths, seed, umi, out):
    """the grid from the current directory into `out`: --depths with a list of depth rates, -r with one (a number)"""
    import fastf_b200
    if cli:
        dep = ["--depths", ",".join(str(r) for r in depths)] if isinstance(depths, list) else ["-r", str(depths)]
        cmd = [cli, "bam2db", "-b", "in.bam", "-f", "features.tsv.gz", "-a", "barcodes.tsv.gz", "-d", "x.db", "--cells", ",".join(str(c) for c in cells)] + dep + ["-o", out, "-s", str(seed)]
        os.makedirs(out)
        r = subprocess.run(cmd + (["-u"] if umi else []), stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True)
        assert r.returncode == 0, r.stderr
    else:
        assert fastf_b200.bam2db_grid("in.bam", "x.db", out, "barcodes.tsv.gz", "features.tsv.gz", cells, depths, seed) == 0


def _check_against_singles(cli, d, cells, depths, seed, umi, tmp, out, golden=None):
    """every set of the grid in `out` equals the single-rate run (files, tables) and the oracle (counters, COO, through the API); the
    set `golden` = (c, r, expect dir) equals the reference's recorded files and tables instead"""
    from fastf_b200 import _lib, bam2db_host as B
    from dbdigest import db_digest
    import oracle_binding
    O = oracle_binding.load()
    files = FILES + (["umi.tsv.gz"] if umi else [])
    ctx = _lib.Context(0)
    union = B.Bam2dbInputs.grid(ctx.lib, "barcodes.tsv.gz", "features.tsv.gz", cells, seed)
    api = B.run_device_grid(ctx, np.fromfile("in.bam", dtype=np.uint8), union, depths if isinstance(depths, list) else [depths], seed)
    ctx.close()
    for i, c in enumerate(cells):
        for j, r in enumerate(depths if isinstance(depths, list) else [depths]):
            got = os.path.join(out, "cell_" + str(c)) + ("/depth_" + str(r) if isinstance(depths, list) else "")
            if golden and (c, r) == golden[:2]:
                assert same_files(got, golden[2], files), (d, c, r)
                assert db_digest(os.path.join(got, "x.db")) == json.load(open(os.path.join(golden[2], "db_digest.json"))), (d, c, r)
                continue
            want = os.path.join(tmp, "single_%d_%d" % (i, j))
            single_run(cli, c, r, seed, umi, want)
            assert same_files(got, want, files), (d, c, r)
            assert db_digest(os.path.join(got, "x.db")) == db_digest(os.path.join(want, "x.db")), (d, c, r)
            o = O.bam2db(os.path.join(os.getcwd(), "in.bam"), os.path.join(os.getcwd(), "barcodes.tsv.gz"), os.path.join(os.getcwd(), "features.tsv.gz"), c, r, seed)
            st, arr = api[i][j]
            assert [st[x] for x in KEYS] == [o[x] for x in KEYS], (d, c, r)
            for x in ("m_gene", "m_cell", "m_count"):
                assert np.array_equal(arr[x], o[x]), (d, c, r, x)
    return union, api


def _worker_golden(case_name, use_cli, tmp):
    _imports()
    from fastf_b200 import bam2db_host as B
    c = {c["name"]: c for c in bam2db_cases()}[case_name]
    d = os.path.join(GOLD, c["dir"])
    rc_, rd, seed, umi = c["rate_cell"], c["rate_depth"], c["seed"], bool(c.get("umicopies"))
    cli = os.environ.get("FASTF_EMU_CLI") if use_cli else None
    B._umi_copies_flag = 1 if umi else 0
    os.chdir(d)   # the matrix header records the BAM path as passed: the golden run used "in.bam"
    cells, depths = _grid_cells(rc_), _grid_depths(rd)
    out = os.path.join(tmp, "grid")
    _grid(cli, cells, depths, seed, umi, out)
    _check_against_singles(cli, case_name, cells, depths, seed, umi, tmp, out, golden=(rc_, rd, os.path.join(d, c["expect"])))
    print("ok", case_name, "cli" if cli else "python")


def _worker_duplicates(use_cli, tmp):
    _imports()
    from fastf_b200 import _lib, bam2db_host as B
    cli = os.environ.get("FASTF_EMU_CLI") if use_cli else None
    B._umi_copies_flag = 1
    w, seed = dup_barcodes(tmp, _lib.load())
    os.chdir(w)
    cells, depths = [1.0, 0.5, 0.8], [0.6, 1.0]
    out = os.path.join(tmp, "grid")
    _grid(cli, cells, depths, seed, True, out)
    union, _ = _check_against_singles(cli, "dup", cells, depths, seed, True, tmp, out)
    # the union is not the largest table
    assert set(union.tables[1].cells) - set(union.tables[0].cells) and len(union.cells) > len(union.tables[0].cells)
    print("ok duplicates", seed)


def _worker_edge(use_cli, tmp):
    """a cell rate that samples no cell, 1.0 and 0.99 side by side; the -r layout (OUT/cell_<c>/); reads that consume a draw but would
    not be inserted, in cells only some tables hold"""
    _imports()
    from fastf_b200 import bam2db_host as B
    cli = os.environ.get("FASTF_EMU_CLI") if use_cli else None
    B._umi_copies_flag = 0
    for d, cells in (("synth4k", [0.99, 0.01, 1.0, 0.6]), ("edge", [1.0, 0.99, 0.02])):
        os.chdir(os.path.join(GOLD, d))
        t = os.path.join(tmp, d)
        out = os.path.join(t, "grid")
        _grid(cli, cells, 0.5, 926, False, out)
        union, api = _check_against_singles(cli, d, cells, 0.5, 926, False, t, out)
        sizes = [len(x.cells) for x in union.tables]
        assert 0 in sizes and max(sizes) == len(union.cells), sizes
        if d == "synth4k":
            # reads that consume a draw but would not be inserted lie in cells that only some tables hold
            from fastf_b200 import _lib
            with _lib.Context(0) as ctx:
                st, _ = B.run_device(ctx, np.fromfile("in.bam", dtype=np.uint8), union.tables[3], 1.0, 926)
            assert 0 < sizes[3] < len(union.cells) and st["cb_valid"] > st["valid"] and api[3][0][0]["cb_valid"] == st["cb_valid"], st
    print("ok edge", "cli" if cli else "python")


def _worker_streaming(tmp):
    """the same grid from many streamed chunks and odd feed pieces, and on a BAM whose records straddle BGZF blocks"""
    _imports()
    import fastf_b200
    import bamgen
    from fastf_b200 import _lib, bam2db_host as B
    from dbdigest import db_digest
    ctx = _lib.Context(0)
    cells, depths = [0.8, 0.3, 1.0], [0.9, 0.1, 1.0]
    for d in ("edge", "synth4k"):
        g = os.path.join(GOLD, d)
        union = B.Bam2dbInputs.grid(ctx.lib, os.path.join(g, "barcodes.tsv.gz"), os.path.join(g, "features.tsv.gz"), cells, 926)
        bam = np.fromfile(os.path.join(g, "in.bam"), dtype=np.uint8)
        ref = None
        for chunk, piece in ((0, 0), (1 << 20, 777), (1 << 20, 50001)):
            res = B.run_device_grid(ctx, bam, union, depths, 926, chunk_inflated_bytes=chunk, feed_piece=piece)
            key = [[(tuple(st[x] for x in KEYS), tuple(a[x].tobytes() for x in ARRAYS)) for st, a in per] for per in res]
            if ref is None:
                ref = key
                for i, t in enumerate(union.tables):   # and the single-rate sweep over each table
                    sw = B.run_device_sweep(ctx, bam, t, depths, 926)
                    assert key[i] == [(tuple(st[x] for x in KEYS), tuple(a[x].tobytes() for x in ARRAYS)) for st, a in sw], (d, i)
            assert key == ref, (d, chunk, piece)
        w = os.path.join(tmp, d)
        os.makedirs(w)
        whole = gzip.decompress(open(os.path.join(g, "in.bam"), "rb").read())
        cut = 997 if d == "edge" else 30011
        open(os.path.join(w, "in.bam"), "wb").write(bamgen.bgzf_file([whole[i:i + cut] for i in range(0, len(whole), cut)]))
        for f in ("barcodes.tsv.gz", "features.tsv.gz"):
            shutil.copy(os.path.join(g, f), w)
        os.chdir(w)
        B._umi_copies_flag = 1
        assert fastf_b200.bam2db_grid("in.bam", "x.db", os.path.join(w, "cut"), "barcodes.tsv.gz", "features.tsv.gz", cells, depths, 926, ctx=ctx) == 0
        os.chdir(g)
        assert fastf_b200.bam2db_grid("in.bam", "x.db", os.path.join(w, "orig"), "barcodes.tsv.gz", "features.tsv.gz", cells, depths, 926, ctx=ctx) == 0
        for c in cells:
            for r in depths:
                a, b = os.path.join(w, "cut", "cell_%s" % c, "depth_%s" % r), os.path.join(w, "orig", "cell_%s" % c, "depth_%s" % r)
                assert same_files(a, b, FILES + ["umi.tsv.gz"]), (d, c, r)
                assert db_digest(os.path.join(a, "x.db")) == db_digest(os.path.join(b, "x.db")), (d, c, r)
        print("ok", d)
    ctx.close()


def _expect_fail(ctx, rc, needle):
    from fastf_b200 import _lib
    assert rc != 0, needle
    msg = ctx.lib.fastf_last_error(ctx.h).decode()
    assert needle in msg, (needle, msg)


def _worker_library_refusals():
    _imports()
    from fastf_b200 import _lib, bam2db_host as B
    ctx = _lib.Context(0)
    lib = ctx.lib
    g = os.path.join(GOLD, "synth4k")
    union = B.Bam2dbInputs.grid(lib, os.path.join(g, "barcodes.tsv.gz"), os.path.join(g, "features.tsv.gz"), [0.5, 1.0], 926)
    bam = np.fromfile(os.path.join(g, "in.bam"), dtype=np.uint8)
    thr = np.array([lib.fastf_keep_threshold(C.c_float(0.5))], dtype=np.uint64)
    rows = (_lib.Bam2dbSweepResult * 33)()

    def grid_job():
        j = B.Bam2dbJob(ctx, union, 0.0, 926, grid=True)
        B._feed_all(j, bam, 0)
        return j

    def finish_grid(j, crs):
        arr = (_lib.Bam2dbCellRate * max(len(crs), 1))()
        keep = []
        for k, (m, n, d0) in enumerate(crs):
            m = np.ascontiguousarray(m, dtype=np.uint32)
            keep.append(m)
            arr[k].cell_index, arr[k].n_cells, arr[k].d0 = m.ctypes.data_as(_lib.c_u32p), n, d0
        rc = lib.fastf_bam2db_finish_grid(j.job, len(crs), arr, 1, thr.ctypes.data_as(_lib.c_u64p), rows)
        for k in range(33):
            lib.fastf_bam2db_sweep_result_free(C.byref(rows[k]))
        return rc

    good = B.grid_cell_rates(union)
    # wrong kind of job, both ways
    with B.Bam2dbJob(ctx, union.tables[0], 0.5, 926) as j:
        B._feed_all(j, bam, 0)
        _expect_fail(ctx, finish_grid(j, good), "not begun with fastf_bam2db_begin_grid")
    for call in ("finish", "finish_sweep", "sample", "sample_sweep"):
        with grid_job() as j:
            if call == "finish":
                rc = lib.fastf_bam2db_finish(j.job, C.byref(_lib.Bam2dbResult()))
            elif call == "finish_sweep":
                rc = lib.fastf_bam2db_finish_sweep(j.job, 1, thr.ctypes.data_as(_lib.c_u64p), C.byref(rows[0]))
                lib.fastf_bam2db_sweep_result_free(C.byref(rows[0]))
            elif call == "sample":
                rc = lib.fastf_bam2db_sample(j.job, 0)
            else:
                rc = lib.fastf_bam2db_sample_sweep(j.job, 0, 1, thr.ctypes.data_as(_lib.c_u64p), None, None)
            _expect_fail(ctx, rc, "begun with fastf_bam2db_begin_grid")
    # cell_index out of range, repeated; a table that is not inside the union; 0 and 33 cell rates
    m0, n0, d00 = good[0]
    big = m0.copy()
    big[np.nonzero(big)[0][0]] = n0 + 1
    rep = m0.copy()
    nz = np.nonzero(rep)[0]
    rep[nz[1]] = rep[nz[0]]
    for crs, needle in (([(big, n0, d00)], "exceeds its n_cells"), ([good[1], (rep, n0, d00)], "twice"), ([(m0, n0 + 1, d00)], "maps"),
                        ([(m0, len(union.cells) + 1, d00)], "exceeds the union"), ([], "1..32 cell rates"), ([good[0]] * 33, "1..32 cell rates")):
        with grid_job() as j:
            _expect_fail(ctx, finish_grid(j, crs), needle)
    # and a good call after all of these, on the same context
    with grid_job() as j:
        assert finish_grid(j, good) == 0
        _expect_fail(ctx, finish_grid(j, good), "already finished")
    ctx.close()
    print("ok library refusals")


# ------------------------------------------------------------------------------------------------------------------------------
# CPU tests (emulator build)
# ------------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("case", [c["name"] for c in bam2db_cases()])
def test_emu_grid_reproduces_golden_python(emu_lib, case, tmp_path):
    """every golden bam2db case as one set of an unsorted grid with cell rate 1.0 and a smaller one (Python host): that set equals the
    reference's recorded files and tables, every other set equals the single-rate run (files, tables) and the oracle (counters, COO)"""
    spawn(__file__, emu_lib, ["golden", case, "python", str(tmp_path)])


@pytest.mark.parametrize("case", [c["name"] for c in bam2db_cases()])
def test_emu_grid_reproduces_golden_cli(emu_lib, emu_cli, case, tmp_path):
    """the same through `fastF bam2db --cells --depths` (C host), -u where the golden case has it"""
    spawn(__file__, emu_lib, ["golden", case, "cli", str(tmp_path)], cli=emu_cli)


@pytest.mark.parametrize("host", ["python", "cli"])
def test_emu_grid_duplicate_barcodes(emu_lib, emu_cli, host, tmp_path):
    """a smaller cell rate's table holds a barcode the largest rate's table lacks: the union of the tables, not the largest one"""
    spawn(__file__, emu_lib, ["duplicates", host, str(tmp_path)], cli=emu_cli if host == "cli" else None)


@pytest.mark.parametrize("host", ["python", "cli"])
def test_emu_grid_edge_cell_rates(emu_lib, emu_cli, host, tmp_path):
    """a cell rate that samples no cell, 1.0 next to 0.99, one depth rate (-r: OUT/cell_<c>/)"""
    spawn(__file__, emu_lib, ["edge", host, str(tmp_path)], cli=emu_cli if host == "cli" else None)


def test_emu_grid_streamed_and_straddling(emu_lib, tmp_path):
    spawn(__file__, emu_lib, ["streaming", str(tmp_path)])


def test_emu_grid_library_refusals(emu_lib):
    spawn(__file__, emu_lib, ["refusals"])


@pytest.mark.parametrize("extra,needle", [
    (["-c", "0.5", "--cells", "0.2,0.4", "-r", "0.5"], "exclude each other"),
    (["--cells", "0.2,0.4"], "needs -r or --depths"),
    (["--cells", "0.5,0.2,0.5", "-r", "0.5"], "twice"),
    (["--cells", "0.5,0.50", "-r", "0.5"], "twice"),
    (["--cells", ",".join("%.2f" % (0.01 * (i + 1)) for i in range(33)), "-r", "0.5"], "at most 32"),
    (["--cells", "0.2,1.5", "--depths", "0.1,0.2"], "Sample size must be smaller"),
    (["--cells", "0.2,0.4", "-r", "0.5", "--gpus", "2"], "one GPU"),
    (["--cells", "0.2,0.4", "--depths", "0.1,0.2", "--gpus", "1", "FASTF_GPUS=2"], "one GPU"),
    (["--cells", "0.2,0.4", "--depths", "0.1,0.2"], "already exists"),
    (["--cells", "0.2,0.4", "-r", "0.5"], "already exists"),
])
def test_emu_cli_grid_refusals(emu_cli, tmp_path, extra, needle):
    """refused before any work (no device job, no database written, no output directory made)"""
    if needle == "already exists":
        where = tmp_path / "out" / "cell_0.4" / ("depth_0.2" if "--depths" in extra else "")
        os.makedirs(where, exist_ok=True)
        open(where / "x.db", "wb").close()
    cli_refusal(emu_cli, tmp_path, extra, needle, tmp_path / "out" / "cell_0.2")


# ------------------------------------------------------------------------------------------------------------------------------
# B200
# ------------------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_gpu_grid_equals_single_rate_jobs(gpu_ctx, bam_4m, oracle):
    """about 4 M reads in several chunks, cell rates {0.25, 0.5, 0.8, 1.0} x depths {0.1, 0.3, 0.5, 0.7, 1.0} (unsorted): every set's
    counters, COO and rows equal a single-rate job's on the same context; the oracle agrees at three sets"""
    from fastf_b200 import bam2db_host as B
    cells, depths = [0.5, 1.0, 0.25, 0.8], [0.3, 1.0, 0.1, 0.7, 0.5]
    chunk = 64 << 20
    union = B.Bam2dbInputs.grid(gpu_ctx.lib, bam_4m["barcodes"], bam_4m["features"], cells, 926)
    bam = np.fromfile(bam_4m["bam"], dtype=np.uint8)
    grid = B.run_device_grid(gpu_ctx, bam, union, depths, 926, chunk_inflated_bytes=chunk)
    assert grid[0][0][0]["n_chunks"] > 1 and grid[0][0][0]["total"] == 4_000_000
    for i, (c, t) in enumerate(zip(cells, union.tables)):
        for j, r in enumerate(depths):
            st, arr = grid[i][j]
            st1, arr1 = B.run_device(gpu_ctx, bam, t, r, 926, chunk_inflated_bytes=chunk)
            assert [st[k] for k in KEYS] == [st1[k] for k in KEYS], (c, r, st, st1)
            assert st["status"] == 0 and (st["bits_cell"], st["bits_gene"], st["bits_umi"]) == (st1["bits_cell"], st1["bits_gene"], st1["bits_umi"])
            for k in ARRAYS:
                assert np.array_equal(arr[k], arr1[k]), (c, r, k)
            if (c, r) in ((0.25, 0.1), (0.8, 0.5), (1.0, 1.0)):
                o = oracle.bam2db(bam_4m["bam"], bam_4m["barcodes"], bam_4m["features"], c, r, 926)
                assert [st[k] for k in KEYS] == [o[k] for k in KEYS], (c, r)
                for k in ("m_gene", "m_cell", "m_count"):
                    assert np.array_equal(arr[k], o[k]), (c, r, k)


@pytest.mark.gpu
def test_gpu_grid_one_by_one_equals_finish(gpu_ctx, bam_4m):
    from fastf_b200 import bam2db_host as B
    union = B.Bam2dbInputs.grid(gpu_ctx.lib, bam_4m["barcodes"], bam_4m["features"], [0.6], 926)
    bam = np.fromfile(bam_4m["bam"], dtype=np.uint8)
    (((st, arr),),) = B.run_device_grid(gpu_ctx, bam, union, [0.42], 926)
    st1, arr1 = B.run_device(gpu_ctx, bam, union.tables[0], 0.42, 926)
    assert [st[k] for k in KEYS + ("bits_cell",)] == [st1[k] for k in KEYS + ("bits_cell",)]
    for k in ARRAYS:
        assert np.array_equal(arr[k], arr1[k]), k


if __name__ == "__main__":
    assert "libfastf_emu" in os.environ.get("FASTF_GPU_LIB", ""), "this worker is for the emulator build only"
    if sys.argv[1] == "golden":
        _worker_golden(sys.argv[2], sys.argv[3] == "cli", sys.argv[4])
    elif sys.argv[1] == "duplicates":
        _worker_duplicates(sys.argv[2] == "cli", sys.argv[3])
    elif sys.argv[1] == "edge":
        _worker_edge(sys.argv[2] == "cli", sys.argv[3])
    elif sys.argv[1] == "streaming":
        _worker_streaming(sys.argv[2])
    elif sys.argv[1] == "refusals":
        _worker_library_refusals()
