"""TEST INFRASTRUCTURE shared by the tests of the bam2db runs with several output sets (test_depth_sweep, test_cell_grid,
test_bam2db_hosts): the golden cases, the emulator builds, the worker launcher, one single-rate run, the CLI refusal check and the
B200 input.  A test module imports the fixtures it uses from here."""
import gzip
import json
import os
import shutil
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden")
FILES = ["matrix.mtx.gz", "barcodes.tsv.gz", "features.tsv.gz"]
KEYS = ("total", "cb_valid", "sampled", "valid", "nnz")


def bam2db_cases():
    return [c for c in json.load(open(os.path.join(GOLD, "manifest.json")))["cases"] if c["kind"] == "bam2db"]


def same_files(a, b, files):
    return all(gzip.open(os.path.join(a, f), "rb").read() == gzip.open(os.path.join(b, f), "rb").read() for f in files)


def single_run(cli, rc_, rate, seed, umi, where):
    """one `-c rc_ -r rate` run (Python host, or the C CLI `cli`) from the current directory into `where`"""
    import fastf_b200
    os.makedirs(where)
    if cli:
        cmd = [cli, "bam2db", "-b", "in.bam", "-f", "features.tsv.gz", "-a", "barcodes.tsv.gz", "-d", os.path.join(where, "x.db"), "-c", str(rc_), "-r", str(rate), "-o", where, "-s", str(seed)]
        assert subprocess.run(cmd + (["-u"] if umi else []), stdout=subprocess.DEVNULL).returncode == 0
    else:
        assert fastf_b200.bam2db("in.bam", os.path.join(where, "x.db"), where, "barcodes.tsv.gz", "features.tsv.gz", rc_, rate, seed) == 0


def dup_barcodes(tmp, lib):
    """synth4k with a barcode list that repeats one barcode: the seed is chosen (deterministically, by fastf_sample_cells through
    Bam2dbInputs) so that the 0.5 table holds a barcode the 1.0 table lacks -- the 1.0 table stops at the repeated line"""
    from fastf_b200 import bam2db_host as B
    g = os.path.join(GOLD, "synth4k")
    lines = gzip.decompress(open(os.path.join(g, "barcodes.tsv.gz"), "rb").read()).splitlines(keepends=True)
    w = os.path.join(tmp, "dup")
    os.makedirs(w)
    with gzip.open(os.path.join(w, "barcodes.tsv.gz"), "wb") as f:
        f.write(b"".join(lines[:20] + [lines[3]] + lines[20:]))
    for x in ("in.bam", "features.tsv.gz"):
        shutil.copy(os.path.join(g, x), w)
    for seed in range(1, 1000):
        small = B.Bam2dbInputs(lib, os.path.join(w, "barcodes.tsv.gz"), os.path.join(w, "features.tsv.gz"), 0.5, seed)
        full = B.Bam2dbInputs(lib, os.path.join(w, "barcodes.tsv.gz"), os.path.join(w, "features.tsv.gz"), 1.0, seed)
        if set(small.cells) - set(full.cells):
            return w, seed
    raise AssertionError("no seed below 1000 gives a 0.5 table with a barcode the 1.0 table lacks")


@pytest.fixture(scope="module")
def emu_lib():
    from fastf_b200 import build
    return build.build_emu()


@pytest.fixture(scope="module")
def emu_cli(emu_lib):
    from fastf_b200 import build
    return build.build_cli(emu=True)


def spawn(script, emu_lib, args, cli=None):
    """run the worker `script` with `args` under the emulator build (and the emulator CLI `cli`); it prints "ok ..." when it passes"""
    env = dict(os.environ, FASTF_GPU_LIB=emu_lib)
    if cli:
        env["FASTF_EMU_CLI"] = cli
    r = subprocess.run([sys.executable, os.path.abspath(script)] + args, env=env, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=1500)
    assert r.returncode == 0 and "ok " in r.stdout, r.stdout[-3000:]


def cli_refusal(cli, tmp_path, args, needle, absent):
    """`fastF bam2db` on synth4k with `args` (KEY=VALUE items set the environment instead), from tmp_path into tmp_path/out, is refused
    before any work: exit code 1, `needle` on stderr, no directory `absent`, no database written"""
    env = dict(os.environ)
    env.pop("FASTF_GPUS", None)
    env.update(x.split("=", 1) for x in args if "=" in x)
    g = os.path.join(GOLD, "synth4k")
    cmd = [cli, "bam2db", "-b", os.path.join(g, "in.bam"), "-f", os.path.join(g, "features.tsv.gz"), "-a", os.path.join(g, "barcodes.tsv.gz"), "-d", "x.db",
           "-o", str(tmp_path / "out")] + [x for x in args if "=" not in x]
    r = subprocess.run(cmd, cwd=tmp_path, env=env, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=600)
    assert r.returncode == 1 and needle in r.stderr, (r.returncode, r.stderr)
    assert not os.path.exists(absent), "a refused run created an output directory"
    assert not os.path.exists(tmp_path / "x.db")


@pytest.fixture(scope="module")
def bam_4m(tmp_path_factory, synth):
    d = str(tmp_path_factory.mktemp("bam4m"))
    paths, st = synth.write_bam_set(d, n_reads=4_000_000, n_cells=3000, n_genes=20000, seed=11, p_umi_n=0.01, n_molecules=1_500_000)
    return paths
