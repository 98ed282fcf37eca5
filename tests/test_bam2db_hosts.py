"""The C host (`fastF bam2db`) and the Python host (fastf_b200.bam2db / bam2db_sweep / bam2db_grid) side by side, in every run shape:
-c/-r, -c/--depths, --cells/-r and --cells/--depths.  Both run from the same directory on the same inputs into two trees, which must
hold the same files, the same .gz contents and the same tables, and both must print the same stdout and stderr lines.  On the CPU through
the SIMT-emulator build (this file, run as a script, is the worker that runs the Python host)."""
import gzip
import json
import os
import subprocess
import sys

import pytest

from bam2db_harness import GOLD, ROOT, bam2db_cases, dup_barcodes, emu_cli, emu_lib  # noqa: F401 (fixtures)

SHAPES = ("c_r", "c_depths", "cells_r", "cells_depths")
CASES = {c["name"]: c for c in bam2db_cases()}


def _rates(shape, rc_, rd):
    """(cell axis, depth axis) of a shape: a list for --cells / --depths, one number for -c / -r"""
    cells = [rc_] + [c for c in (1.0, 0.5) if c != rc_][:1]
    depths = [rd] + [r for r in (0.2, 0.7) if r != rd][:1]
    return (cells if shape.startswith("cells") else rc_), (depths if shape.endswith("depths") else rd)


def _cli_args(cells, depths, db, out, seed, umi):
    axis = lambda opt, many, v: [many, ",".join(str(x) for x in v)] if isinstance(v, list) else [opt, str(v)]
    return (["-b", "in.bam", "-f", "features.tsv.gz", "-a", "barcodes.tsv.gz", "-d", db] + axis("-c", "--cells", cells) + axis("-r", "--depths", depths) +
            ["-o", out, "-s", str(seed)] + (["-u"] if umi else []))


def _worker_host(spec):
    """the Python host's run of `spec` from the current directory; exits with its return code"""
    sys.path.insert(0, ROOT)
    import fastf_b200
    from fastf_b200 import bam2db_host as B
    cells, depths, out, seed = spec["cells"], spec["depths"], spec["out"], spec["seed"]
    B._umi_copies_flag = 1 if spec["umi"] else 0
    if isinstance(cells, list):
        rc = fastf_b200.bam2db_grid("in.bam", "x.db", out, "barcodes.tsv.gz", "features.tsv.gz", cells, depths, seed)
    elif isinstance(depths, list):
        rc = fastf_b200.bam2db_sweep("in.bam", "x.db", out, "barcodes.tsv.gz", "features.tsv.gz", cells, depths, seed)
    else:
        rc = fastf_b200.bam2db("in.bam", os.path.join(out, "x.db"), out, "barcodes.tsv.gz", "features.tsv.gz", cells, depths, seed)
    sys.stdout.flush()
    sys.exit(rc)


def _worker_dup(tmp):
    sys.path.insert(0, ROOT)
    from fastf_b200 import _lib
    w, seed = dup_barcodes(tmp, _lib.load())
    print(json.dumps([w, seed]))


def _tree(root):
    return sorted(os.path.relpath(os.path.join(d, f), root) for d, _, fs in os.walk(root) for f in fs)


def _both_hosts(emu_lib, cli, where, tmp, cells, depths, seed, umi):
    """the CLI and the Python host from `where` into tmp/cli and tmp/py: the same trees, .gz contents, tables and lines"""
    from dbdigest import db_digest
    env = dict(os.environ, FASTF_GPU_LIB=emu_lib)
    env.pop("FASTF_GPUS", None)
    runs = {}
    for host in ("cli", "py"):
        out = os.path.join(tmp, host)
        os.makedirs(out)
        if host == "cli":
            db = os.path.join(out, "x.db") if not isinstance(cells, list) and not isinstance(depths, list) else "x.db"
            cmd = [cli, "bam2db"] + _cli_args(cells, depths, db, out, seed, umi)
        else:
            cmd = [sys.executable, os.path.abspath(__file__), "host", json.dumps(dict(cells=cells, depths=depths, out=out, seed=seed, umi=umi))]
        r = subprocess.run(cmd, cwd=where, env=env, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=900)
        assert r.returncode == 0, (host, r.stdout[-2000:], r.stderr[-2000:])
        runs[host] = [s.replace(out, "<OUT>").splitlines() for s in (r.stdout, r.stderr)]
    a, b = os.path.join(tmp, "cli"), os.path.join(tmp, "py")
    assert _tree(a) == _tree(b)
    assert any(f.endswith(".db") for f in _tree(a))
    for f in _tree(a):
        if f.endswith(".gz"):
            assert gzip.open(os.path.join(a, f), "rb").read() == gzip.open(os.path.join(b, f), "rb").read(), f
        elif f.endswith(".db"):
            assert db_digest(os.path.join(a, f)) == db_digest(os.path.join(b, f)), f
    for k, stream in enumerate(("stdout", "stderr")):
        assert runs["cli"][k] == runs["py"][k], (stream, runs["cli"][k], runs["py"][k])


@pytest.mark.parametrize("shape", SHAPES)
@pytest.mark.parametrize("case", ["synth4k-c0.5-r0.5-s926", "edge-c0.8-r0.6-s3"])
def test_emu_hosts_print_and_write_the_same(emu_lib, emu_cli, case, shape, tmp_path):
    """a golden case (synth4k with -u, and edge) in each run shape"""
    c = CASES[case]
    cells, depths = _rates(shape, c["rate_cell"], c["rate_depth"])
    _both_hosts(emu_lib, emu_cli, os.path.join(GOLD, c["dir"]), str(tmp_path), cells, depths, c["seed"], bool(c.get("umicopies")))


def test_emu_hosts_agree_on_duplicate_barcodes(emu_lib, emu_cli, tmp_path):
    """a grid whose 0.5 table holds a barcode the 1.0 table lacks: each table's duplicate-barcode warning, in its place"""
    r = subprocess.run([sys.executable, os.path.abspath(__file__), "dup", str(tmp_path)], env=dict(os.environ, FASTF_GPU_LIB=emu_lib), stdout=subprocess.PIPE, text=True,
                       timeout=900)
    assert r.returncode == 0, r.stdout
    w, seed = json.loads(r.stdout.splitlines()[-1])
    _both_hosts(emu_lib, emu_cli, w, str(tmp_path / "runs"), [1.0, 0.5], [0.6, 1.0], seed, True)


if __name__ == "__main__":
    assert "libfastf_emu" in os.environ.get("FASTF_GPU_LIB", ""), "this worker is for the emulator build only"
    if sys.argv[1] == "host":
        _worker_host(json.loads(sys.argv[2]))
    elif sys.argv[1] == "dup":
        _worker_dup(sys.argv[2])
