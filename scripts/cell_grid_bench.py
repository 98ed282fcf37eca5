#!/usr/bin/env python
"""Cell-rate grid against one depth sweep per cell rate, on one GPU.

    python scripts/cell_grid_bench.py --out DIR [--reads 64000000] [--cli-reads 16000000] [--reps 3]

Device leg: --reads DISTINCT synthetic reads (bench.py's generator and lists, -s 926), compressed image and block index resident in
HBM (fastf_bam2db_feed_device), cell rates 0.25, 0.5, 0.75, 1.0 x depth rates 0.1 .. 1.0.  Per repetition, four depth-sweep jobs
(fastf_bam2db_finish_sweep, one per cell rate, each begun with that rate's cell table) and one grid job (fastf_bam2db_finish_grid over
the union table) run alternately; each job is timed with CUDA events on fastf_compute_stream from before fastf_bam2db_begin to after
its results are on the host, and by the host wall clock.  Both report the library's per-stage clocks (the grid per cell rate).  Every
(cell rate, depth rate)'s counters and a sha256 of its COO must agree between the two, or the script fails.

CLI leg: the first --cli-reads reads (whole blocks) as files on /dev/shm; `fastF bam2db --cells ... --depths ...` once against four
`fastF bam2db -c C --depths ...` runs, host wall clock of the whole processes (CUDA start-up included); every set's matrix.mtx.gz must
be identical between the two.

The GPU name and power limit are read with nvidia-smi in the same run.  Writes DIR/cell_grid.json."""
import argparse
import ctypes as C
import gzip
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.join(ROOT, "scripts"))

from depth_sweep_bench import COUNTERS, RATES, STAGES, coo_hash, gpu_identity   # noqa: E402

CELLS = [0.25, 0.5, 0.75, 1.0]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--reads", type=int, default=64_000_000)
    ap.add_argument("--cli-reads", type=int, default=16_000_000)
    ap.add_argument("--reps", type=int, default=3)
    args = ap.parse_args()
    os.makedirs(args.out, exist_ok=True)
    import torch
    import bench
    from fastf_b200 import _lib, build, bam2db_host as B
    gpu = gpu_identity()
    lib = _lib.load()
    ctx = _lib.Context(0)
    base = bench.make_base(args.reads, os.cpu_count() or 1)
    tmp = tempfile.mkdtemp(prefix="fastf_grid_", dir="/dev/shm" if os.path.isdir("/dev/shm") else None)
    try:
        paths, _ = bench.write_inputs(base, tmp, write_bam=False)
        union = B.Bam2dbInputs.grid(lib, paths["barcodes"], paths["features"], CELLS, bench.SEED)
        bam = np.frombuffer(base["bam"], dtype=np.uint8)
        cap = base["n_blocks"] + 8
        in_off, in_len, isz = np.zeros(cap, np.uint64), np.zeros(cap, np.uint32), np.zeros(cap, np.uint32)
        used = C.c_size_t()
        nb = lib.fastf_bgzf_index_host(C.c_void_p(bam.ctypes.data), bam.size, in_off.ctypes.data_as(_lib.c_u64p), in_len.ctypes.data_as(_lib.c_u32p), isz.ctypes.data_as(_lib.c_u32p), cap, C.byref(used))
        in_off, in_len, isz = in_off[:nb].copy(), in_len[:nb].copy(), isz[:nb].copy()
        dptr = C.c_void_p()
        ctx.check(lib.fastf_device_alloc(ctx.h, bam.size + 64, C.byref(dptr)), "device_alloc")
        ctx.check(lib.fastf_memcpy_h2d(ctx.h, dptr, C.c_void_p(bam.ctypes.data), bam.size), "h2d")
        stream = torch.cuda.ExternalStream(lib.fastf_compute_stream(ctx.h), device=torch.device("cuda", 0))

        def timed(run):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            t = time.perf_counter()
            e0.record(stream)
            out = run()
            e1.record(stream)
            e1.synchronize()
            return e0.elapsed_time(e1), 1e3 * (time.perf_counter() - t), out

        def sweep(table):
            with B.Bam2dbJob(ctx, table, 0.0, bench.SEED, want_rows=False) as job:
                job.feed_device(dptr.value, bam.size, in_off, in_len, isz)
                return job.finish_sweep(RATES)

        def grid():
            with B.Bam2dbJob(ctx, union, 0.0, bench.SEED, want_rows=False, grid=True) as job:
                job.feed_device(dptr.value, bam.size, in_off, in_len, isz)
                return job.finish_grid(B.grid_cell_rates(union), RATES)

        # warm-up: every shape once
        sweep(union.tables[0])
        grid()
        reps = []
        for rep in range(args.reps):
            sweeps_ev, sweeps_wall, sweep_res = [], [], []
            for t in union.tables:
                ev, wall, res = timed(lambda: sweep(t))
                sweeps_ev.append(ev)
                sweeps_wall.append(wall)
                sweep_res.append(res)
            g_ev, g_wall, g = timed(grid)
            for c, per_s, per_g in zip(CELLS, sweep_res, g):
                for r, (s1, a1), (s2, a2) in zip(RATES, per_s, per_g):
                    assert [s1[k] for k in COUNTERS] == [s2[k] for k in COUNTERS], ("counters differ", c, r, s1, s2)
                    assert coo_hash(a1) == coo_hash(a2), ("COO differs", c, r)
            reps.append({"sweep_jobs_ms": [round(x, 2) for x in sweeps_ev], "four_sweep_jobs_ms": round(sum(sweeps_ev), 2), "grid_job_ms": round(g_ev, 2),
                         "four_sweep_jobs_wall_ms": round(sum(sweeps_wall), 2), "grid_job_wall_ms": round(g_wall, 2),
                         "sweep_stages_ms": [{k: round(per[0][0][k], 2) for k in STAGES} for per in sweep_res],
                         "grid_stages_ms_per_cell_rate": [{k: round(per[0][0][k], 2) for k in STAGES} for per in g]})
            print(f"[grid] rep {rep}: four sweep jobs {sum(sweeps_ev):.1f} ms ({sum(sweeps_wall):.1f} wall), one grid job {g_ev:.1f} ms ({g_wall:.1f} wall)", file=sys.stderr, flush=True)
        per_set = [{"rate_cell": c, "rate_depth": r, **{k: int(s[k]) for k in COUNTERS}, "coo_sha256_16": coo_hash(a)} for c, per in zip(CELLS, g) for r, (s, a) in zip(RATES, per)]
        lib.fastf_device_free(ctx.h, dptr)
        med = lambda k: sorted(x[k] for x in reps)[len(reps) // 2]   # noqa: E731
        device = {"reads": base["reads"], "cell_rates": CELLS, "depth_rates": RATES, "cells_per_table": [len(t.cells) for t in union.tables], "union_cells": len(union.cells),
                  "repetitions": reps, "per_set": per_set,
                  "median_four_sweep_jobs_ms": med("four_sweep_jobs_ms"), "median_grid_job_ms": med("grid_job_ms"),
                  "median_four_sweep_jobs_wall_ms": med("four_sweep_jobs_wall_ms"), "median_grid_job_wall_ms": med("grid_job_wall_ms"),
                  "agreement": "per (cell rate, depth rate): total, cb_valid, sampled, valid, nnz and a sha256 of (m_gene, m_cell, m_count) equal between the sweep job and the grid",
                  "timing": "CUDA events on fastf_compute_stream, and the host wall clock, around each whole job (begin, device-resident feed, finish, results on the host)"}

        # ---- CLI: --cells --depths once against four -c --depths runs ----
        cli = build.build_cli()
        cdir = os.path.join(tmp, "cli")
        os.makedirs(cdir)
        cpaths, _ = bench.write_inputs(base, cdir, prefix_reads=min(args.cli_reads, base["reads"]))
        common = ["-b", cpaths["bam"], "-f", cpaths["features"], "-a", cpaths["barcodes"], "-s", str(bench.SEED), "--depths", ",".join(str(x) for x in RATES)]
        os.makedirs(os.path.join(cdir, "grid"))
        t = time.time()
        r = subprocess.run([cli, "bam2db"] + common + ["-d", "grid.db", "-o", os.path.join(cdir, "grid"), "--cells", ",".join(str(c) for c in CELLS)], stdout=subprocess.PIPE,
                           stderr=subprocess.PIPE, text=True, cwd=cdir)
        t_grid = time.time() - t
        assert r.returncode == 0, r.stderr[-2000:]
        t_sweeps = 0.0
        for c in CELLS:
            o = os.path.join(cdir, "c%s" % c)
            os.makedirs(o)
            t = time.time()
            r = subprocess.run([cli, "bam2db"] + common + ["-d", "sweep.db", "-o", o, "-c", str(c)], stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, cwd=cdir)
            t_sweeps += time.time() - t
            assert r.returncode == 0, r.stderr[-2000:]
            for x in RATES:
                a = gzip.open(os.path.join(o, "depth_%s" % x, "matrix.mtx.gz"), "rb").read()
                b = gzip.open(os.path.join(cdir, "grid", "cell_%s" % c, "depth_%s" % x, "matrix.mtx.gz"), "rb").read()
                assert a == b, ("matrix.mtx differs between --cells and -c", c, x)
        cli_leg = {"reads": min(args.cli_reads, base["reads"]), "cells_depths_run_seconds": round(t_grid, 2), "four_depths_runs_seconds": round(t_sweeps, 2),
                   "speedup": round(t_sweeps / t_grid, 2), "compared": "decompressed matrix.mtx.gz of every (cell rate, depth rate) identical",
                   "what": "whole CLI processes, files on /dev/shm -> sqlite databases + gz files; includes CUDA context creation"}
        out = {"gpu": gpu, "device": device, "cli": cli_leg, "build": _lib.build_info()}
        with open(os.path.join(args.out, "cell_grid.json"), "w") as f:
            json.dump(out, f, indent=1)
        print(json.dumps({"gpu": gpu, "median_four_sweep_jobs_ms": device["median_four_sweep_jobs_ms"], "median_grid_job_ms": device["median_grid_job_ms"],
                          "cli": {k: cli_leg[k] for k in ("cells_depths_run_seconds", "four_depths_runs_seconds")}}))
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
        ctx.close()


if __name__ == "__main__":
    main()
