#!/usr/bin/env python
"""Depth sweep against one job per rate, on one GPU (BASELINE.json configs[4]: -r 0.1 .. 1.0 at a fixed seed).

    python scripts/depth_sweep_bench.py --out DIR [--reads 64000000] [--cli-reads 16000000] [--reps 3]

Device leg: --reads DISTINCT synthetic reads (bench.py's generator and lists, -c 1.0 -s 926), compressed image and block index
resident in HBM (fastf_bam2db_feed_device).  Per repetition, ten single-rate jobs (rates 0.1 .. 1.0) and one sweep job
(fastf_bam2db_finish_sweep over the same ten rates) run alternately; each job is timed with CUDA events on fastf_compute_stream
from before fastf_bam2db_begin to after its results are on the host.  Both report the library's per-stage clocks.  Every rate's
counters and a sha256 of its COO must agree between the two, or the script fails.

CLI leg: the first --cli-reads reads (whole blocks) as files on /dev/shm; `fastF bam2db --depths 0.1,...,1.0` once against ten
`fastF bam2db -r R` runs, host wall clock of the whole processes (CUDA start-up included); every rate's matrix.mtx.gz must be
identical between the two.

The GPU name and power limit are read with nvidia-smi in the same run.  Writes DIR/depth_sweep.json.

    python scripts/depth_sweep_bench.py --out DIR --gpus G [--reads N] [--reps 3]

Multi-GPU leg instead (the one-process driver of the library): one BAM image of --reads distinct reads (default 64 M per GPU) in host
memory.  Per repetition, ten fastf_bam2db_run_sharded calls (one per rate) and one fastf_bam2db_run_sharded_sweep over the same ten
rates run alternately over devices 0..G-1; each call is timed by the host wall clock and includes what the driver does inside it:
context creation on every device, H2D copies of the shards, and the copy of the results to the host.  Both report the library's
stage clocks (maximum over devices; the sweep's ms_sort / ms_count are its local unique + partition and its receiving-side count).  As
the scaling reference, the one-GPU sweep (fastf_bam2db_finish_sweep, host-fed, context creation included) on the same image.  Every
rate's counters and COO hash must agree between the three, or the script fails.  Writes DIR/depth_sweep_<G>gpu.json."""
import argparse
import ctypes as C
import gzip
import hashlib
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

RATES = [0.1, 0.2, 0.3, 0.4, 0.5, 0.6, 0.7, 0.8, 0.9, 1.0]
STAGES = ("ms_inflate", "ms_crc", "ms_parse", "ms_gather", "ms_mt", "ms_sample", "ms_sort", "ms_count", "ms_device_total")
COUNTERS = ("total", "cb_valid", "sampled", "valid", "nnz")


def gpu_identity():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True)
    if r.returncode != 0:
        raise RuntimeError("nvidia-smi failed: " + r.stderr)
    name, power = [x.strip() for x in r.stdout.splitlines()[0].split(",")]
    return {"name": name, "power_limit": power}


def coo_hash(arr):
    h = hashlib.sha256()
    for k in ("m_gene", "m_cell", "m_count"):
        h.update(np.ascontiguousarray(arr[k]).tobytes())
    return h.hexdigest()[:16]


def gpus_identity(n):
    r = subprocess.run(["nvidia-smi", "--query-gpu=index,name,power.limit", "--format=csv,noheader"], stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True)
    if r.returncode != 0:
        raise RuntimeError("nvidia-smi failed: " + r.stderr)
    rows = [[x.strip() for x in ln.split(",")] for ln in r.stdout.splitlines() if ln.strip()]
    if len(rows) < n:
        raise RuntimeError("%d GPUs requested, %d present" % (n, len(rows)))
    return [{"index": int(i), "name": name, "power_limit": power} for i, name, power in rows[:n]]


def main_multi(args):
    """--gpus G: K x run_sharded against one run_sharded_sweep, and the one-GPU sweep as the scaling reference"""
    import bench
    from fastf_b200 import _lib, bam2db_host as B
    G = args.gpus
    gpus = gpus_identity(G)
    lib = _lib.load()
    reads = args.reads or 64_000_000 * G
    base = bench.make_base(reads, os.cpu_count() or 1)
    tmp = tempfile.mkdtemp(prefix="fastf_sweep_", dir="/dev/shm" if os.path.isdir("/dev/shm") else None)
    try:
        paths, _ = bench.write_inputs(base, tmp, write_bam=False)
        inputs = B.Bam2dbInputs(lib, paths["barcodes"], paths["features"], bench.RATE_CELL, bench.SEED)
        bam = np.frombuffer(base["bam"], dtype=np.uint8)

        def wall(run):
            t = time.perf_counter()
            out = run()
            return 1e3 * (time.perf_counter() - t), out

        def one_gpu():
            with _lib.Context(0) as ctx:
                return B.run_device_sweep(ctx, bam, inputs, RATES, bench.SEED, want_rows=False)

        def check(what, got, ref):
            for r, (s1, a1), (s2, a2) in zip(RATES, ref, got):
                assert [s1[k] for k in COUNTERS] == [s2[k] for k in COUNTERS], (what, "counters differ", r)
                assert coo_hash(a1) == coo_hash(a2), (what, "COO differs", r)

        # warm-up: every path once
        ref = one_gpu()
        B.run_sharded(lib, bam, inputs, RATES[0], bench.SEED, G, want_rows=False)
        B.run_sharded_sweep(lib, bam, inputs, RATES, bench.SEED, G, want_rows=False)
        reps = []
        for rep in range(args.reps):
            singles, single_res = [], []
            for r in RATES:
                ms, res = wall(lambda: B.run_sharded(lib, bam, inputs, r, bench.SEED, G, want_rows=False))
                singles.append(ms)
                single_res.append(res)
            ms_sweep, sweep = wall(lambda: B.run_sharded_sweep(lib, bam, inputs, RATES, bench.SEED, G, want_rows=False))
            ms_one, one = wall(one_gpu)
            check("run_sharded", single_res, ref)
            check("run_sharded_sweep", sweep, ref)
            check("one-GPU finish_sweep", one, ref)
            reps.append({"run_sharded_ms": [round(x, 2) for x in singles], "ten_run_sharded_ms": round(sum(singles), 2), "run_sharded_sweep_ms": round(ms_sweep, 2),
                         "one_gpu_sweep_ms": round(ms_one, 2),
                         "run_sharded_stages_ms_sum": {k: round(sum(s[k] for s, _ in single_res), 2) for k in STAGES},
                         "run_sharded_sweep_stages_ms": {k: round(sweep[0][0][k], 2) for k in STAGES},
                         "one_gpu_sweep_stages_ms": {k: round(one[0][0][k], 2) for k in STAGES},
                         "exchanged_keys_sweep": sweep[0][0]["exchanged_keys"]})
            print(f"[sweep {G} GPU] rep {rep}: ten run_sharded {sum(singles):.1f} ms, one run_sharded_sweep {ms_sweep:.1f} ms, one-GPU sweep {ms_one:.1f} ms", file=sys.stderr, flush=True)
        med = lambda k: sorted(x[k] for x in reps)[len(reps) // 2]   # noqa: E731
        out = {"gpus": gpus, "n_devices": G, "reads": base["reads"], "bam_bytes": int(bam.size), "rates": RATES, "repetitions": reps,
               "per_rate": [{"rate": r, **{k: int(s[k]) for k in COUNTERS}, "coo_sha256_16": coo_hash(a)} for r, (s, a) in zip(RATES, ref)],
               "median_ten_run_sharded_ms": med("ten_run_sharded_ms"), "median_run_sharded_sweep_ms": med("run_sharded_sweep_ms"), "median_one_gpu_sweep_ms": med("one_gpu_sweep_ms"),
               "agreement": "per rate: total, cb_valid, sampled, valid, nnz and a sha256 of (m_gene, m_cell, m_count) equal between run_sharded, run_sharded_sweep and the one-GPU sweep",
               "timing": "host wall clock around each whole call from a BAM image in host memory: context creation, H2D of the compressed bytes, all device work, results on the host",
               "build": _lib.build_info()}
        with open(os.path.join(args.out, "depth_sweep_%dgpu.json" % G), "w") as f:
            json.dump(out, f, indent=1)
        print(json.dumps({k: out[k] for k in ("gpus", "reads", "median_ten_run_sharded_ms", "median_run_sharded_sweep_ms", "median_one_gpu_sweep_ms")}))
    finally:
        shutil.rmtree(tmp, ignore_errors=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--reads", type=int, default=None, help="distinct reads (default 64 M; with --gpus, 64 M per GPU)")
    ap.add_argument("--cli-reads", type=int, default=16_000_000)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--gpus", type=int, default=0, help="run the multi-GPU leg over devices 0..G-1 instead")
    args = ap.parse_args()
    os.makedirs(args.out, exist_ok=True)
    if args.gpus:
        return main_multi(args)
    args.reads = args.reads or 64_000_000
    import torch
    import bench
    from fastf_b200 import _lib, build, bam2db_host as B
    gpu = gpu_identity()
    lib = _lib.load()
    ctx = _lib.Context(0)
    base = bench.make_base(args.reads, os.cpu_count() or 1)
    tmp = tempfile.mkdtemp(prefix="fastf_sweep_", dir="/dev/shm" if os.path.isdir("/dev/shm") else None)
    try:
        paths, _ = bench.write_inputs(base, tmp, write_bam=False)
        inputs = B.Bam2dbInputs(lib, paths["barcodes"], paths["features"], bench.RATE_CELL, bench.SEED)
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
            e0.record(stream)
            out = run()
            e1.record(stream)
            e1.synchronize()
            return e0.elapsed_time(e1), out

        def single(rate):
            with B.Bam2dbJob(ctx, inputs, rate, bench.SEED, want_rows=False) as job:
                job.feed_device(dptr.value, bam.size, in_off, in_len, isz)
                return job.finish()

        def sweep():
            with B.Bam2dbJob(ctx, inputs, 0.0, bench.SEED, want_rows=False) as job:
                job.feed_device(dptr.value, bam.size, in_off, in_len, isz)
                return job.finish_sweep(RATES)

        # warm-up: every shape once
        single(RATES[0])
        sweep()
        reps = []
        for rep in range(args.reps):
            singles, single_stats = [], []
            for r in RATES:
                ms, (st, arr) = timed(lambda: single(r))
                singles.append(ms)
                single_stats.append((st, arr))
            ms_sweep, res = timed(sweep)
            for r, (s1, a1), (s2, a2) in zip(RATES, single_stats, res):
                assert [s1[k] for k in COUNTERS] == [s2[k] for k in COUNTERS], ("counters differ", r, s1, s2)
                assert coo_hash(a1) == coo_hash(a2), ("COO differs", r)
            reps.append({"single_jobs_ms": [round(x, 2) for x in singles], "ten_single_jobs_ms": round(sum(singles), 2), "sweep_job_ms": round(ms_sweep, 2),
                         "single_stages_ms_sum": {k: round(sum(s[k] for s, _ in single_stats), 2) for k in STAGES},
                         "sweep_stages_ms": {k: round(res[0][0][k], 2) for k in STAGES}})
            print(f"[sweep] rep {rep}: ten single-rate jobs {sum(singles):.1f} ms, one sweep job {ms_sweep:.1f} ms", file=sys.stderr, flush=True)
        per_rate = [{"rate": r, **{k: int(s[k]) for k in COUNTERS}, "coo_sha256_16": coo_hash(a)} for r, (s, a) in zip(RATES, res)]
        lib.fastf_device_free(ctx.h, dptr)
        ten = sorted(x["ten_single_jobs_ms"] for x in reps)
        one = sorted(x["sweep_job_ms"] for x in reps)
        device = {"reads": base["reads"], "rates": RATES, "repetitions": reps, "per_rate": per_rate,
                  "median_ten_single_jobs_ms": ten[len(ten) // 2], "median_sweep_job_ms": one[len(one) // 2],
                  "speedup_median": round(ten[len(ten) // 2] / one[len(one) // 2], 2),
                  "agreement": "per rate: total, cb_valid, sampled, valid, nnz and a sha256 of (m_gene, m_cell, m_count) equal between the single-rate job and the sweep",
                  "timing": "CUDA events on fastf_compute_stream around each whole job (begin, device-resident feed, finish, results on the host)"}

        # ---- CLI: --depths once against ten -r runs ----
        cli = build.build_cli()
        cdir = os.path.join(tmp, "cli")
        os.makedirs(cdir)
        cpaths, _ = bench.write_inputs(base, cdir, prefix_reads=min(args.cli_reads, base["reads"]))
        common = ["-b", cpaths["bam"], "-f", cpaths["features"], "-a", cpaths["barcodes"], "-c", str(bench.RATE_CELL), "-s", str(bench.SEED)]
        os.makedirs(os.path.join(cdir, "sweep"))
        t = time.time()
        r = subprocess.run([cli, "bam2db"] + common + ["-d", "sweep.db", "-o", os.path.join(cdir, "sweep"), "--depths", ",".join(str(x) for x in RATES)], stdout=subprocess.PIPE, stderr=subprocess.PIPE,
                           text=True, cwd=cdir)
        t_sweep = time.time() - t
        assert r.returncode == 0, r.stderr[-2000:]
        t_single = 0.0
        total = None
        for x in RATES:
            o = os.path.join(cdir, "r%s" % x)
            os.makedirs(o)
            t = time.time()
            r = subprocess.run([cli, "bam2db"] + common + ["-d", os.path.join(o, "single.db"), "-o", o, "-r", str(x)], stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, cwd=cdir)
            t_single += time.time() - t
            assert r.returncode == 0, r.stderr[-2000:]
            for ln in r.stdout.splitlines():
                if "total fastQ reads:" in ln:
                    total = int(ln.rsplit(":", 1)[1])
            a = gzip.open(os.path.join(o, "matrix.mtx.gz"), "rb").read()
            b = gzip.open(os.path.join(cdir, "sweep", "depth_%s" % x, "matrix.mtx.gz"), "rb").read()
            assert a == b, ("matrix.mtx differs between --depths and -r", x)
        cli_leg = {"reads": total, "depths_run_seconds": round(t_sweep, 2), "ten_r_runs_seconds": round(t_single, 2), "speedup": round(t_single / t_sweep, 2),
                   "compared": "decompressed matrix.mtx.gz of every rate identical",
                   "what": "whole CLI processes, files on /dev/shm -> sqlite databases + gz files; includes CUDA context creation"}
        out = {"gpu": gpu, "device": device, "cli": cli_leg, "build": _lib.build_info()}
        with open(os.path.join(args.out, "depth_sweep.json"), "w") as f:
            json.dump(out, f, indent=1)
        print(json.dumps({"gpu": gpu, "median_ten_single_jobs_ms": device["median_ten_single_jobs_ms"], "median_sweep_job_ms": device["median_sweep_job_ms"],
                          "cli": {k: cli_leg[k] for k in ("depths_run_seconds", "ten_r_runs_seconds")}}))
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
        ctx.close()


if __name__ == "__main__":
    main()
