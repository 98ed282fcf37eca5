#!/usr/bin/env python
"""bench.py -- `fastF bam2db` hot path on B200: reads/s through libfastf_gpu.so, roofline of the dominant kernel, the
reference's CPU path timed beside it.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--reads R] [--base-reads B] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Workload (BASELINE.json configs[2]): synthetic 10x-v3 BAM, 10k cells, 36k genes, `-c 1.0 -r 0.3 -s 926`, R reads per GPU
(default 500M).  The BAM is a zlib-6 BGZF image of B DISTINCT reads per rank (--base-reads; default 0 = 64 M / ranks, between
8 M and 64 M and at most R, whatever the host: 64 M reads = 9.6 GB compressed / 26 GB inflated; data seed
DATA_SEED + rank) whose record blocks are cycled T = ceil(R/B) times through the same job -- 5e8 distinct reads would take
~12 min of host zlib time per GPU.  The MT19937 draw ordinal keeps running across cycles, so every cycle keeps a different
30 % of its reads.  One step = one whole job (begin -> feed all cycles -> sample -> sort -> dedup/count -> COO on the host).
Before timing, the job's counters and COO of a bounded prefix (--check-reads) are compared with the oracle's.

  value : reads/s with the compressed bytes + block index already resident in HBM (fastf_bam2db_feed_device)
  e2e   : the same job fed from pinned HOST memory through fastf_bam2db_feed (H2D of every compressed byte inside the timed
          region, COO + counters copied back)
  roofline : the dominant kernel (bgzf_inflate): algorithmic bytes = compressed read + inflated written per launch, over the
          launch's CUDA-event duration, against MEASURED_PEAKS.json hbm_gbs
  cpu_baseline : oracle/_ref/fastF_ref (the unmodified reference compiled against the header shims) on a bounded prefix of the
          same BAM, 1 core (the reference path is single-threaded)
  --dump-outputs DIR : after the timed steps, what the last timed job returned to its caller as float64 .npy files (see
          dump_outputs), so that two builds can be compared output for output on the same input
"""
import argparse
import ctypes as C
import json
import os
import shutil
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

N_CELLS, N_GENES, RATE_CELL, RATE_DEPTH, SEED, DATA_SEED = 10000, 36000, 1.0, 0.3, 926, 11
# DRAM bytes of ONE launch of the inflate kernel on a full chunk of 2 x 148 x 224 BGZF blocks (ncu --set full, not a bench run)
INFLATE_TRAFFIC = (27.272e9 + 4.611e9, "profiles/r02c_ncu_inflate_crc_parse.txt (27.272 GB read + 4.611 GB written per launch over one 66304-block chunk, 4.31 GB inflated: "
                   "the LZ77 windows of 33152 concurrent streams (1 GB) do not fit the 126 MB L2, so most match sources are 32-byte sector reads from DRAM)")


def inflate_kernel_name():
    """Name of the instantiation the library launches, from its build record (streams / decoder lanes / service warps)."""
    from fastf_b200 import _lib
    info = _lib.build_info()
    return "fastf_bgzf_inflate_tps_kernel<%s,%s> (%s streams per SM)" % (info.get("lanes", "?"), info.get("svc", "?"), info.get("streams", "?"))


def log(*a):
    print(*a, file=sys.stderr, flush=True)


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region"""
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx = float(f[1])
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


def make_base(base_reads, threads, seed=None):
    """Synthetic base segment + barcode / feature lists.  Returns dict with the BGZF image (numpy u8) and text lists."""
    import synth_binding
    S = synth_binding.load()
    p = S.params(n_reads=base_reads, n_cells=N_CELLS, n_genes=N_GENES, seed=DATA_SEED if seed is None else seed)
    t = time.time()
    bam, st = S.bam(p, threads)
    log(f"[bench] generated {base_reads} reads: {st.compressed_bytes / 1e6:.0f} MB BGZF, {st.inflated_bytes / 1e6:.0f} MB inflated, {st.n_blocks} blocks in {time.time() - t:.1f}s on {threads} threads")
    return {"bam": bam, "barcodes": S.barcodes(p), "features": S.features(p), "reads": base_reads, "n_blocks": st.n_blocks,
            "inflated": st.inflated_bytes, "compressed": st.compressed_bytes}


def write_inputs(base, d, prefix_reads=None, write_bam=True):
    """files for the reference CLI; with prefix_reads a BAM holding only about that many reads (whole blocks)"""
    import gzip
    paths = {"bam": os.path.join(d, "synth.bam"), "barcodes": os.path.join(d, "barcodes.tsv.gz"), "features": os.path.join(d, "features.tsv.gz")}
    with gzip.open(paths["barcodes"], "wb", compresslevel=1) as f:
        f.write(base["barcodes"])
    with gzip.open(paths["features"], "wb", compresslevel=1) as f:
        f.write(base["features"])
    bam = base["bam"]
    reads = base["reads"]
    if prefix_reads and prefix_reads < base["reads"]:
        # cut at a block boundary in proportion; the EOF block (28 bytes) is re-appended
        from fastf_b200 import _lib
        lib = _lib.load()
        buf = np.frombuffer(bam, dtype=np.uint8)
        cap = base["n_blocks"] + 8
        in_off, in_len, isz = np.zeros(cap, np.uint64), np.zeros(cap, np.uint32), np.zeros(cap, np.uint32)
        used = C.c_size_t()
        nb = lib.fastf_bgzf_index_host(C.c_void_p(buf.ctypes.data), buf.size, in_off.ctypes.data_as(_lib.c_u64p), in_len.ctypes.data_as(_lib.c_u32p), isz.ctypes.data_as(_lib.c_u32p), cap, C.byref(used))
        k = max(2, int(nb * prefix_reads / base["reads"]))
        cut = int(in_off[k]) - 18
        bam = bam[:cut] + bam[-28:]
        reads = None   # counted by the reference itself
    if write_bam:
        with open(paths["bam"], "wb") as f:
            f.write(bam)
    return paths, reads


def run_reference_cli(paths, outdir, rate_cell, rate_depth, seed):
    """One run of the unmodified reference (oracle/_ref/fastF_ref).  Returns (seconds, total reads)."""
    ref = os.path.join(ROOT, "oracle", "_ref", "fastF_ref")
    kind = "reference"
    shutil.rmtree(outdir, ignore_errors=True)
    os.makedirs(outdir)
    db = os.path.join(outdir, "ref.db")
    if os.path.exists(ref):
        cmd = [ref, "bam2db", "-b", paths["bam"], "-f", paths["features"], "-a", paths["barcodes"], "-d", db, "-c", str(rate_cell), "-r", str(rate_depth), "-o", outdir, "-s", str(seed)]
    else:
        kind = "port"
        cmd = [os.path.join(ROOT, "oracle", "_build", "oracle_cli"), "bam2db", paths["bam"], paths["barcodes"], paths["features"], str(rate_cell), str(rate_depth), str(seed), outdir]
    t = time.time()
    r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True)
    dt = time.time() - t
    if r.returncode != 0:
        raise RuntimeError("reference run failed: " + r.stderr[-400:])
    total = None
    for ln in r.stdout.splitlines():
        if "total fastQ reads:" in ln:
            total = int(ln.rsplit(":", 1)[1])
        if ln.startswith("total="):
            total = int(ln.split()[0].split("=")[1])
    return dt, total, kind


def cli_leg(paths, ref_out, our_out, total, ref_seconds, ref_kind, device):
    """wall clock of `fastf_b200/_build/fastF bam2db` on the files the reference CLI just processed; every output compared"""
    import gzip
    from fastf_b200 import build
    from dbdigest import db_digest
    cli = build.build_cli()
    shutil.rmtree(our_out, ignore_errors=True)
    os.makedirs(our_out)
    cmd = [cli, "bam2db", "-b", paths["bam"], "-f", paths["features"], "-a", paths["barcodes"], "-d", os.path.join(our_out, "ours.db"), "-c", str(RATE_CELL), "-r", str(RATE_DEPTH), "-o", our_out, "-s", str(SEED)]
    t = time.time()
    r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, env=dict(os.environ, FASTF_DEVICE=str(device)))
    ours = time.time() - t
    if r.returncode != 0:
        return {"failed": r.stderr[-300:]}
    out = {"reads": total, "ours_seconds": round(ours, 3), "reference_seconds": round(ref_seconds, 3), "speedup": round(ref_seconds / ours, 1), "reference_kind": ref_kind,
           "what": "whole CLI run, file on /dev/shm -> sqlite database + matrix/barcodes/features gz files; includes CUDA context creation"}
    if ref_kind == "reference":
        same = all(gzip.open(os.path.join(our_out, f), "rb").read() == gzip.open(os.path.join(ref_out, f), "rb").read() for f in ("matrix.mtx.gz", "barcodes.tsv.gz", "features.tsv.gz"))
        t = time.time()
        a, b = db_digest(os.path.join(our_out, "ours.db")), db_digest(os.path.join(ref_out, "ref.db"))
        out["outputs_identical"] = bool(same and all(a[k] == b[k] for k in ("cell", "feature", "umi", "mtx")))
        out["compared"] = "decompressed matrix.mtx / barcodes / features bytes; sha256 of every row of tables cell, feature, umi, mtx"
        assert out["outputs_identical"], "the drop-in CLI and the reference CLI disagree"
    return out


def cpu_model():
    try:
        for ln in open("/proc/cpuinfo"):
            if ln.startswith("model name"):
                return ln.split(":", 1)[1].strip()
    except OSError:
        pass
    return "unknown"


DUMP_BYTES, DUMP_SEED = 64 << 20, 926


def dump_outputs(d, stats, coo):
    """Writes a bam2db job's result as float64 .npy files under d: counters.npy (total, cb_valid, sampled, valid, nnz) and the COO
    matrix m_gene.npy, m_cell.npy, m_count.npy.  A COO too large for DUMP_BYTES is cut to a fixed, seeded sample of its entries
    (sorted, so file order is kept); coo_index.npy holds the positions of the entries written, in every case."""
    os.makedirs(d, exist_ok=True)
    nnz = len(coo["m_gene"])
    cap = (DUMP_BYTES - (1 << 20)) // (4 * 8)   # four float64 arrays of cap entries, 1 MB left for the counters and the .npy headers
    idx = np.arange(nnz) if nnz <= cap else np.sort(np.random.default_rng(DUMP_SEED).choice(nnz, cap, replace=False))
    np.save(os.path.join(d, "counters.npy"), np.array([stats[k] for k in ("total", "cb_valid", "sampled", "valid", "nnz")], dtype=np.float64))
    np.save(os.path.join(d, "coo_index.npy"), idx.astype(np.float64))
    for k in ("m_gene", "m_cell", "m_count"):
        np.save(os.path.join(d, k + ".npy"), coo[k][idx].astype(np.float64))   # uint32 values: exact in float64
    log(f"[bench] --dump-outputs: {len(idx)} of {nnz} COO entries and the counters written to {d}")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--reads", type=int, default=500_000_000, help="reads per GPU per step")
    ap.add_argument("--base-reads", type=int, default=0, help="DISTINCT reads generated per GPU (a zlib-6 BGZF image, every rank its own data seed) and cycled ceil(reads/base) times per step; "
                    "0 = 64 M / ranks, between 8 M and 64 M")
    ap.add_argument("--check-reads", type=int, default=2_000_000, help="prefix of the data whose single-GPU result is compared with the CPU oracle before anything is timed (0 = skip)")
    ap.add_argument("--cli-reads", type=int, default=0, help="also time `fastF bam2db` (file in /dev/shm -> sqlite + gz files) against the reference CLI on a file of this many reads, outputs compared (0 = on the cpu_baseline sample)")
    ap.add_argument("--freq-reads", type=int, default=32_000_000, help="reads of the `freq` run reported as the `secondary` object of the line (0 = skip)")
    ap.add_argument("--ref-sample-reads", type=int, default=5_000_000)
    ap.add_argument("--e2e-steps", type=int, default=2)
    ap.add_argument("--lanes", type=int, default=0)
    ap.add_argument("--engine", default="sm", choices=["sm", "hw"], help="inflate engine of the main line: hand-written SM kernel (default) or the B200 hardware decompression engine")
    ap.add_argument("--no-hw-extra", action="store_true", help="skip the extra pass that reports the hardware decompression engine beside the main line")
    ap.add_argument("--chunk-mb", type=int, default=0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--config", type=int, default=2, choices=[2, 3], help="BASELINE.json configs[N] shape: 2 = 10k cells, -c 1.0 -r 0.3 (the headline); 3 = 50k cells, -c 0.2 -r 0.5 (the sharded 2 B-read case: --gpus 8 --reads 250000000)")
    ap.add_argument("--depth-sweep", action="store_true", help="after the main line: -r 0.1..1.0 over the same resident input (BASELINE.json configs[4])")
    ap.add_argument("--workload", default="bam2db", choices=["bam2db", "freq", "crb", "extract"], help="bam2db = BASELINE.json configs[2] (the headline); freq = configs[1] (use --reads 100000000)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write the counters and COO matrix of the last timed job to DIR/*.npy (float64; "
                    "a fixed, seeded sample of the COO when it exceeds 64 MB)")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl != "ours" or args.workload != "bam2db"):
        ap.error("--dump-outputs writes the results of the bam2db timed path (--impl ours --workload bam2db)")
    global N_CELLS, RATE_CELL, RATE_DEPTH
    if args.config == 3:
        N_CELLS, RATE_CELL, RATE_DEPTH = 50000, 0.2, 0.5
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    threads = os.cpu_count() or 1
    if args.base_reads <= 0:
        # zlib-6 generation runs at ~44 k reads/s per host thread, so 64 M reads over all ranks take ~90 s on 16 host cores.  The
        # size does not depend on the host's core count: the same arguments give the same input everywhere.
        args.base_reads = int(min(64_000_000, max(8_000_000, 64_000_000 // max(1, world)), max(args.reads, 1_000_000)))
    workload = f"bam2db synthetic 10x-v3 BAM: {args.reads} reads/GPU, {N_CELLS} cells, {N_GENES} genes, -c {RATE_CELL} -r {RATE_DEPTH} -s {SEED} (BASELINE.json configs[{args.config}])"

    # ------------------------------------------------------------------ reference arm: the reference's own CPU path
    if args.impl == "reference" and args.workload == "freq":
        if rank != 0:
            return 0
        import synth_binding
        S = synth_binding.load()
        n = min(args.ref_sample_reads, 3_000_000)
        fq, _ = S.fastq(S.params(n_reads=n, n_cells=20000, seed=DATA_SEED, p_umi_n=0.001), threads)
        tmp = tempfile.mkdtemp(prefix="fastf_ref_", dir="/dev/shm" if os.path.isdir("/dev/shm") else None)
        try:
            open(os.path.join(tmp, "R1.fastq.gz"), "wb").write(fq)
            os.makedirs(os.path.join(tmp, "o"))
            ref = os.path.join(ROOT, "oracle", "_ref", "fastF_ref")
            kind = "reference" if os.path.exists(ref) else "port"
            cmd = [ref, "freq", "-R", os.path.join(tmp, "R1.fastq.gz"), "-o", os.path.join(tmp, "o"), "-l", "16", "-u", "12"] if kind == "reference" else \
                  [os.path.join(ROOT, "oracle", "_build", "oracle_cli"), "freq", os.path.join(tmp, "R1.fastq.gz"), "16", "12", os.path.join(tmp, "o", "whitelist.txt")]
            times = []
            for i in range(args.warmup + args.steps):
                t0 = time.time()
                subprocess.run(cmd, check=True, stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
                if i >= args.warmup:
                    times.append(time.time() - t0)
        finally:
            shutil.rmtree(tmp, ignore_errors=True)
        ms = 1e3 * sum(times) / len(times)
        v = n / (ms / 1e3)
        sample = f"{n}-read synthetic R1 FASTQ per step (whole run of the reference CLI `freq -l 16 -u 12`; wall clock)"
        print(json.dumps({"impl": "reference", "metric": "freq reads/sec (device-timed)", "value": v, "unit": "reads/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms,
                          "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic", "config": {"workload": "freq (BASELINE.json configs[1] shape)", "sample": sample},
                          "cpu_baseline": {"value": v, "unit": "reads/s", "cores": 1, "kind": kind, "sample": sample, "cpu": cpu_model(), "host_cores": threads},
                          "e2e": {"value": v, "unit": "reads/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))
        return 0
    if args.impl == "reference" and args.workload in ("crb", "extract"):
        if rank != 0:
            return 0
        base = make_base(min(args.base_reads, args.ref_sample_reads), threads)
        tmp = tempfile.mkdtemp(prefix="fastf_ref_", dir="/dev/shm" if os.path.isdir("/dev/shm") else None)
        try:
            paths, _ = write_inputs(base, tmp)
            times = [tags_reference_cli(args.workload, paths["bam"], tmp)[0] for _ in range(args.warmup + args.steps)][args.warmup:]
            kind = tags_reference_cli(args.workload, paths["bam"], tmp, dry=True)[1]
        finally:
            shutil.rmtree(tmp, ignore_errors=True)
        ms = 1e3 * sum(times) / len(times)
        v = base["reads"] / (ms / 1e3)
        sample = f"{base['reads']}-read synthetic BAM per step (whole run of the reference CLI `{TAGS_CMD[args.workload]}`; wall clock)"
        print(json.dumps({"impl": "reference", "metric": args.workload + " reads/sec (device-timed)", "value": v, "unit": "reads/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms,
                          "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic", "config": {"workload": args.workload + " (SURVEY 8f)", "sample": sample},
                          "cpu_baseline": {"value": v, "unit": "reads/s", "cores": 1, "kind": kind, "sample": sample, "cpu": cpu_model(), "host_cores": threads},
                          "e2e": {"value": v, "unit": "reads/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))
        return 0
    if args.impl == "reference":
        if rank != 0:
            return 0
        from fastf_b200 import build
        build.build_synth()
        base = make_base(min(args.base_reads, args.ref_sample_reads), threads)
        tmp = tempfile.mkdtemp(prefix="fastf_ref_", dir="/dev/shm" if os.path.isdir("/dev/shm") else None)
        try:
            paths, _ = write_inputs(base, tmp)
            times, total, kind = [], None, "reference"
            for i in range(args.warmup + args.steps):
                dt, total, kind = run_reference_cli(paths, os.path.join(tmp, "out"), RATE_CELL, RATE_DEPTH, SEED)
                if i >= args.warmup:
                    times.append(dt)
                log(f"[bench] reference step {i}: {dt:.2f}s for {total} reads")
        finally:
            shutil.rmtree(tmp, ignore_errors=True)
        ms = 1e3 * sum(times) / len(times)
        v = total / (ms / 1e3)
        sample = f"{total}-read prefix of the same synthetic BAM per step (whole run of the unmodified reference CLI: inflate, parse, sample, sqlite insert + GROUP BY, gz output; wall clock)"
        print(json.dumps({"impl": "reference", "metric": "bam2db reads/sec (device-timed)", "value": v, "unit": "reads/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms,
                          "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
                          "config": {"workload": workload, "sample": sample},
                          "cpu_baseline": {"value": v, "unit": "reads/s", "cores": 1, "kind": kind, "sample": sample, "cpu": cpu_model(), "host_cores": threads},
                          "e2e": {"value": v, "unit": "reads/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))
        return 0

    if args.workload == "freq":
        if args.reads == 500_000_000:
            args.reads = 100_000_000
        return bench_freq(args)
    if args.workload in ("crb", "extract"):
        if args.reads == 500_000_000:
            args.reads = 32_000_000
        return bench_tags(args)

    # ------------------------------------------------------------------ our arm
    import torch
    from fastf_b200 import _lib
    from fastf_b200 import bam2db_host as B
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the hot path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dist = None
    saved_stdout = None
    if world > 1:
        import torch.distributed as dist
        # NCCL prints its version banner on stdout when NCCL_DEBUG asks for it: keep stdout for the one JSON line
        sys.stdout.flush()
        saved_stdout = os.dup(1)
        os.dup2(2, 1)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    ctx = _lib.Context(local_rank)
    lib = ctx.lib
    # every rank generates its OWN distinct reads (data seed + rank) on its share of the host cores: nothing is replayed across GPUs
    base = make_base(args.base_reads, max(1, threads // max(1, world)), seed=DATA_SEED + rank)
    if dist:
        dist.barrier()
    tmp = tempfile.mkdtemp(prefix=f"fastf_bench_{rank}_", dir="/dev/shm" if os.path.isdir("/dev/shm") else None)
    try:
        paths, _ = write_inputs(base, tmp, write_bam=False)   # the lists only: the image stays in memory
        inputs = B.Bam2dbInputs(lib, paths["barcodes"], paths["features"], RATE_CELL, SEED)
        bam = np.frombuffer(base["bam"], dtype=np.uint8)
        nbytes = bam.size
        # block index of the image (host, once)
        cap = base["n_blocks"] + 8
        in_off, in_len, isz = np.zeros(cap, np.uint64), np.zeros(cap, np.uint32), np.zeros(cap, np.uint32)
        used = C.c_size_t()
        nb = lib.fastf_bgzf_index_host(C.c_void_p(bam.ctypes.data), nbytes, in_off.ctypes.data_as(_lib.c_u64p), in_len.ctypes.data_as(_lib.c_u32p), isz.ctypes.data_as(_lib.c_u32p), cap, C.byref(used))
        assert nb == base["n_blocks"] and used.value == nbytes, (nb, used.value, nbytes)
        in_off, in_len, isz = in_off[:nb].copy(), in_len[:nb].copy(), isz[:nb].copy()
        # block 0 = BAM header (own block), block nb-1 = EOF; record blocks are 1..nb-2
        rec_lo, rec_hi = 1, nb - 1
        tiles = max(1, -(-args.reads // base["reads"]))
        reads_per_step = tiles * base["reads"]
        comp_rec_bytes = int(in_off[rec_hi] - 18 - (in_off[rec_lo] - 18))
        infl_rec_bytes = int(isz[rec_lo:rec_hi].sum())
        # device copy of the image (value leg) and pinned host copy (e2e leg)
        dptr = C.c_void_p()
        ctx.check(lib.fastf_device_alloc(ctx.h, nbytes + 64, C.byref(dptr)), "device_alloc")
        ctx.check(lib.fastf_memcpy_h2d(ctx.h, dptr, C.c_void_p(bam.ctypes.data), nbytes), "h2d")
        hptr = C.c_void_p()
        ctx.check(lib.fastf_host_alloc(ctx.h, nbytes, C.byref(hptr)), "host_alloc")
        C.memmove(hptr, bam.ctypes.data, nbytes)
        hdr_end = int(in_off[rec_lo]) - 18          # first byte of the first record block
        eof_start = int(in_off[rec_hi]) - 18
        chunk = args.chunk_mb << 20

        HW = 0x100   # FASTF_INFLATE_HW_ENGINE
        engine = {"lanes": args.lanes | (HW if args.engine == "hw" else 0)}

        # ---- parity before speed: a prefix of this very data through the GPU path and through the CPU oracle (bit-exact), and the
        # counters of ONE tile, which every timed job must reproduce tiles-fold ----
        checks = {"oracle_prefix_reads": 0}
        if args.check_reads and rank == 0:
            import oracle_binding
            O = oracle_binding.load()
            dck = os.path.join(tmp, "check")
            os.makedirs(dck, exist_ok=True)
            pck, _ = write_inputs(base, dck, prefix_reads=min(args.check_reads, base["reads"]))
            t0 = time.time()
            want = O.bam2db(pck["bam"], pck["barcodes"], pck["features"], RATE_CELL, RATE_DEPTH, SEED)
            gst, gout = B.run_device(ctx, np.fromfile(pck["bam"], dtype=np.uint8), inputs, RATE_DEPTH, SEED, want_rows=False, inflate_lanes=engine["lanes"])
            for k in ("total", "cb_valid", "sampled", "valid", "nnz"):
                assert gst[k] == want[k], ("GPU result differs from the oracle on the check prefix", k, gst[k], want[k])
            assert np.array_equal(gout["m_gene"], want["m_gene"]) and np.array_equal(gout["m_cell"], want["m_cell"]) and np.array_equal(gout["m_count"], want["m_count"]), "COO differs from the oracle"
            checks = {"oracle_prefix_reads": int(want["total"]), "oracle_prefix_nnz": int(want["nnz"]), "oracle_prefix_seconds": round(time.time() - t0, 1), "oracle_prefix": "counters + COO bit-exact"}
            log(f"[bench] check: {want['total']}-read prefix, GPU == oracle (nnz {want['nnz']}) in {time.time() - t0:.1f}s")
        with B.Bam2dbJob(ctx, inputs, RATE_DEPTH, SEED, want_rows=False, inflate_lanes=engine["lanes"], headerless=False) as job1:
            job1.feed_device(dptr.value, nbytes, in_off[0:rec_hi], in_len[0:rec_hi], isz[0:rec_hi])
            tile_stats, _ = job1.finish(copy=False)
        assert tile_stats["total"] == base["reads"], ("one tile does not hold the generated reads", tile_stats["total"], base["reads"])

        rate = {"depth": RATE_DEPTH}

        def check_job(st_):
            """what every timed job must satisfy (a silent miscount at chunk 40 of 80 would otherwise still print reads/s)"""
            if world > 1:
                return
            assert st_["total"] == tiles * base["reads"], ("total", st_["total"], tiles * base["reads"])
            assert st_["cb_valid"] == tiles * tile_stats["cb_valid"], ("cb_valid", st_["cb_valid"], tiles * tile_stats["cb_valid"])
            n_, p_ = float(st_["cb_valid"]), float(rate["depth"])   # the rate of THIS job (--depth-sweep varies it)
            assert abs(st_["sampled"] - n_ * p_) <= 6.0 * (n_ * p_ * (1 - p_)) ** 0.5 + 1, ("sampled is not a Binomial(cb_valid, rate) draw", st_["sampled"], n_ * p_)
            assert st_["valid"] <= st_["sampled"] and st_["nnz"] <= st_["valid"], ("valid / nnz", st_["valid"], st_["sampled"], st_["nnz"])
            if rate["depth"] >= RATE_DEPTH:   # tile_stats was taken at RATE_DEPTH
                assert tile_stats["nnz"] <= st_["nnz"], ("nnz below one tile's", st_["nnz"], tile_stats["nnz"])
            assert st_["status"] == 0, ("status", st_["status"])

        kept = []   # --dump-outputs: (stats, COO) of the last timed job

        def one_job(device_resident, want_copy=False, keep=False):
            with B.Bam2dbJob(ctx, inputs, rate["depth"], SEED, want_rows=False, inflate_lanes=engine["lanes"], chunk_inflated_bytes=chunk, headerless=(rank != 0)) as job:
                for t in range(tiles):
                    if device_resident:
                        lo = 0 if (t == 0 and rank == 0) else rec_lo
                        job.feed_device(dptr.value, nbytes, in_off[lo:rec_hi], in_len[lo:rec_hi], isz[lo:rec_hi])
                    else:
                        lo = 0 if (t == 0 and rank == 0) else hdr_end
                        job.feed(hptr.value + lo, eof_start - lo)
                if world > 1:
                    st_, out_ = multi_gpu_tail(job, dist, torch, ctx, rank, world, inputs)   # out_: rank 0's gathered COO (numpy)
                    if keep:
                        kept.append((st_, out_))
                    return st_, out_
                if not keep:
                    return job.finish(copy=want_copy)
                # the library's result arrays are held until after the timed region instead of being copied inside it
                res = _lib.Bam2dbResult()
                ctx.check(lib.fastf_bam2db_finish(job.job, C.byref(res)), "bam2db_finish")
                st_ = {f: getattr(res, f) for f, _ in _lib.Bam2dbResult._fields_ if not f.startswith("m_") and f != "row_keys"}
                kept.append((st_, res))
                return st_, None

        def timed(device_resident, steps, warmup, sampler=None, keep_last=False):
            for _ in range(warmup):
                one_job(device_resident)
            if dist:
                dist.barrier()
            torch.cuda.synchronize()
            ctx.check(lib.fastf_synchronize(ctx.h), "sync")
            l0 = ctx.launches
            if sampler:
                sampler.start()
            # CUDA events on the stream the library launches its kernels on (torch's current stream would see nothing)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            t0 = time.time()
            e0.record(lib_stream)
            stats_all = []
            for i in range(steps):
                st, _out = one_job(device_resident, keep=keep_last and i == steps - 1)
                stats_all.append(st)
            for st in stats_all:
                check_job(st)
            assert all(x["nnz"] == stats_all[0]["nnz"] and x["valid"] == stats_all[0]["valid"] for x in stats_all), "steps over the same input disagree"
            e1.record(lib_stream)
            ctx.check(lib.fastf_synchronize(ctx.h), "sync")
            torch.cuda.synchronize()
            if dist:
                dist.barrier()
            wall = time.time() - t0
            clocks = sampler.stop() if sampler else None
            return wall, stats_all, ctx.launches - l0, clocks, e0.elapsed_time(e1)

        lib_stream = torch.cuda.ExternalStream(lib.fastf_compute_stream(ctx.h), device=torch.device("cuda", local_rank))
        sampler = ClockSampler(local_rank) if rank == 0 else None
        wall, stats_all, launches, clocks, dev_ms_total = timed(True, args.steps, args.warmup, sampler, keep_last=bool(args.dump_outputs))
        if args.dump_outputs:
            kst, kout = kept.pop()
            if world == 1:
                res = kout
                kout = {k: np.ctypeslib.as_array(getattr(res, k), (res.nnz,)) if res.nnz else np.zeros(0, np.uint32) for k in ("m_gene", "m_cell", "m_count")}
                dump_outputs(args.dump_outputs, kst, kout)
                lib.fastf_bam2db_result_free(C.byref(res))
            elif rank == 0:
                dump_outputs(args.dump_outputs, kst, kout)
        ms_step = dev_ms_total / args.steps
        ms_step_wall = 1e3 * wall / args.steps
        ms_job_dev = float(np.mean([s["ms_device_total"] for s in stats_all]))   # library's own first-chunk -> last-kernel clock
        if dist:
            tt = torch.tensor([ms_step, ms_step_wall], dtype=torch.float64, device="cuda")
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            ms_step, ms_step_wall = float(tt[0]), float(tt[1])
        value = world * reads_per_step / (ms_step / 1e3)
        st = stats_all[-1]
        e2e = None
        if not args.no_e2e:
            ew, estats, _, _, _ = timed(False, args.e2e_steps, 1)
            e_ms = 1e3 * ew / args.e2e_steps
            if dist:
                tt = torch.tensor([e_ms], dtype=torch.float64, device="cuda")
                dist.all_reduce(tt, op=dist.ReduceOp.MAX)
                e_ms = float(tt[0])
            d2h = int(estats[-1].get("nnz") or 0) * 12 + 64
            e2e = {"value": world * reads_per_step / (e_ms / 1e3), "unit": "reads/s", "h2d_bytes_per_step": int(tiles * comp_rec_bytes + hdr_end), "d2h_bytes_per_step": d2h,
                   "ms_per_step": e_ms, "steps": args.e2e_steps, "timing": "host wall clock around begin..finish (pinned host BGZF bytes in, COO out)"}
        sweep = None
        if args.depth_sweep:
            # BASELINE.json configs[4]: -r 0.1 .. 1.0 at a fixed seed over the same resident input; per rate one warm-up and one timed job
            sweep = []
            for r10 in range(1, 11):
                rate["depth"] = r10 / 10.0
                _, sst, _, _, sdev = timed(True, 1, 1)
                sms = sdev
                if dist:
                    tt = torch.tensor([sms], dtype=torch.float64, device="cuda")
                    dist.all_reduce(tt, op=dist.ReduceOp.MAX)
                    sms = float(tt[0])
                q = sst[-1]
                row = {"rate_depth": rate["depth"], "reads_per_s": world * reads_per_step / (sms / 1e3), "ms_per_job": sms, "sampled": q.get("sampled"), "valid": q.get("valid"), "nnz": q.get("nnz")}
                if world == 1:
                    row.update({"ms_sample": round(q["ms_sample"], 3), "ms_sort": round(q["ms_sort"], 3), "ms_count": round(q["ms_count"], 3),
                                "sample_dedup_keys_per_s": (q["valid"] / ((q["ms_sample"] + q["ms_sort"] + q["ms_count"]) * 1e-3)) if q["valid"] else None})
                else:
                    row["exchanged_keys"] = q.get("exchanged_keys")
                sweep.append(row)
            rate["depth"] = RATE_DEPTH
        hw_extra = None
        if args.engine == "sm" and not args.no_hw_extra:
            # the same job with BGZF inflate on the B200 hardware decompression engine instead of the SM kernel (reported beside the main line)
            engine["lanes"] = args.lanes | HW
            try:
                hw_wall, hw_stats, _, _, hw_dev_ms = timed(True, max(1, min(args.steps, 2)), 1)
                hw_ms = hw_dev_ms / max(1, min(args.steps, 2))
                hw_e2e_ms = None
                if not args.no_e2e:
                    hw_ew, _, _, _, _ = timed(False, 1, 1)
                    hw_e2e_ms = 1e3 * hw_ew
                if dist:
                    tt = torch.tensor([hw_ms, hw_e2e_ms or 0.0], dtype=torch.float64, device="cuda")
                    dist.all_reduce(tt, op=dist.ReduceOp.MAX)
                    hw_ms, hw_e2e_ms = float(tt[0]), (float(tt[1]) if hw_e2e_ms is not None else None)
                hs = hw_stats[-1]
                hw_extra = {"what": "same job, BGZF inflate by the hardware decompression engine (cuMemBatchDecompressAsync, DEFLATE) instead of fastf_bgzf_inflate_kernel; not the headline",
                            "value": world * reads_per_step / (hw_ms / 1e3), "unit": "reads/s", "ms_per_step": hw_ms,
                            "e2e_value": (world * reads_per_step / (hw_e2e_ms / 1e3)) if hw_e2e_ms else None,
                            "inflate_ms": hs.get("ms_inflate"), "inflate_alg_GBps": ((hs["compressed_bytes"] + hs["inflated_bytes"]) / (hs["ms_inflate"] * 1e-3) / 1e9) if hs.get("ms_inflate") else None,
                            "parse_ms": hs.get("ms_parse")}
            except Exception as e:   # engine absent on this GPU / driver: say so, the main line stands
                hw_extra = {"unavailable": str(e)[:200]}
            engine["lanes"] = args.lanes
        if rank != 0:
            return 0
        peak, peak_src = measured_peak()
        n_chunks = max(1, st["n_chunks"])
        infl_ms_launch = st["ms_inflate"] / n_chunks
        alg_bytes_launch = (st["compressed_bytes"] + st["inflated_bytes"]) / n_chunks
        achieved = alg_bytes_launch / (infl_ms_launch * 1e-3) / 1e9
        stages = {}
        for k, bytes_ in (("inflate", st["compressed_bytes"] + st["inflated_bytes"]), ("crc", st["inflated_bytes"]), ("parse", st["inflated_bytes"] + 8 * st["total"]), ("mt", st["cb_valid"] / 8.0 + 0),
                          ("sample", st["cb_valid"] * 8 * 2 + st["valid"] * 8), ("sort", st["valid"] * 16 * 7), ("count", st["valid"] * 8 + st["nnz"] * 12)):
            if world > 1 and k in ("sort", "count", "sample", "mt"):
                continue   # rank 0's local clocks only cover the streaming stages in the sharded job
            ms = st["ms_" + k]
            stages[k] = {"ms": round(ms, 3), "alg_GBps": round(bytes_ / (ms * 1e-3) / 1e9, 1) if ms > 0 else None}
        line = {"metric": "bam2db reads/sec (device-timed)", "value": value, "unit": "reads/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_step,
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
                "timing": "value: device-timed (CUDA events), compressed bytes resident in HBM and the BGZF block index (header walk) precomputed on the host outside the timed region; e2e: host wall clock from pinned host memory, header walk and every H2D / D2H copy inside",
                "config": {"workload": workload, "tiling": f"{base['reads']} DISTINCT reads per GPU (zlib-6 BGZF image, {base['compressed'] / 1e6:.0f} MB compressed, {base['inflated'] / 1e6:.0f} MB inflated; data seed {DATA_SEED}+rank) cycled {tiles}x per step "
                                     f"(5e8 distinct reads take ~12 min of host zlib time per GPU; the MT19937 draw ordinal keeps running, so every cycle keeps a different {RATE_DEPTH:.0%})",
                           "checks": dict(checks, per_job="total == tiles x reads, cb_valid == tiles x one-tile cb_valid, sampled within 6 sigma of Binomial(cb_valid, rate), status 0, steps agree"),
                           "l2": "inputs larger than L2 (compressed segment >> 126 MB); no explicit flush", "timing": "CUDA events on the library's launching stream around the K timed jobs, barrier + synchronize on both sides; max over ranks",
                           "ms_per_step_wall": ms_step_wall, "ms_per_job_library_clock": ms_job_dev, "counters": {k: st.get(k) for k in ("total", "cb_valid", "sampled", "valid", "nnz", "n_blocks", "n_chunks", "exchanged_keys")},
                           "parallelism": ("single GPU" if world == 1 else f"{world} ranks: contiguous BGZF block shards, all-gather of counts, NCCL all-to-all of locally deduplicated keys by cell hash, gather of COO")},
                "roofline": {"bound": "hbm", "kernel": "hardware decompression engine" if args.engine == "hw" else (inflate_kernel_name() if args.lanes == 0 else "inflate (--lanes %d)" % args.lanes),
                             "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                             # dram__bytes_read.sum + dram__bytes_write.sum of ONE launch of this kernel on a full chunk (ncu --set full)
                             "traffic": INFLATE_TRAFFIC[0] if (args.engine == "sm" and args.lanes == 0 and chunk == 0) else None, "traffic_source": INFLATE_TRAFFIC[1],
                             "peak_source": peak_src, "algorithmic_bytes_per_launch": alg_bytes_launch, "ms_per_launch": infl_ms_launch},
                "stages": stages, "gpu_launches": launches, "clocks": clocks, "e2e": e2e, "inflate_engine": args.engine, "hw_decompress_engine": hw_extra}
        if sweep is not None:
            line["depth_sweep"] = sweep
        if world > 1:
            assert st["total"] == world * tiles * base["reads"], ("gathered total", st["total"], world * tiles * base["reads"])
        if not args.no_cpu_baseline:
            d2 = os.path.join(tmp, "refin")
            os.makedirs(d2, exist_ok=True)
            p2, _ = write_inputs(base, d2, prefix_reads=args.cli_reads or args.ref_sample_reads)
            dt, total, kind = run_reference_cli(p2, os.path.join(tmp, "refout"), RATE_CELL, RATE_DEPTH, SEED)
            line["cpu_baseline"] = {"value": total / dt, "unit": "reads/s", "cores": 1, "kind": kind, "cpu": cpu_model(), "host_cores": threads,
                                    "sample": f"one run of the unmodified reference CLI on a {total}-read prefix of the same synthetic BAM ({dt:.1f}s wall; inflate via zlib shim, sqlite on /dev/shm)"}
            # the drop-in CLI on the very same files: the number a user of `fastF bam2db` sees (file -> sqlite database + gz files), outputs compared
            line["cli"] = cli_leg(p2, os.path.join(tmp, "refout"), os.path.join(tmp, "ourout"), total, dt, kind, local_rank)
        if args.freq_reads and world == 1:
            # BASELINE.json configs[1] rides in the same driver-parsed line
            fa = argparse.Namespace(**vars(args))
            fa.reads, fa.base_reads, fa.steps, fa.warmup, fa.e2e_steps = args.freq_reads, args.freq_reads, max(1, min(args.steps, 3)), 1, 1
            lib.fastf_device_free(ctx.h, dptr)
            lib.fastf_host_free(ctx.h, hptr)
            ctx.close()
            try:
                line["secondary"] = bench_freq(fa, emit=False)
            except Exception as e:   # the headline stands on its own
                line["secondary"] = {"workload": "freq", "failed": str(e)[:300]}
        if saved_stdout is not None:
            sys.stdout.flush()
            os.dup2(saved_stdout, 1)
        print(json.dumps(line))
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    return 0


def bench_freq(args, emit=True):
    """`fastF freq` (BASELINE.json configs[1]): R1 FASTQ, 20k true barcodes + 5 % single-base errors, -l 16 -u 12.  One step = one
    fastf_freq_gpu call over the whole BGZF image (value: image + index resident in HBM; e2e: pinned host bytes in, histogram out)."""
    import torch
    import synth_binding
    from fastf_b200 import _lib
    threads = os.cpu_count() or 1
    ctx = _lib.Context(0)
    lib = ctx.lib
    S = synth_binding.load()
    base_reads = min(args.base_reads, args.reads)
    p = S.params(n_reads=base_reads, n_cells=20000, seed=DATA_SEED, p_umi_n=0.001)
    t = time.time()
    fq, st = S.fastq(p, threads)
    log(f"[bench] generated {base_reads} FASTQ reads: {st.compressed_bytes / 1e6:.0f} MB BGZF, {st.inflated_bytes / 1e6:.0f} MB text in {time.time() - t:.1f}s")
    tiles = max(1, -(-args.reads // base_reads))
    body = fq[:-28]   # without the EOF block
    img = np.frombuffer(body * tiles + fq[-28:], dtype=np.uint8)
    n_reads = tiles * base_reads
    cap = int(st.n_blocks) * tiles + 8
    io, il, isz = np.zeros(cap, np.uint64), np.zeros(cap, np.uint32), np.zeros(cap, np.uint32)
    used = C.c_size_t()
    nb = lib.fastf_bgzf_index_host(C.c_void_p(img.ctypes.data), img.size, io.ctypes.data_as(_lib.c_u64p), il.ctypes.data_as(_lib.c_u32p), isz.ctypes.data_as(_lib.c_u32p), cap, C.byref(used))
    assert nb > 0 and used.value == img.size
    dptr, hptr = C.c_void_p(), C.c_void_p()
    ctx.check(lib.fastf_device_alloc(ctx.h, img.size + 64, C.byref(dptr)), "device_alloc")
    ctx.check(lib.fastf_memcpy_h2d(ctx.h, dptr, C.c_void_p(img.ctypes.data), img.size), "h2d")
    ctx.check(lib.fastf_host_alloc(ctx.h, img.size, C.byref(hptr)), "host_alloc")
    C.memmove(hptr, img.ctypes.data, img.size)
    klen = 28
    lib_stream = torch.cuda.ExternalStream(lib.fastf_compute_stream(ctx.h), device=torch.device("cuda", 0))

    def one(device_resident):
        res = _lib.FreqResult()
        if device_resident:
            ctx.check(lib.fastf_freq_gpu_device(ctx.h, dptr, img.size, io.ctypes.data_as(_lib.c_u64p), il.ctypes.data_as(_lib.c_u32p), isz.ctypes.data_as(_lib.c_u32p), nb, klen, args.lanes, C.byref(res)), "freq_gpu_device")
        else:
            ctx.check(lib.fastf_freq_gpu(ctx.h, hptr, img.size, klen, args.lanes, C.byref(res)), "freq_gpu")
        st_ = {f: getattr(res, f) for f, t_ in _lib.FreqResult._fields_ if t_ in (C.c_uint64, C.c_uint32, C.c_float, C.c_uint8)}
        lib.fastf_freq_result_free(C.byref(res))
        return st_

    def timed(device_resident, steps, warmup, sampler=None):
        for _ in range(warmup):
            one(device_resident)
        torch.cuda.synchronize()
        l0 = ctx.launches
        if sampler:
            sampler.start()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.time()
        e0.record(lib_stream)
        sts = [one(device_resident) for _ in range(steps)]
        e1.record(lib_stream)
        ctx.check(lib.fastf_synchronize(ctx.h), "sync")
        torch.cuda.synchronize()
        wall = time.time() - t0
        return wall, sts, ctx.launches - l0, (sampler.stop() if sampler else None), e0.elapsed_time(e1)

    sampler = ClockSampler(0)
    wall, sts, launches, clocks, dev_ms = timed(True, args.steps, args.warmup, sampler)
    ms_step = dev_ms / args.steps
    stq = sts[-1]
    e2e = None
    if not args.no_e2e:
        ew, ests, _, _, _ = timed(False, args.e2e_steps, 1)
        e_ms = 1e3 * ew / args.e2e_steps
        e2e = {"value": n_reads / (e_ms / 1e3), "unit": "reads/s", "h2d_bytes_per_step": int(img.size), "d2h_bytes_per_step": int(ests[-1]["n_keys"] * 16 + ests[-1]["n_exceptions"] * 36),
               "ms_per_step": e_ms, "steps": args.e2e_steps, "timing": "host wall clock around fastf_freq_gpu (pinned host BGZF bytes in, (key, count, first) + exceptions out)"}
    peak, peak_src = measured_peak()
    alg = stq["compressed_bytes"] + stq["inflated_bytes"]
    ach = alg / (stq["ms_inflate"] * 1e-3) / 1e9
    line = {"metric": "freq reads/sec (device-timed)", "value": n_reads / (ms_step / 1e3), "unit": "reads/s", "n_gpus": 1, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_step,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": {"workload": f"freq on synthetic R1 FASTQ: {n_reads} reads, 16 bp barcode + 12 bp UMI, 20000 true cells + 5 % error variants, -l 16 -u 12 (BASELINE.json configs[1])",
                       "tiling": f"{base_reads}-read BGZF segment x {tiles}", "l2": "inputs larger than L2", "ms_per_step_wall": 1e3 * wall / args.steps,
                       "counters": {k: stq[k] for k in ("n_reads", "n_keys", "n_exceptions", "n_blocks")}},
            "roofline": {"bound": "hbm", "kernel": "fastf_bgzf_inflate_tps_kernel", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak, "traffic": None, "peak_source": peak_src,
                         "algorithmic_bytes_per_launch": alg, "ms_per_launch": stq["ms_inflate"]},
            "stages": {k: round(stq["ms_" + k], 3) for k in ("inflate", "keys", "sort", "rle")}, "gpu_launches": launches, "clocks": clocks, "e2e": e2e}
    if not args.no_cpu_baseline:
        tmp = tempfile.mkdtemp(prefix="fastf_freq_", dir="/dev/shm" if os.path.isdir("/dev/shm") else None)
        try:
            sub = S.params(n_reads=min(base_reads, 3_000_000), n_cells=20000, seed=DATA_SEED, p_umi_n=0.001)
            sfq, _ = S.fastq(sub, threads)
            open(os.path.join(tmp, "R1.fastq.gz"), "wb").write(sfq)
            os.makedirs(os.path.join(tmp, "o"))
            ref = os.path.join(ROOT, "oracle", "_ref", "fastF_ref")
            kind = "reference" if os.path.exists(ref) else "port"
            cmd = [ref, "freq", "-R", os.path.join(tmp, "R1.fastq.gz"), "-o", os.path.join(tmp, "o"), "-l", "16", "-u", "12"] if kind == "reference" else \
                  [os.path.join(ROOT, "oracle", "_build", "oracle_cli"), "freq", os.path.join(tmp, "R1.fastq.gz"), "16", "12", os.path.join(tmp, "o", "whitelist.txt")]
            t0 = time.time()
            subprocess.run(cmd, check=True, stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
            dt = time.time() - t0
            line["cpu_baseline"] = {"value": sub.n_reads / dt, "unit": "reads/s", "cores": 1, "kind": kind, "cpu": cpu_model(), "host_cores": threads,
                                    "sample": f"one run of the reference CLI `freq -l 16 -u 12` on {sub.n_reads} reads of the same shape ({dt:.1f}s wall)"}
        finally:
            shutil.rmtree(tmp, ignore_errors=True)
    ctx.close()
    if not emit:
        return line
    print(json.dumps(line))
    return 0


TAGS_CMD = {"crb": "crb -b BAM -o out.gz", "extract": "extract -b BAM -t GX -T 0"}


def tags_reference_cli(workload, bam, tmp, dry=False):
    """one run of the reference's crb / extract (oracle/_ref/fastF_ref, else the oracle port) on bam -> (seconds, kind)"""
    ref = os.path.join(ROOT, "oracle", "_ref", "fastF_ref")
    kind = "reference" if os.path.exists(ref) else "port"
    if dry:
        return 0.0, kind
    if kind == "reference":
        cmd = [ref, "crb", "-b", bam, "-o", os.path.join(tmp, "ref_crb.gz")] if workload == "crb" else [ref, "extract", "-b", bam, "-t", "GX", "-T", "0"]
    else:
        cli = os.path.join(ROOT, "oracle", "_build", "oracle_cli")
        cmd = [cli, "crb", bam, os.path.join(tmp, "ref_crb.txt")] if workload == "crb" else [cli, "extract", bam, "GX", "0", os.path.join(tmp, "ref_extract.csv")]
    t0 = time.time()
    subprocess.run(cmd, check=True, cwd=tmp, stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
    return time.time() - t0, kind


def bench_tags(args):
    """`fastF crb` / `fastF extract -t GX` (SURVEY 8f.2-3) on the synthetic 10x-v3 BAM: one step = one fastf_taghist_gpu call over the whole
    BGZF image in pinned host memory.  value = reads / sum of the device stage clocks (inflate, tag kernel, sort, RLE + verification;
    the H2D copy is outside); e2e = reads / wall clock of the call (H2D of the file, groups + value strings back)."""
    from fastf_b200 import _lib
    threads = os.cpu_count() or 1
    ctx = _lib.Context(0)
    lib = ctx.lib
    base = make_base(min(args.base_reads, args.reads), threads)
    bam = np.frombuffer(base["bam"], dtype=np.uint8)
    hptr = C.c_void_p()
    ctx.check(lib.fastf_host_alloc(ctx.h, bam.size, C.byref(hptr)), "host_alloc")
    C.memmove(hptr, bam.ctypes.data, bam.size)
    tag_a, tag_b = (b"CB", b"CR") if args.workload == "crb" else (b"GX", None)

    def one():
        res = _lib.TaghistResult()
        ctx.check(lib.fastf_taghist_gpu(ctx.h, hptr, bam.size, tag_a, 0, tag_b, args.lanes, C.byref(res)), "taghist")
        st_ = {f: getattr(res, f) for f, t_ in _lib.TaghistResult._fields_ if t_ in (C.c_uint64, C.c_uint32, C.c_float)}
        lib.fastf_taghist_result_free(C.byref(res))
        return st_

    for _ in range(max(args.warmup, 1)):
        one()
    sampler = ClockSampler(0)
    sampler.start()
    l0 = ctx.launches
    t0 = time.time()
    sts = [one() for _ in range(args.steps)]
    wall = time.time() - t0
    clocks = sampler.stop()
    launches = ctx.launches - l0
    st = sts[-1]
    dev_ms = sum(sum(x["ms_" + k] for k in ("inflate", "tags", "sort", "rle")) for x in sts) / args.steps
    n_reads = int(st["n_records"])
    peak, peak_src = measured_peak()
    alg = st["compressed_bytes"] + st["inflated_bytes"]
    ach = alg / (st["ms_inflate"] * 1e-3) / 1e9
    line = {"metric": args.workload + " reads/sec (device-timed)", "value": n_reads / (dev_ms / 1e3), "unit": "reads/s", "n_gpus": 1, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dev_ms,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": {"workload": f"{args.workload} ({TAGS_CMD[args.workload]}) on the synthetic 10x-v3 BAM: {n_reads} reads, {N_CELLS} cells, {N_GENES} genes (SURVEY 8f)",
                       "l2": "inputs larger than L2", "counters": {k: st[k] for k in ("n_records", "n_hits", "n_groups", "n_blocks", "hash_rounds")}},
            "roofline": {"bound": "hbm", "kernel": inflate_kernel_name(), "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak, "traffic": None, "peak_source": peak_src,
                         "algorithmic_bytes_per_launch": alg, "ms_per_launch": st["ms_inflate"]},
            "stages": {k: {"ms": round(st["ms_" + k], 3)} for k in ("inflate", "tags", "sort", "rle")}, "gpu_launches": launches, "clocks": clocks,
            "e2e": {"value": n_reads / (wall / args.steps), "unit": "reads/s", "h2d_bytes_per_step": int(bam.size), "d2h_bytes_per_step": int(st["n_groups"] * 40 + st["strings_bytes"]),
                    "ms_per_step": 1e3 * wall / args.steps, "steps": args.steps, "timing": "host wall clock around fastf_taghist_gpu (pinned host BAM bytes in, groups + value strings out)"}}
    line["stages"]["tags"]["alg_GBps"] = round(st["inflated_bytes"] / (st["ms_tags"] * 1e-3) / 1e9, 1) if st["ms_tags"] > 0 else None
    if not args.no_cpu_baseline:
        tmp = tempfile.mkdtemp(prefix="fastf_tags_", dir="/dev/shm" if os.path.isdir("/dev/shm") else None)
        try:
            sub = make_base(min(base["reads"], 2_000_000), threads) if base["reads"] > 2_000_000 else base
            paths, _ = write_inputs(sub, tmp)
            dt, kind = tags_reference_cli(args.workload, paths["bam"], tmp)
            line["cpu_baseline"] = {"value": sub["reads"] / dt, "unit": "reads/s", "cores": 1, "kind": kind, "cpu": cpu_model(), "host_cores": threads,
                                    "sample": f"one run of the reference CLI `{TAGS_CMD[args.workload]}` on {sub['reads']} reads of the same shape ({dt:.1f}s wall)"}
        finally:
            shutil.rmtree(tmp, ignore_errors=True)
    print(json.dumps(line))
    return 0


def multi_gpu_tail(job, dist, torch, ctx, rank, world, inputs):
    """counts all-gather -> sample at the global ordinal -> unique + partition by cell hash -> NCCL all-to-all -> local dedup/count -> gather"""
    from fastf_b200 import sharded
    res = sharded.sharded_tail(ctx, job, dist, torch, "cuda", rank, world, len(inputs.cells), want_rows=False)
    st = job.stats()           # this rank's stage clocks and byte counts
    if res is not None:
        st.update({k: v for k, v in res[0].items() if k in ("total", "cb_valid", "sampled", "valid", "nnz", "exchanged_keys")})
    return st, (res[1] if res is not None else None)


if __name__ == "__main__":
    sys.exit(main())
