"""CPU tests (SIMT-emulator build) that the library gives back every device allocation, pinned allocation and CUDA event it makes,
on the success paths and on the error paths.  A variant of the emulator library counts the live ones (tests/emu/capi_counted.cpp,
read through fastf_emu_live_counts).  Every case runs in a process of its own: it makes a context, runs, frees what it made and
destroys the context; then nothing may be left.  Where the context is the test's, it also checks after the job is freed and the
pools are trimmed: no event, no pinned allocation, and device allocations only for the MT19937 jump polynomials the context keeps
once a job has sampled."""
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden")

WORKER = r'''
import ctypes as C, os, sys, tempfile
import numpy as np
sys.path.insert(0, %(root)r)
from fastf_b200 import _lib, bam2db_host as B, freq_host, tags_host

GOLD = %(gold)r
lib = _lib.load()
lib.fastf_emu_live_counts.argtypes = [C.POINTER(C.c_long)] * 3
lib.fastf_emu_live_counts.restype = None


def live():
    v = [C.c_long() for _ in range(3)]
    lib.fastf_emu_live_counts(*v)
    return tuple(x.value for x in v)   # (device allocations, pinned allocations, events)


def golden(d, rate_cell=0.5, seed=926):
    g = os.path.join(GOLD, d)
    inputs = B.Bam2dbInputs(lib, os.path.join(g, "barcodes.tsv.gz"), os.path.join(g, "features.tsv.gz"), rate_cell, seed)
    return inputs, np.fromfile(os.path.join(g, "in.bam"), dtype=np.uint8).tobytes()


def refused(fn, needle):
    try:
        fn()
    except _lib.FastfError as e:
        assert needle in str(e), str(e)
        return
    raise AssertionError("not refused: expected " + needle)


def single(ctx):
    inputs, bam = golden("synth4k")
    B.run_device(ctx, bam, inputs, 0.5, 926)
    return 1


def sweep(ctx):
    inputs, bam = golden("synth4k")
    B.run_device_sweep(ctx, bam, inputs, [0.3, 1.0, 0.6], 926)
    return 1


def grid_union():
    g = os.path.join(GOLD, "synth4k")
    return B.Bam2dbInputs.grid(lib, os.path.join(g, "barcodes.tsv.gz"), os.path.join(g, "features.tsv.gz"), [0.5, 1.0], 926), golden("synth4k")[1]


def grid(ctx):
    union, bam = grid_union()
    B.run_device_grid(ctx, bam, union, [0.4, 1.0], 926)
    return 1


def freq(ctx):
    freq_host.cell_counts(os.path.join(GOLD, "freq", "synth.fastq.gz"), 16, 12, ctx=ctx)
    return 0


def crb(ctx):
    with tempfile.TemporaryDirectory() as t:
        tags_host.crb(ctx, os.path.join(GOLD, "tags", "tags.bam"), os.path.join(t, "crb.gz"))
    return 0


def unique_counts(ctx):
    keys = np.random.default_rng(5).integers(0, 1 << 20, 20000, dtype=np.uint64)
    u, c = B.unique_counts(ctx, keys, 20)
    assert int(c.sum()) == keys.size
    return 0


def inflate(ctx):
    data = np.fromfile(os.path.join(GOLD, "synth4k", "in.bam"), dtype=np.uint8)
    out, n = C.c_void_p(), C.c_size_t()
    ctx.check(lib.fastf_inflate_host(ctx.h, C.c_void_p(data.ctypes.data), data.size, 0, C.byref(out), C.byref(n), None), "inflate_host")
    assert n.value > data.size
    lib.fastf_free(out)
    return 0


def sort(ctx):
    rng = np.random.default_rng(6)
    keys = rng.integers(0, 1 << 40, 30000, dtype=np.uint64)
    vals = np.arange(keys.size, dtype=np.uint32)
    want = np.sort(keys)
    ctx.check(lib.fastf_sort_u64_host(ctx.h, keys.ctypes.data_as(_lib.c_u64p), vals.ctypes.data_as(_lib.c_u32p), keys.size, 40), "sort_u64_host")
    assert np.array_equal(keys, want)
    return 0


def umi_too_long(ctx):
    inputs, bam = golden("synth4k")
    with B.Bam2dbJob(ctx, inputs, 0.5, 926, umi_max_bytes=1) as job:
        B._feed_all(job, bam, 0)
        refused(job.counts, "umi-too-long")
    return 0


def not_bgzf(ctx):
    inputs, _ = golden("synth4k")
    junk = np.frombuffer(b"this is not a BGZF stream " * 40, dtype=np.uint8)
    with B.Bam2dbJob(ctx, inputs, 0.5, 926) as job:
        refused(lambda: job.feed(junk.ctypes.data, junk.size), "not a BGZF")
    return 0


def grid_refusal(ctx):
    union, bam = grid_union()
    rates = B.grid_cell_rates(union)
    ci, n, d0 = rates[1]
    ci = ci.copy()
    held = np.nonzero(ci)[0]
    ci[held[1]] = ci[held[0]]   # one cell index twice within one rate
    with B.Bam2dbJob(ctx, union, 0.0, 926, grid=True) as job:
        B._feed_all(job, bam, 0)
        refused(lambda: job.finish_grid([rates[0], (ci, n, d0)], [0.5]), "twice")
    return 0


def begin_refusal(ctx):
    inputs, _ = golden("synth4k")
    refused(lambda: B.Bam2dbJob(ctx, inputs, 0.5, 926, umi_max_bytes=5), "umi_max_bytes must be 1..4")
    return 0


def sharded():
    inputs, bam = golden("synth4k")
    B.run_sharded_sweep(lib, bam, inputs, [0.3, 1.0], 926, 2)


name = sys.argv[1]
if name == "sharded":
    sharded()
else:
    ctx = _lib.Context(0)
    polys = globals()[name](ctx)
    lib.fastf_ctx_trim(ctx.h)
    assert live() == (polys, 0, 0), ("after job_free + ctx_trim", live())
    ctx.close()
assert live() == (0, 0, 0), ("after ctx_destroy", live())
print("ok", name)
''' % {"root": ROOT, "gold": GOLD}

CASES = ["single", "sweep", "grid", "freq", "crb", "unique_counts", "inflate", "sort", "sharded", "umi_too_long", "umi_too_long_feed_timing", "not_bgzf",
         "grid_refusal", "begin_refusal"]


@pytest.fixture(scope="module")
def emu_lib(tmp_path_factory):
    """the emulator library with counted allocations and events (tests/emu/capi_counted.cpp in place of capi.cu)"""
    from fastf_b200 import build
    out = str(tmp_path_factory.mktemp("emu_counted") / "libfastf_emu_counted.so")
    subprocess.run(["g++", "-O2", "-std=c++17", "-DFASTF_EMU", '-DFASTF_SRC_HASH="%s"' % build.source_hash(), "-I" + os.path.join(ROOT, "tests", "emu"), "-x", "c++", "-fPIC",
                    "-shared", "-o", out, os.path.join(ROOT, "tests", "emu", "capi_counted.cpp"), os.path.join(ROOT, "fastf_b200", "csrc", "sharded.cu"), "-lz", "-lpthread"],
                   check=True)
    return out


@pytest.mark.parametrize("case", CASES)
def test_emu_nothing_left_behind(emu_lib, case):
    env = dict(os.environ, FASTF_GPU_LIB=emu_lib)
    env.pop("FASTF_FEED_TIMING", None)
    if case == "umi_too_long_feed_timing":
        case, env["FASTF_FEED_TIMING"] = "umi_too_long", "1"
    if case == "sharded":
        env["FASTF_EMU_DEVICES"] = "2"
    r = subprocess.run([sys.executable, "-c", WORKER, case], env=env, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=1500)
    assert r.returncode == 0 and ("ok " + case) in r.stdout, r.stdout[-3000:]
