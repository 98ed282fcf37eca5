"""The depth sweep over several GPUs of one node (fastf_bam2db_run_sharded_sweep, bam2db_host.run_sharded_sweep,
fastf_b200.bam2db_sweep(gpus=N)): the result of one single-job sweep over the whole file, whatever the number of devices.  On the CPU
through the SIMT-emulator build with emulated devices (tests/sharded_sweep_worker.py in a subprocess); on B200s through the device copy
(one GPU) and the NCCL all-to-all (two or more)."""
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
WORKER = os.path.join(ROOT, "tests", "sharded_sweep_worker.py")
KEYS = ("total", "cb_valid", "sampled", "valid", "nnz")


def _emu(args, devices):
    from fastf_b200 import build
    env = dict(os.environ, FASTF_GPU_LIB=build.build_emu(), FASTF_EMU_DEVICES=str(devices), FASTF_MT_JUMP_MIN="0")
    r = subprocess.run([sys.executable, WORKER] + args, env=env, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=1500)
    assert r.returncode == 0 and "ok " in r.stdout, r.stdout[-3000:]


@pytest.mark.parametrize("g,n_reads,seed", [(2, 3000, 31), (3, 4000, 926), (5, 2500, 4)])
def test_emu_sharded_sweep_equals_single_job(g, n_reads, seed):
    """unsorted rates with NaN, -1, 0, 1, inf and two pairs of equal thresholds: every rate's counters and COO, the rows and their rate
    indices equal the single-job sweep at G = 1 and G; three rates also equal run_sharded and the oracle; keys with far-apart copies
    of different rate indices exist"""
    _emu(["driver", str(g), str(n_reads), str(seed)], g)


def test_emu_sharded_sweep_streamed_chunks_and_empty_shards():
    _emu(["chunks"], 5)


@pytest.mark.parametrize("case,g", [("synth4k-c0.5-r0.5-s926", 3), ("synth4k-c1.0-r0.3-s926", 3), ("edge-c0.8-r0.6-s3", 3)])
def test_emu_sharded_sweep_golden_python(case, g, tmp_path):
    """a golden case as one rate of an unsorted sweep through bam2db_sweep(gpus=g): that rate equals the recorded files and table
    digests (with -u for synth4k), every other rate the one-GPU sweep byte for byte"""
    _emu(["golden", case, str(g), str(tmp_path)], g)


def test_emu_sharded_sweep_refusals(tmp_path):
    """a corrupted shard, 0 or 33 rates, a threshold above 2^32, records that straddle blocks: each fails with a message"""
    _emu(["refusals", str(tmp_path)], 3)


# ------------------------------------------------------------------------------------------------------------------------------
# B200
# ------------------------------------------------------------------------------------------------------------------------------
RATES_4M = [0.5, 0.1, 1.0, 0.3, 0.8, 0.2, 0.9, 0.4, 0.7, 0.6, float("nan"), -1.0, 0.0, float("inf"), 1e-12, 2e-12]


@pytest.fixture(scope="module")
def bam_4m(tmp_path_factory, synth):
    d = str(tmp_path_factory.mktemp("shsweep4m"))
    paths, _ = synth.write_bam_set(d, n_reads=4_000_000, n_cells=3000, n_genes=20000, seed=13, p_umi_n=0.01, n_molecules=1_000_000)
    return paths


def _driver_vs_finish_sweep(ctx, paths, g):
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import sharded_sweep_worker as W
    from fastf_b200 import bam2db_host as B
    inputs = B.Bam2dbInputs(ctx.lib, paths["barcodes"], paths["features"], 0.5, 926)
    bam = np.fromfile(paths["bam"], dtype=np.uint8)
    one = W.single_job(ctx, bam, inputs, RATES_4M, 926)
    got = W.sharded(ctx.lib, bam, inputs, RATES_4M, 926, g)
    W.assert_same(got, one, ("B200", g))
    st = got[0][0][0]
    assert st["total"] == 4_000_000 and st["status"] == 0 and st["ms_sort"] > 0 and st["ms_count"] > 0, st
    return one


@pytest.mark.gpu
def test_gpu_sharded_sweep_one_device(gpu_ctx, bam_4m):
    """G = 1 (the driver's device-to-device copy instead of NCCL), 4 M reads, ten rates plus the threshold edge cases"""
    _driver_vs_finish_sweep(gpu_ctx, bam_4m, 1)


@pytest.mark.gpu
def test_gpu_sharded_sweep_nccl(gpu_ctx, bam_4m, oracle):
    """NCCL all-to-all of (key, rate index) over min(n, 4) GPUs: every rate equals the one-device sweep, three the oracle"""
    import torch
    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip("needs 2 GPUs")
    one = _driver_vs_finish_sweep(gpu_ctx, bam_4m, min(n, 4))
    for r in (0.1, 0.5, 1.0):
        st, arr = one[0][RATES_4M.index(r)]
        o = oracle.bam2db(bam_4m["bam"], bam_4m["barcodes"], bam_4m["features"], 0.5, r, 926)
        assert [st[k] for k in KEYS] == [o[k] for k in KEYS], r
        for k in ("m_gene", "m_cell", "m_count"):
            assert np.array_equal(arr[k], o[k]), (r, k)
