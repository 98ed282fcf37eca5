"""The one-process multi-GPU driver of the library (fastf_b200/csrc/sharded.cu) on CPU: the same code linked against the SIMT emulator
with several emulated devices (the NCCL all-to-all is replaced by host copies there; the NCCL path itself runs in the -m gpu test)."""
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.parametrize("g,n_reads,rc,rd,seed", [(2, 6000, 0.7, 0.6, 31), (3, 5000, 1.0, 0.3, 926), (5, 2500, 0.5, 0.9, 4)])
def test_c_sharded_driver_equals_single_job_and_oracle(g, n_reads, rc, rd, seed):
    from fastf_b200 import build
    env = dict(os.environ, FASTF_GPU_LIB=build.build_emu(), FASTF_EMU_DEVICES=str(g))
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "sharded_c_worker.py"), str(g), str(n_reads), str(rc), str(rd), str(seed)], env=env,
                       stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=900)
    assert r.returncode == 0 and "OK sharded C driver" in r.stdout, r.stdout[-3000:]


@pytest.mark.parametrize("name,how", [("synth4k-c0.5-r0.5-s926", "--gpus"), ("edge-c0.8-r0.6-s3", "FASTF_GPUS")])
def test_c_cli_gpus_option_on_the_emulator(name, how, tmp_path):
    """`fastF bam2db ... --gpus 3` (and FASTF_GPUS=3 under the reference's own main.c): the files equal the reference's goldens"""
    import gzip
    import json
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from dbdigest import db_digest
    from fastf_b200 import build
    gold = os.path.join(ROOT, "tests", "golden")
    case = [c for c in json.load(open(os.path.join(gold, "manifest.json")))["cases"] if c["name"] == name][0]
    d = os.path.join(gold, case["dir"])
    out = str(tmp_path)
    env = dict(os.environ, FASTF_EMU_DEVICES="3")
    if how == "--gpus":
        exe, extra = build.build_cli(emu=True), ["--gpus", "3"]
    else:
        exe, extra = build.build_ref_main_emu(), []
        if not exe:
            pytest.skip("reference sources absent and no prebuilt fastF_gpu_emu")
        env["FASTF_GPUS"] = "3"
    cmd = [exe, "bam2db", "-b", "in.bam", "-f", "features.tsv.gz", "-a", "barcodes.tsv.gz", "-d", os.path.join(out, "x.db"), "-c", str(case["rate_cell"]), "-r", str(case["rate_depth"]),
           "-o", out, "-s", str(case["seed"])] + (["-u"] if case.get("umicopies") else []) + extra
    r = subprocess.run(cmd, cwd=d, env=env, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-2000:]
    for f in ["matrix.mtx.gz", "barcodes.tsv.gz", "features.tsv.gz"] + (["umi.tsv.gz"] if case.get("umicopies") else []):
        assert gzip.open(os.path.join(out, f), "rb").read() == gzip.open(os.path.join(d, case["expect"], f), "rb").read(), f
    assert db_digest(os.path.join(out, "x.db")) == json.load(open(os.path.join(d, case["expect"], "db_digest.json")))


@pytest.mark.gpu
def test_c_sharded_driver_nccl(tmp_path):
    """NCCL all-to-all inside the library on real GPUs (needs >= 2; gpurun --gpus 2)"""
    import torch
    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip("needs 2 GPUs")
    g = min(n, 4)
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "sharded_c_worker.py"), str(g), "600000", "0.8", "0.5", "926"], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=900)
    assert r.returncode == 0 and "OK sharded C driver" in r.stdout, r.stdout[-3000:]
