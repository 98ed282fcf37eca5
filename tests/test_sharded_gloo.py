"""world_size-2 CPU test (gloo) of the multi-GPU path: the sharded job must reproduce the reference's recorded output byte for byte."""
import gzip
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden")


def test_shard_ranges():
    from fastf_b200.sharded import shard_ranges
    assert shard_ranges(10, 3) == [(0, 4), (4, 7), (7, 10)]
    assert shard_ranges(2, 4) == [(0, 1), (1, 2), (2, 2), (2, 2)]
    assert shard_ranges(0, 2) == [(0, 0), (0, 0)]


@pytest.mark.parametrize("name,world", [("edge-c0.5-r0.5-s926", 2), ("synth4k-c0.5-r0.5-s926", 3)])
def test_sharded_equals_reference(name, world, tmp_path):
    from fastf_b200 import build
    from dbdigest import db_digest
    emu = build.build_emu()
    case = [c for c in json.load(open(os.path.join(GOLD, "manifest.json")))["cases"] if c["name"] == name][0]
    d = os.path.join(GOLD, case["dir"])
    env = dict(os.environ, FASTF_GPU_LIB=emu, OMP_NUM_THREADS="1")
    port = 29600 + (os.getpid() % 300)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(world), "--master-addr", "127.0.0.1", "--master-port", str(port),
           os.path.join(ROOT, "tests", "sharded_worker.py"), d, str(tmp_path), str(case["rate_cell"]), str(case["rate_depth"]), str(case["seed"])]
    r = subprocess.run(cmd, env=env, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-3000:]
    for f in ("matrix.mtx.gz", "barcodes.tsv.gz", "features.tsv.gz"):
        assert gzip.open(os.path.join(tmp_path, f), "rb").read() == gzip.open(os.path.join(d, case["expect"], f), "rb").read(), f
    want = json.load(open(os.path.join(d, case["expect"], "db_digest.json")))
    got = db_digest(os.path.join(tmp_path, "x.db"))
    for t in ("cell", "feature", "umi", "mtx"):
        assert got[t] == want[t], t


def test_every_rank_finds_its_own_shard():
    """shard discovery without walking the file: a block boundary is a header whose BSIZE chain continues; the gzip magic inside
    payloads (here: stored blocks made of nothing but the magic) does not fool it, and unusual extra fields are fine"""
    import struct
    import zlib
    from fastf_b200.sharded import find_block_start, shard_bytes

    def block(payload, level, extra=b""):
        c = zlib.compressobj(level, zlib.DEFLATED, -15)
        comp = c.compress(payload) + c.flush()
        xtra = extra + b"BC" + struct.pack("<HH", 2, 12 + len(extra) + 6 + len(comp) + 8 - 1)
        return b"\x1f\x8b\x08\x04\0\0\0\0\0\xff" + struct.pack("<H", len(xtra)) + xtra + comp + struct.pack("<II", zlib.crc32(payload), len(payload))

    magic = b"\x1f\x8b\x08\x04\0\0\0\0\0\xff\x06\0BC\x02\0\x30\0"   # a complete, plausible-looking BGZF header as DATA
    blocks = [block(magic * 200, 0), block(b"ACGT" * 5000, 6, extra=b"XY\x03\0abc"), block(magic * 500, 0), block(b"", 6), block(bytes(range(256)) * 40, 1)] * 7
    img = np.frombuffer(b"".join(blocks), dtype=np.uint8)
    starts = np.cumsum([0] + [len(b) for b in blocks])
    for pos in list(range(0, img.size, 997)) + [int(x) for x in starts[:-1]] + [int(x) + 1 for x in starts[:-1]]:
        want = int(starts[np.searchsorted(starts, pos, side="left")])
        assert find_block_start(img, pos) == want, pos
    for world in (1, 2, 3, 5, 64):
        cuts = [shard_bytes(img, r, world) for r in range(world)]
        assert cuts[0][0] == 0 and cuts[-1][1] == img.size
        assert all(a[1] == b[0] for a, b in zip(cuts, cuts[1:])) and all(lo in starts and hi in starts for lo, hi in cuts)


def test_a_failing_rank_does_not_hang_the_others(tmp_path):
    """the second half of the BAM is garbage: rank 1 fails in its feed, the ranks agree on it before any collective, all of them return 1"""
    import shutil
    from fastf_b200 import build
    emu = build.build_emu()
    case = [c for c in json.load(open(os.path.join(GOLD, "manifest.json")))["cases"] if c["name"] == "synth4k-c0.5-r0.5-s926"][0]
    d = tmp_path / "in"
    shutil.copytree(os.path.join(GOLD, case["dir"]), str(d))
    raw = bytearray(open(d / "in.bam", "rb").read())
    half = len(raw) // 2
    # keep the BGZF framing of rank 1's shard (the ranks must find it) but break its deflate payloads
    from fastf_b200.sharded import find_block_start, _bgzf_block_size
    o = find_block_start(np.frombuffer(bytes(raw), dtype=np.uint8), half)
    bs = _bgzf_block_size(np.frombuffer(bytes(raw), dtype=np.uint8), o)
    for k in range(o + 18, o + bs - 8):
        raw[k] = 0xff
    open(d / "in.bam", "wb").write(bytes(raw))
    out = tmp_path / "out"
    out.mkdir()
    env = dict(os.environ, FASTF_GPU_LIB=emu, OMP_NUM_THREADS="1")
    port = 29900 + (os.getpid() % 90)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1", "--master-port", str(port),
           os.path.join(ROOT, "tests", "sharded_worker.py"), str(d), str(out), str(case["rate_cell"]), str(case["rate_depth"]), str(case["seed"])]
    r = subprocess.run(cmd, env=env, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=300)
    assert r.returncode != 0
    assert "bam2db (rank 1)" in r.stdout and "bam2db (rank 0)" in r.stdout and "another rank failed" in r.stdout, r.stdout[-2000:]
