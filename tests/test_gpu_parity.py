"""GPU parity tests (run on the B200 with `-m gpu`): the CUDA path, called through the C-ABI, against the CPU oracle on the
same seeded inputs, against the golden fixtures recorded from the unmodified reference, and -- at large sizes -- through
size-independent properties.  Bit-exact everywhere (integer / byte work)."""
import ctypes as C
import gzip
import json
import os
import zlib

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden")


def _cases(kind):
    p = os.path.join(GOLD, "manifest.json")
    return [c for c in json.load(open(p))["cases"] if c["kind"] == kind] if os.path.exists(p) else []


# ------------------------------------------------------------------------------------------------ single kernels
def test_mt19937_stream_matches_reference_generator(gpu_ctx, oracle):
    from fastf_b200 import _lib
    n = 3_000_001
    for seed in (926, 5489, 0, 0xFFFFFFFF):
        out = np.zeros(n, dtype=np.uint32)
        gpu_ctx.check(gpu_ctx.lib.fastf_mt19937_host(gpu_ctx.h, seed, n, out.ctypes.data_as(_lib.c_u32p)), "mt")
        assert np.array_equal(out, oracle.mt_stream(seed, n))
    out = np.zeros(10000, dtype=np.uint32)
    gpu_ctx.check(gpu_ctx.lib.fastf_mt19937_host(gpu_ctx.h, 5489, 10000, out.ctypes.data_as(_lib.c_u32p)), "mt")
    assert int(out[-1]) == 4123659995   # public mt19937ar known answer


@pytest.mark.parametrize("seed,first", [(926, 1), (926, 623), (926, 624), (926, 1000003), (5489, 123456789), (7, 3_000_000_017)])
def test_mt19937_jump_ahead_lands_on_the_reference_stream(gpu_ctx, oracle, seed, first):
    """GF(2) jump-ahead (mt_jump.h + fastf_mt_jump_batch_kernel): the outputs from stream index `first` on must be the reference generator's"""
    from fastf_b200 import _lib
    n = 5000
    out = np.zeros(n, dtype=np.uint32)
    gpu_ctx.check(gpu_ctx.lib.fastf_mt19937_host_from(gpu_ctx.h, seed, first, n, out.ctypes.data_as(_lib.c_u32p)), "mt from")
    if first + n <= 200_000_000:
        want = oracle.mt_stream(seed, first + n)[first:]
    else:
        # too far for a full oracle run in a test: jump-ahead must at least be consistent with a jump to an earlier point + sequential generation
        back = 2_000_000
        ref = np.zeros(back + n, dtype=np.uint32)
        gpu_ctx.check(gpu_ctx.lib.fastf_mt19937_host_from(gpu_ctx.h, seed, first - back, back + n, ref.ctypes.data_as(_lib.c_u32p)), "mt from")
        want = ref[back:]
    assert np.array_equal(out, want)


@pytest.mark.parametrize("rate", [0.0, 0.1, 0.3, 0.5, 0.9, 1.0])
def test_keep_bits_match_reference_rule(gpu_ctx, oracle, rate):
    from fastf_b200 import _lib
    n = 1_000_003
    T = gpu_ctx.lib.fastf_keep_threshold(C.c_float(rate))
    bits = np.zeros((n + 31) // 32, dtype=np.uint32)
    gpu_ctx.check(gpu_ctx.lib.fastf_mt19937_keepbits_host(gpu_ctx.h, 926, n, T, bits.ctypes.data_as(_lib.c_u32p)), "keepbits")
    got = np.unpackbits(bits.view(np.uint8), bitorder="little")[:n].astype(bool)
    u = oracle.mt_stream(926, n)
    want = (u.astype(np.float64) * (1.0 / 4294967295.0)) < np.float64(np.float32(rate))   # genrand_real1() >= rate -> drop
    assert np.array_equal(got, want)


def _inflate(gpu_ctx, img, lanes):
    buf = np.frombuffer(img, dtype=np.uint8)
    out, n, ms = C.c_void_p(), C.c_size_t(), C.c_float()
    rc = gpu_ctx.lib.fastf_inflate_host(gpu_ctx.h, C.c_void_p(buf.ctypes.data), buf.size, lanes, C.byref(out), C.byref(n), C.byref(ms))
    if rc:
        return None
    data = C.string_at(out, n.value)
    gpu_ctx.lib.fastf_free(out)
    return data


@pytest.mark.parametrize("lanes", [32, 16, 8, 1])   # 1 = thread-per-stream kernel
def test_inflate_adversarial_blocks(gpu_ctx, lanes):
    import bamgen
    rng = np.random.default_rng(3)
    payloads = [b"", b"a", b"abc" * 20000, bytes(rng.integers(0, 256, 65280, dtype=np.uint8)), bytes(rng.integers(0, 4, 65536, dtype=np.uint8)),
                b"\0" * 65536, bytes(rng.integers(65, 70, 40000, dtype=np.uint8)), (b"ACGT" * 7 + b"N") * 2000, bytes(range(256)) * 255]
    modes = [(6, zlib.Z_DEFAULT_STRATEGY), (0, zlib.Z_DEFAULT_STRATEGY), (6, zlib.Z_FIXED), (9, zlib.Z_DEFAULT_STRATEGY), (1, zlib.Z_HUFFMAN_ONLY), (6, zlib.Z_RLE), (1, zlib.Z_DEFAULT_STRATEGY)]
    for shift in range(len(modes)):
        use = []
        for i, p in enumerate(payloads):
            lvl, strat = modes[(i + shift) % len(modes)]
            if lvl == 0 and len(p) > 65000:
                lvl = 1   # a stored 64 KiB payload does not fit one BGZF block
            if len(p) > 65000 and strat in (zlib.Z_HUFFMAN_ONLY, zlib.Z_FIXED) and p[:1] != b"\0":
                strat = zlib.Z_DEFAULT_STRATEGY
            use.append((lvl, strat))
        img = b"".join(bamgen.bgzf_block(p, *m) for p, m in zip(payloads, use)) + bamgen.EOF_BLOCK
        assert _inflate(gpu_ctx, img, lanes) == b"".join(payloads)


def test_inflate_flags_corrupt_streams(gpu_ctx):
    import bamgen
    good = bamgen.bgzf_block(b"hello world, hello world, hello world" * 100)
    for pos in (20, 25, 40):
        bad = bytearray(good)
        bad[pos] ^= 0xFF
        img = bytes(bad) + bamgen.EOF_BLOCK
        out = _inflate(gpu_ctx, img, 32)
        assert (_inflate(gpu_ctx, img, 1) is None) == (out is None)
        want = None
        try:
            want = zlib.decompress(bytes(bad[18:-8]), -15)
        except zlib.error:
            pass
        if want is None or len(want) != 3700:
            assert out is None, "corrupt stream at byte %d must be reported" % pos
            assert b"malformed" in gpu_ctx.lib.fastf_last_error(gpu_ctx.h)
        elif want != bytes(b"hello world, hello world, hello world" * 100):
            assert out is None and b"crc32" in gpu_ctx.lib.fastf_last_error(gpu_ctx.h)


def test_inflate_checks_the_bgzf_crc32(gpu_ctx):
    """htslib verifies the CRC32 of every BGZF block (bgzf_read_block, reached from sam_read1, reference src/bam2db_ds.c:360): a
    payload that inflates cleanly to the wrong bytes, or a wrong CRC field, must fail; FASTF_INFLATE_NO_CRC skips the check."""
    import bamgen
    rng = np.random.default_rng(5)
    payloads = [bytes(rng.integers(0, 256, n, dtype=np.uint8)) for n in (1, 15, 16, 17, 511, 512, 513, 4096, 40001, 65280)] + [b"", b"ACGT" * 16384]
    blocks = [bamgen.bgzf_block(p, 0 if len(p) < 65000 else 1, zlib.Z_DEFAULT_STRATEGY) for p in payloads[:-1]] + [bamgen.bgzf_block(payloads[-1])]
    img = b"".join(blocks) + bamgen.EOF_BLOCK
    for lanes in (0, 32):
        assert _inflate(gpu_ctx, img, lanes) == b"".join(payloads)          # every segment split of the warp-parallel CRC agrees with zlib's
    off = 0
    for k, b in enumerate(blocks):
        if len(payloads[k]) and len(payloads[k]) < 65000 and k < len(blocks) - 1:
            bad = bytearray(img)
            bad[off + 18 + 5 + len(payloads[k]) // 2] ^= 0x20                      # inside the stored payload: still a valid deflate stream
            assert _inflate(gpu_ctx, bytes(bad), 0) is None, "block %d" % k
            assert b"crc32" in gpu_ctx.lib.fastf_last_error(gpu_ctx.h)
            assert _inflate(gpu_ctx, bytes(bad), 0x200) is not None             # FASTF_INFLATE_NO_CRC
        bad = bytearray(img)
        bad[off + len(b) - 8] ^= 1                                               # the CRC32 field itself
        assert _inflate(gpu_ctx, bytes(bad), 0) is None and b"crc32" in gpu_ctx.lib.fastf_last_error(gpu_ctx.h)
        off += len(b)


def test_inflate_synthetic_bam_vs_zlib(gpu_ctx, synth, oracle):
    p = synth.params(n_reads=100000, n_cells=500, n_genes=800, seed=21)
    bam, st = synth.bam(p)
    want = oracle.inflate(bam)
    for lanes in (32, 16, 8, 1):
        assert _inflate(gpu_ctx, bam, lanes) == want


@pytest.mark.parametrize("n,bits", [(1, 64), (1000, 20), (2049, 64), (1 << 20, 54), (3_000_017, 58)])
def test_radix_sort_is_a_stable_sort(gpu_ctx, n, bits):
    from fastf_b200 import _lib
    rng = np.random.default_rng(n)
    keys = rng.integers(0, 2**63, n, dtype=np.uint64) >> np.uint64(64 - bits) if bits < 64 else rng.integers(0, 2**64, n, dtype=np.uint64)
    keys[: n // 3] = keys[n // 2: n // 2 + n // 3]   # plenty of duplicates
    vals = np.arange(n, dtype=np.uint32)
    k2, v2 = keys.copy(), vals.copy()
    gpu_ctx.check(gpu_ctx.lib.fastf_sort_u64_host(gpu_ctx.h, k2.ctypes.data_as(_lib.c_u64p), v2.ctypes.data_as(_lib.c_u32p), n, bits), "sort")
    order = np.argsort(keys, kind="stable")
    assert np.array_equal(k2, keys[order]) and np.array_equal(v2, order.astype(np.uint32))
    k3 = keys.copy()
    gpu_ctx.check(gpu_ctx.lib.fastf_sort_u64_host(gpu_ctx.h, k3.ctypes.data_as(_lib.c_u64p), None, n, bits), "sort")
    assert np.array_equal(k3, k2)


@pytest.mark.parametrize("n,bits,distinct", [(0, 40, 1), (1, 64, 1), (5000, 30, 7), (1 << 20, 54, 90_000), (2_500_003, 58, 2_400_000)])
def test_unique_counts_equal_numpy_unique(gpu_ctx, n, bits, distinct):
    """copies per distinct key (what -u/--umicopies groups by, reference src/bam2db_ds.c:527-530): device sort + run-length heads"""
    from fastf_b200 import bam2db_host
    rng = np.random.default_rng(n + bits)
    pool = rng.integers(0, 2**63, distinct, dtype=np.uint64) >> np.uint64(63 - min(bits, 63))
    keys = pool[rng.integers(0, distinct, n)] if n else np.zeros(0, np.uint64)
    uniq, counts = bam2db_host.unique_counts(gpu_ctx, keys, bits)
    wu, wc = np.unique(keys, return_counts=True)
    assert np.array_equal(uniq, wu) and np.array_equal(counts.astype(np.int64), wc)


HW = 0x100   # FASTF_INFLATE_HW_ENGINE


def test_hw_decompress_engine_matches_zlib_and_sm_kernel(gpu_ctx, synth, oracle, tmp_path):
    """optional engine: the B200 hardware decompression engine must give the same bytes as zlib / our SM kernel and the same bam2db result"""
    from fastf_b200 import bam2db_host as B
    paths, _ = synth.write_bam_set(str(tmp_path), n_reads=200000, n_cells=500, n_genes=800, seed=21, p_umi_n=0.004)
    bam = open(paths["bam"], "rb").read()
    got = _inflate(gpu_ctx, bam, HW)
    if got is None and b"unavailable" in gpu_ctx.lib.fastf_last_error(gpu_ctx.h):
        pytest.skip("hardware decompression engine not available on this GPU / driver")
    assert got == oracle.inflate(bam)
    _check_against_oracle(gpu_ctx, oracle, paths, 0.5, 0.5, 926, inflate_lanes=HW, chunk_inflated_bytes=8 << 20)


# ------------------------------------------------------------------------------------------------ bam2db
def _oracle_rows_as_keys(o, stats):
    bg, bu, mb = stats["bits_gene"], stats["bits_umi"], stats["umi_max_bytes"]
    nb = o["row_umi_nbytes"].astype(np.int64)
    content = (o["row_umi"].astype(np.uint64) >> np.uint64(64 - 8 * mb))
    code = np.where(nb >= 0, (np.uint64(1) << np.uint64(bu - 1)) | (content << np.uint64(3)) | np.maximum(nb, 0).astype(np.uint64), np.uint64(0))
    return (o["row_cell"].astype(np.uint64) << np.uint64(bg + bu)) | (o["row_gene"].astype(np.uint64) << np.uint64(bu)) | code


def _check_against_oracle(gpu_ctx, oracle, paths, rc, rd, seed, **kw):
    from fastf_b200 import bam2db_host as B
    want = oracle.bam2db(paths["bam"], paths["barcodes"], paths["features"], rc, rd, seed)
    inputs = B.Bam2dbInputs(gpu_ctx.lib, paths["barcodes"], paths["features"], rc, seed)
    assert inputs.d0 == want["d0"] and len(inputs.cells) == want["n_cell_rows"] and len(inputs.features) == want["n_features"]
    stats, out = B.run_device(gpu_ctx, np.fromfile(paths["bam"], dtype=np.uint8), inputs, rd, seed, want_rows=True, **kw)
    for k in ("total", "cb_valid", "sampled", "valid", "nnz"):
        assert stats[k] == want[k], (k, stats[k], want[k])
    assert np.array_equal(out["m_gene"], want["m_gene"])
    assert np.array_equal(out["m_cell"], want["m_cell"])
    assert np.array_equal(out["m_count"], want["m_count"])
    assert np.array_equal(out["row_keys"], _oracle_rows_as_keys(want, stats))   # the sqlite `umi` table, in read order
    return stats, out


@pytest.mark.parametrize("rc,rd,seed", [(0.5, 0.5, 926), (1.0, 0.3, 926), (1.0, 1.0, 1), (0.2, 0.9, 77), (0.9, 0.1, 4242), (0.5, 0.0, 5)])
def test_bam2db_matches_oracle(gpu_ctx, oracle, synth, tmp_path, rc, rd, seed):
    paths, _ = synth.write_bam_set(str(tmp_path), n_reads=300000, n_cells=1000, n_genes=2000, seed=seed, p_umi_n=0.005, n_molecules=100000)
    _check_against_oracle(gpu_ctx, oracle, paths, rc, rd, seed)


def test_bam2db_config1_shape(gpu_ctx, oracle, synth, tmp_path):
    """BASELINE.json configs[0]: 1M reads, 1k cells, 2k genes, -c 0.5 -r 0.5 -s 926"""
    paths, _ = synth.write_bam_set(str(tmp_path), n_reads=1000000, n_cells=1000, n_genes=2000, seed=11, p_umi_n=0.001)
    stats, _ = _check_against_oracle(gpu_ctx, oracle, paths, 0.5, 0.5, 926)
    assert stats["total"] == 1000000


def test_bam2db_parallel_draw_segments(gpu_ctx, oracle, synth, tmp_path):
    """enough CB-valid reads (~2.9 M) that the keep bits are generated by all 32 jump-ahead segments at once, and a non-zero D0"""
    paths, _ = synth.write_bam_set(str(tmp_path), n_reads=3000000, n_cells=3000, n_genes=4000, seed=13, p_umi_n=0.001, p_cb_in_list=0.97, p_cb_not_in_list=0.02)
    stats, _ = _check_against_oracle(gpu_ctx, oracle, paths, 0.999, 0.37, 20240, chunk_inflated_bytes=256 << 20)
    assert stats["cb_valid"] > 2_700_000


@pytest.mark.parametrize("lanes,chunk,piece", [(32, 1 << 20, 0), (16, 3 << 20, 1000003), (8, 0, 65536), (32, 1 << 20, 777), (1, 2 << 20, 0), (1, 0, 250000)])
def test_bam2db_streaming_is_invariant(gpu_ctx, oracle, synth, tmp_path, lanes, chunk, piece):
    """any chunking of the inflated stream and any split of the compressed bytes (also inside BGZF blocks) gives the same result"""
    paths, _ = synth.write_bam_set(str(tmp_path), n_reads=60000, n_cells=300, n_genes=500, seed=9, p_umi_n=0.01, n_molecules=20000)
    _check_against_oracle(gpu_ctx, oracle, paths, 0.7, 0.6, 31, inflate_lanes=lanes, chunk_inflated_bytes=chunk, feed_piece=piece)


@pytest.mark.parametrize("case", _cases("bam2db"), ids=lambda c: c["name"])
def test_bam2db_golden_files(gpu_ctx, case, tmp_path):
    """the whole operator (files in, files out) against outputs recorded from the unmodified reference; includes the edge-case BAM"""
    import sqlite3
    import fastf_b200
    from fastf_b200 import bam2db_host
    from dbdigest import db_digest
    d = os.path.join(GOLD, case["dir"])
    out = str(tmp_path)
    cwd = os.getcwd()
    os.chdir(d)
    bam2db_host._umi_copies_flag = 1 if case.get("umicopies") else 0
    try:
        assert fastf_b200.bam2db("in.bam", os.path.join(out, "x.db"), out, "barcodes.tsv.gz", "features.tsv.gz", case["rate_cell"], case["rate_depth"], case["seed"], ctx=gpu_ctx) == 0
    finally:
        os.chdir(cwd)
        bam2db_host._umi_copies_flag = 0
    for f in ["matrix.mtx.gz", "barcodes.tsv.gz", "features.tsv.gz"] + (["umi.tsv.gz"] if case.get("umicopies") else []):
        assert gzip.open(os.path.join(out, f), "rb").read() == gzip.open(os.path.join(d, case["expect"], f), "rb").read(), f
    assert db_digest(os.path.join(out, "x.db")) == json.load(open(os.path.join(d, case["expect"], "db_digest.json")))   # every table, row for row
    db = sqlite3.connect(os.path.join(out, "x.db"))
    n_umi, n_null = db.execute("select count(*), sum(encoded_umi is null) from umi").fetchone()
    assert n_umi == case["counters"][2]
    # the device COO equals what the reference's SQL computes from the umi table the device produced
    sql = db.execute("SELECT feature_index, cell_index, COUNT(DISTINCT encoded_umi) FROM umi GROUP BY cell_index, feature_index").fetchall()
    assert sql == db.execute("select * from mtx").fetchall()


def test_bam2db_rejects_truncated_and_foreign_input(gpu_ctx, synth, tmp_path):
    from fastf_b200 import bam2db_host as B, _lib
    import bamgen
    paths, _ = synth.write_bam_set(str(tmp_path), n_reads=5000, n_cells=50, n_genes=50, seed=2)
    inputs = B.Bam2dbInputs(gpu_ctx.lib, paths["barcodes"], paths["features"], 1.0, 926)
    bam = np.fromfile(paths["bam"], dtype=np.uint8)
    with pytest.raises(_lib.FastfError, match="ends inside a BGZF block"):
        B.run_device(gpu_ctx, bam[:-100].copy(), inputs, 1.0, 926)
    with pytest.raises(_lib.FastfError, match="not a BGZF"):
        B.run_device(gpu_ctx, np.frombuffer(gzip.compress(b"hello" * 100), dtype=np.uint8), inputs, 1.0, 926)
    # one flipped quality byte inside a block whose deflate stream stays valid: the CRC32 of the trailer catches it
    blocks_at = []
    o = 0
    raw = bytes(bam)
    while o < len(raw):
        bs = int.from_bytes(raw[o + 16:o + 18], "little") + 1
        blocks_at.append((o, bs))
        o += bs
    o, bs = blocks_at[len(blocks_at) // 2]
    rebuilt = bytearray(zlib.decompress(raw[o + 18:o + bs - 8], -15))
    rebuilt[len(rebuilt) // 2] ^= 1
    forged = bytearray(bamgen.bgzf_block(bytes(rebuilt)))
    forged[-8:-4] = raw[o + bs - 8:o + bs - 4]                                   # keep the ORIGINAL crc: payload and trailer disagree
    with pytest.raises(_lib.FastfError, match="crc32"):
        B.run_device(gpu_ctx, np.frombuffer(raw[:o] + bytes(forged) + raw[o + bs:], dtype=np.uint8), inputs, 1.0, 926)
    # a record split across two BGZF blocks (foreign writer): reported, never silently mis-parsed
    raw = zlib.decompress(bytes(bam[18:]), -15) if False else None
    whole = gzip.decompress(bytes(bam))
    img = bamgen.bgzf_file([whole[i:i + 10007] for i in range(0, len(whole), 10007)])
    with pytest.raises(_lib.FastfError, match="straddles"):
        B.run_device(gpu_ctx, np.frombuffer(img, dtype=np.uint8), inputs, 1.0, 926)


def test_bam2db_default_chunking_vs_oracle_14M_reads(gpu_ctx, oracle, synth, tmp_path):
    """BASELINE configs[2] shape (10k cells, 36k genes, -c 1.0 -r 0.3 -s 926) at 14 M distinct reads with the DEFAULT chunking the
    benchmark runs with: several chunks of 2 x n_sm x streams-per-SM BGZF blocks (blocks pending across feed calls, ring-buffer reuse,
    `cand` growth from counter snapshots, 4 M draws through the jump-ahead segments), fed in 256 MiB pieces like the file readers do.
    Counters, COO and the kept rows (the sqlite `umi` table, in read order) equal the oracle's."""
    paths, st = synth.write_bam_set(str(tmp_path), n_reads=14_000_000, n_cells=10000, n_genes=36000, seed=1234, p_umi_n=0.001)
    stats, _ = _check_against_oracle(gpu_ctx, oracle, paths, 1.0, 0.3, 926, feed_piece=256 << 20)
    assert stats["total"] == 14_000_000 and stats["n_chunks"] >= 2, stats["n_chunks"]


def test_bam2db_large_properties(gpu_ctx, synth, tmp_path):
    """size-independent properties on a run too large for the oracle to be comfortable: counters are consistent, the COO is
    strictly ascending in (cell, gene), sum(count) = number of distinct non-NULL keys, -r 1.0 keeps every draw but u = 2^32-1,
    feeding the record blocks twice doubles the read counters and leaves distinct counts unchanged (idempotence of dedup)."""
    from fastf_b200 import bam2db_host as B
    from fastf_b200 import _lib
    paths, st = synth.write_bam_set(str(tmp_path), n_reads=4_000_000, n_cells=5000, n_genes=20000, seed=77, p_umi_n=0.002)
    inputs = B.Bam2dbInputs(gpu_ctx.lib, paths["barcodes"], paths["features"], 1.0, 926)
    bam = np.fromfile(paths["bam"], dtype=np.uint8)
    stats, out = B.run_device(gpu_ctx, bam, inputs, 1.0, 926, want_rows=True)
    assert stats["total"] == 4_000_000 and stats["sampled"] == stats["cb_valid"] and stats["valid"] <= stats["sampled"]
    ck = out["m_cell"].astype(np.uint64) << np.uint64(32) | out["m_gene"].astype(np.uint64)
    assert np.all(ck[1:] > ck[:-1])
    rows = out["row_keys"]
    nn = (rows >> np.uint64(stats["bits_umi"] - 1)) & np.uint64(1)
    assert int(out["m_count"].sum()) == np.unique(rows[nn == 1]).size
    assert stats["nnz"] == np.unique(rows >> np.uint64(stats["bits_umi"])).size
    # feed the record blocks twice
    cap = int(st.n_blocks) + 8
    io, il, isz = np.zeros(cap, np.uint64), np.zeros(cap, np.uint32), np.zeros(cap, np.uint32)
    used = C.c_size_t()
    nb = gpu_ctx.lib.fastf_bgzf_index_host(C.c_void_p(bam.ctypes.data), bam.size, io.ctypes.data_as(_lib.c_u64p), il.ctypes.data_as(_lib.c_u32p), isz.ctypes.data_as(_lib.c_u32p), cap, C.byref(used))
    first_rec, eof = int(io[1]) - 18, int(io[nb - 1]) - 18
    with B.Bam2dbJob(gpu_ctx, inputs, 1.0, 926, want_rows=False) as job:
        job.feed(bam.ctypes.data, eof)
        job.feed(bam.ctypes.data + first_rec, eof - first_rec)
        job.feed(bam.ctypes.data + eof, bam.size - eof)
        s2, o2 = job.finish()
    assert s2["total"] == 2 * stats["total"] and s2["cb_valid"] == 2 * stats["cb_valid"]
    assert s2["nnz"] == stats["nnz"] and np.array_equal(o2["m_count"], out["m_count"]) and np.array_equal(o2["m_gene"], out["m_gene"])


# ------------------------------------------------------------------------------------------------ freq
@pytest.mark.parametrize("case", _cases("freq"), ids=lambda c: c["name"])
def test_freq_golden_files(gpu_ctx, case, tmp_path):
    import fastf_b200
    d = os.path.join(GOLD, case["dir"])
    assert fastf_b200.freq(os.path.join(d, case["input"]), str(tmp_path), case["l"], case["u"], ctx=gpu_ctx) == 0
    assert open(tmp_path / "whitelist.txt", "rb").read() == gzip.open(os.path.join(d, case["expect"]), "rb").read()


@pytest.mark.parametrize("n,cells,l,u", [(400000, 2000, 16, 12), (400000, 20000, 16, 0), (250000, 300, 16, 10), (100000, 50, 4, 0)])
def test_freq_matches_oracle(gpu_ctx, oracle, synth, tmp_path, n, cells, l, u):
    import fastf_b200
    fq, _ = synth.write_fastq(str(tmp_path), n_reads=n, n_cells=cells, seed=n + l, p_umi_n=0.01)
    assert fastf_b200.freq(fq, str(tmp_path), l, u, ctx=gpu_ctx) == 0
    oracle.freq(fq, l, u, str(tmp_path / "want.txt"))
    assert open(tmp_path / "whitelist.txt", "rb").read() == open(tmp_path / "want.txt", "rb").read()


def test_freq_streaming_10M_reads_vs_oracle(gpu_ctx, oracle, synth, tmp_path, monkeypatch):
    """BASELINE configs[1] shape (20k true barcodes + error variants, -l 16 -u 12) at 10 M reads, streamed through HBM in chunks of 4096
    BGZF blocks (the default chunk would swallow this file whole): ~10^7 distinct keys, whitelist byte-identical to the oracle's"""
    import fastf_b200
    fq, _ = synth.write_fastq(str(tmp_path), n_reads=10_000_000, n_cells=20000, seed=77, p_umi_n=0.001)
    oracle.freq(fq, 16, 12, str(tmp_path / "want.txt"))
    monkeypatch.setenv("FASTF_STREAM_CHUNK_BLOCKS", "4096")
    assert fastf_b200.freq(fq, str(tmp_path), 16, 12, ctx=gpu_ctx) == 0
    assert open(tmp_path / "whitelist.txt", "rb").read() == open(tmp_path / "want.txt", "rb").read()


def test_freq_plain_text_input_and_gzip_refusal(gpu_ctx, oracle, tmp_path):
    import fastf_b200
    raw = gzip.open(os.path.join(GOLD, "freq", "ragged.fastq.gz"), "rb").read()
    (tmp_path / "plain.fastq").write_bytes(raw)
    assert fastf_b200.freq(str(tmp_path / "plain.fastq"), str(tmp_path), 16, 12, ctx=gpu_ctx) == 0
    assert open(tmp_path / "whitelist.txt", "rb").read() == gzip.open(os.path.join(GOLD, "freq", "expect_ragged_l16_u12.txt.gz"), "rb").read()
    (tmp_path / "single.fastq.gz").write_bytes(gzip.compress(raw))
    assert fastf_b200.freq(str(tmp_path / "single.fastq.gz"), str(tmp_path), 16, 12, ctx=gpu_ctx) == 1   # loud refusal, not a CPU fallback


def test_freq_large_properties(gpu_ctx, synth, tmp_path):
    """counts sum to the number of reads; keys strictly ascending; first-occurrence ordinals are a valid insertion order"""
    from fastf_b200 import freq_host as F
    fq, _ = synth.write_fastq(str(tmp_path), n_reads=6_000_000, n_cells=20000, seed=1, p_umi_n=0.001)
    st = {}
    h = F.cell_counts(fq, 16, 12, ctx=gpu_ctx, stats_out=st)
    assert h.n_reads == 6_000_000 and int(np.sum(h.count)) == 6_000_000
    assert all(h.keys[i] < h.keys[i + 1] for i in range(0, len(h.keys) - 1, 997))
    assert len(set(h.first.tolist())) == len(h.keys) and int(h.first.min()) == 0


# ------------------------------------------------------------------------------------------------ the C host
@pytest.mark.parametrize("name", ["synth4k-c0.5-r0.5-s926", "edge-c0.8-r0.6-s3"])
def test_c_cli_bam2db_golden(gpu_ctx, name, tmp_path):
    """`fastF bam2db ...` (fastf_b200/host, C) against the outputs recorded from the reference CLI"""
    import subprocess
    from fastf_b200 import build
    from dbdigest import db_digest
    case = [c for c in _cases("bam2db") if c["name"] == name][0]
    d = os.path.join(GOLD, case["dir"])
    out = str(tmp_path)
    cli = build.build_cli()
    cmd = [cli, "bam2db", "-b", "in.bam", "-f", "features.tsv.gz", "-a", "barcodes.tsv.gz", "-d", os.path.join(out, "x.db"), "-c", str(case["rate_cell"]), "-r", str(case["rate_depth"]), "-o", out,
           "-s", str(case["seed"])] + (["-u"] if case.get("umicopies") else [])
    r = subprocess.run(cmd, cwd=d, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True)
    assert r.returncode == 0, r.stderr
    assert "In in.bam, total fastQ reads: %d" % case["counters"][0] in r.stdout and "Opened database successfully" in r.stderr
    for f in ["matrix.mtx.gz", "barcodes.tsv.gz", "features.tsv.gz"] + (["umi.tsv.gz"] if case.get("umicopies") else []):
        assert gzip.open(os.path.join(out, f), "rb").read() == gzip.open(os.path.join(d, case["expect"], f), "rb").read(), f
    assert db_digest(os.path.join(out, "x.db")) == json.load(open(os.path.join(d, case["expect"], "db_digest.json")))
    # the reference refuses an existing database (src/main.c:341-345)
    r = subprocess.run(cmd, cwd=d, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True)
    assert r.returncode == 1 and "already exists" in r.stderr


def test_c_cli_freq_golden(gpu_ctx, tmp_path):
    import subprocess
    from fastf_b200 import build
    cli = build.build_cli()
    for case in _cases("freq"):
        d = os.path.join(GOLD, case["dir"])
        r = subprocess.run([cli, "freq", "-R", os.path.join(d, case["input"]), "-o", str(tmp_path), "-l", str(case["l"]), "-u", str(case["u"])], stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True)
        assert r.returncode == 0, r.stderr
        assert open(tmp_path / "whitelist.txt", "rb").read() == gzip.open(os.path.join(d, case["expect"]), "rb").read(), case["name"]


# ------------------------------------------------------------------------------------------------ several GPUs
def test_bam2db_two_gpus_equal_reference_and_one_gpu(gpu_ctx, synth, oracle, tmp_path):
    """2 ranks over NCCL (contiguous block shards, global draw ordinals, all-to-all by cell hash) reproduce the single-GPU result
    and the oracle byte for byte.  Needs 2 GPUs (gpurun --gpus 2); skipped on a 1-GPU box, where tests/test_sharded_gloo.py
    covers the same host logic on CPU."""
    import subprocess
    import sys
    import torch
    import fastf_b200
    from dbdigest import db_digest
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    d = tmp_path / "in"
    d.mkdir()
    paths, _ = synth.write_bam_set(str(d), n_reads=400000, n_cells=800, n_genes=1500, seed=5, p_umi_n=0.004, n_molecules=150000)
    os.rename(paths["bam"], str(d / "in.bam"))
    one, two, ora = tmp_path / "one", tmp_path / "two", tmp_path / "ora"
    for x in (one, two, ora):
        x.mkdir()
    cwd = os.getcwd()
    os.chdir(str(d))
    try:
        assert fastf_b200.bam2db("in.bam", str(one / "x.db"), str(one), "barcodes.tsv.gz", "features.tsv.gz", 0.6, 0.4, 926, ctx=gpu_ctx) == 0
        oracle.bam2db("in.bam", "barcodes.tsv.gz", "features.tsv.gz", 0.6, 0.4, 926, str(ora))
    finally:
        os.chdir(cwd)
    env = dict(os.environ, FASTF_SHARDED_BACKEND="nccl")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1", "--master-port", "29733",
           os.path.join(ROOT, "tests", "sharded_worker.py"), str(d), str(two), "0.6", "0.4", "926"]
    r = subprocess.run(cmd, env=env, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-3000:]
    for f in ("matrix.mtx.gz", "barcodes.tsv.gz", "features.tsv.gz"):
        a, b = gzip.open(str(one / f), "rb").read(), gzip.open(str(two / f), "rb").read()
        assert a == b, f
        assert a == open(str(ora / f[:-3]), "rb").read(), f
    d1, d2 = db_digest(str(one / "x.db")), db_digest(str(two / "x.db"))
    assert d1 == d2


# ---- crb / extract (SURVEY section 8f.2-3) ----
def _tags_cases():
    import tags_cases
    return tags_cases.cases()


@pytest.mark.gpu
@pytest.mark.parametrize("case", _tags_cases(), ids=lambda c: c["name"])
def test_crb_extract_golden_files(gpu_ctx, case, tmp_path):
    """outputs recorded from the unmodified reference (scripts/make_golden_tags.py), byte for byte"""
    import tags_cases
    tags_cases.run_case(gpu_ctx, case, str(tmp_path))


@pytest.mark.gpu
def test_crb_extract_match_oracle_on_synthetic_bam(gpu_ctx, oracle, synth, tmp_path):
    """300k reads, 2000 cells: crb (pairs), extract of a high-cardinality string tag (UB: nearly every read distinct), of GX and of two
    integer tags, against the oracle; exercises the 64-bit hash grouping + byte-for-byte verification at scale"""
    from fastf_b200 import tags_host as T
    paths, _ = synth.write_bam_set(str(tmp_path), n_reads=300000, n_cells=2000, n_genes=3000, seed=8)
    assert T.crb(gpu_ctx, paths["bam"], str(tmp_path / "crb.gz")) == oracle.crb(paths["bam"], str(tmp_path / "crb.txt"))
    assert gzip.open(tmp_path / "crb.gz", "rb").read() == open(tmp_path / "crb.txt", "rb").read()
    for tag, typ in (("UB", 0), ("GX", 0), ("CB", 0), ("xf", 1), ("NH", 1), ("ZZ", 0)):
        got = T.extract_bam(gpu_ctx, paths["bam"], tag, typ, str(tmp_path))
        assert got == oracle.extract(paths["bam"], tag, typ, str(tmp_path / "o.csv")), tag
        assert open(tmp_path / "tag_summary.csv", "rb").read() == open(tmp_path / "o.csv", "rb").read(), tag


@pytest.mark.gpu
def test_crb_extract_refuse_what_crashes_the_reference(gpu_ctx, tmp_path):
    """string extraction of a non-string tag and CB without CR make the reference dereference NULL (src/extract.c:97-100,186): refused loudly"""
    from fastf_b200 import tags_host as T, _lib
    import bamgen
    recs = [bamgen.record("a", [bamgen.aux_Z("CB", "ACGT-1"), bamgen.aux_Z("CR", "ACGT"), bamgen.aux_int("NH", "C", 1)]),
            bamgen.record("b", [bamgen.aux_Z("CB", "ACGT-1"), bamgen.aux_int("NH", "C", 1)])]
    p = str(tmp_path / "x.bam")
    open(p, "wb").write(bamgen.bgzf_file(bamgen.pack_records(bamgen.bam_header(), recs)))
    with pytest.raises(_lib.FastfError, match="tag-not-a-string"):
        T.crb(gpu_ctx, p, str(tmp_path / "o.gz"))
    with pytest.raises(_lib.FastfError, match="tag-not-a-string"):
        T.extract_bam(gpu_ctx, p, "NH", 0, str(tmp_path))
    assert T.extract_bam(gpu_ctx, p, "NH", 1, str(tmp_path)) == (4, 2)


@pytest.mark.gpu
def test_c_cli_crb_extract_golden(gpu_ctx, tmp_path):
    import subprocess
    from fastf_b200 import build
    cli = build.build_cli()
    g = os.path.join(os.path.dirname(__file__), "golden", "tags")
    r = subprocess.run([cli, "crb", "-b", os.path.join(g, "tags.bam"), "-o", "o.gz"], cwd=tmp_path, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=600)
    assert r.returncode == 0 and r.stdout.splitlines() == ["Processed all 904 reads", "Writing to file...", "Done."], r.stdout
    assert gzip.open(tmp_path / "o.gz", "rb").read() == gzip.open(os.path.join(g, "expect_tags_crb.txt.gz"), "rb").read()
    r = subprocess.run([cli, "extract", "-b", os.path.join(g, "tags.bam"), "-t", "GX"], cwd=tmp_path, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=600)
    assert r.returncode == 0 and r.stdout.splitlines() == ["Processed all 1808 reads", "Valid reads: 902"], r.stdout
    assert open(tmp_path / "tag_summary.csv", "rb").read() == gzip.open(os.path.join(g, "expect_tags_extract_GX_0.csv.gz"), "rb").read()


@pytest.mark.gpu
def test_crb_extract_streamed_chunks_and_forced_collisions(gpu_ctx, oracle, synth, tmp_path):
    """the file streams through HBM in chunks (test hook: 5 blocks per chunk) whose groups are merged on the host; a mask on the first
    round's hash keys forces collisions, which the byte-for-byte verification must catch (second round wins)"""
    import numpy as np
    import tags_cases
    from fastf_b200 import tags_host as T
    paths, _ = synth.write_bam_set(str(tmp_path), n_reads=60000, n_cells=300, n_genes=500, seed=12)
    try:
        gpu_ctx.lib.fastf_taghist_test_hooks(gpu_ctx.h, 5, 0x3ff)
        for case in tags_cases.cases():
            if case["input"] == "tags.bam":
                tags_cases.run_case(gpu_ctx, case, str(tmp_path))
        st, _ = T.taghist(gpu_ctx, np.fromfile(paths["bam"], dtype=np.uint8), "CB", 0, "CR")
        assert st["hash_rounds"] == 2 and st["n_blocks"] > 20
        assert T.crb(gpu_ctx, paths["bam"], str(tmp_path / "crb.gz")) == oracle.crb(paths["bam"], str(tmp_path / "crb.txt"))
        assert gzip.open(tmp_path / "crb.gz", "rb").read() == open(tmp_path / "crb.txt", "rb").read()
        for tag, typ in (("UB", 0), ("xf", 1)):
            assert T.extract_bam(gpu_ctx, paths["bam"], tag, typ, str(tmp_path)) == oracle.extract(paths["bam"], tag, typ, str(tmp_path / "o.csv"))
            assert open(tmp_path / "tag_summary.csv", "rb").read() == open(tmp_path / "o.csv", "rb").read(), tag
    finally:
        gpu_ctx.lib.fastf_taghist_test_hooks(gpu_ctx.h, 0, 0)


@pytest.mark.gpu
def test_records_straddling_bgzf_blocks(gpu_ctx, oracle, synth, tmp_path):
    """a BAM re-cut into BGZF blocks of odd sizes (records cross block boundaries, as htsjdk or STAR write them): refused by the strict
    default, bit-exact vs the oracle with FASTF_BAM_STRADDLE (guessed record starts, verified by the per-block kernels), for bam2db fed
    in pieces and for crb / extract; the flag changes nothing on an htslib-style file"""
    from fastf_b200 import bam2db_host as B, tags_host as T, _lib
    import bamgen
    paths, _ = synth.write_bam_set(str(tmp_path), n_reads=120000, n_cells=400, n_genes=600, seed=17, p_umi_n=0.01)
    whole = gzip.decompress(open(paths["bam"], "rb").read())
    want = oracle.bam2db(paths["bam"], paths["barcodes"], paths["features"], 0.5, 0.5, 926)
    inputs = B.Bam2dbInputs(gpu_ctx.lib, paths["barcodes"], paths["features"], 0.5, 926)
    for cut in (65280, 40001, 1500):
        p = str(tmp_path / ("cut%d.bam" % cut))
        open(p, "wb").write(bamgen.bgzf_file([whole[i:i + cut] for i in range(0, len(whole), cut)], [(1, zlib.Z_DEFAULT_STRATEGY)]))
        img = np.fromfile(p, dtype=np.uint8)
        with pytest.raises(_lib.FastfError, match="straddles"):
            B.run_device(gpu_ctx, img, inputs, 0.5, 926)
        for piece in (0, 1 << 20):
            st, out = B.run_device(gpu_ctx, img, inputs, 0.5, 926, want_rows=False, inflate_lanes=B.BAM_STRADDLE, feed_piece=piece)
            for k in ("total", "cb_valid", "sampled", "valid", "nnz"):
                assert st[k] == want[k], (cut, k)
            assert np.array_equal(out["m_gene"], want["m_gene"]) and np.array_equal(out["m_cell"], want["m_cell"]) and np.array_equal(out["m_count"], want["m_count"])
    assert T.crb(gpu_ctx, p, str(tmp_path / "crb.gz")) == oracle.crb(paths["bam"], str(tmp_path / "crb.txt"))   # the 1500-byte cut; retried by the operator
    assert gzip.open(tmp_path / "crb.gz", "rb").read() == open(tmp_path / "crb.txt", "rb").read()
    assert T.extract_bam(gpu_ctx, p, "GX", 0, str(tmp_path)) == oracle.extract(paths["bam"], "GX", 0, str(tmp_path / "o.csv"))
    assert open(tmp_path / "tag_summary.csv", "rb").read() == open(tmp_path / "o.csv", "rb").read()
    st, out = B.run_device(gpu_ctx, np.fromfile(paths["bam"], dtype=np.uint8), inputs, 0.5, 926, want_rows=False, inflate_lanes=B.BAM_STRADDLE)
    assert st["nnz"] == want["nnz"] and np.array_equal(out["m_count"], want["m_count"])


@pytest.mark.gpu
@pytest.mark.parametrize("lanes", [0, 1, 3, 4, 32, 8])
def test_inflate_random_streams(gpu_ctx, lanes):
    """seeded random BGZF images (tests/inflate_cases.py) against zlib, every kernel shape"""
    import inflate_cases
    for k, (img, want) in enumerate(inflate_cases.images(40, seed=7 + lanes)):
        assert _inflate(gpu_ctx, img, lanes) == want, k
