"""CPU tests of the drop-in boundary: the C-ABI library loads, exports every symbol include/fastf_gpu.h declares, refuses to
run without a GPU, and its host-side helpers (sampling contract, BGZF indexer, BST pre-order) agree with the oracle."""
import ctypes as C
import os
import re

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib():
    from fastf_b200 import _lib, build
    build.build_cuda()   # nvcc cross-compiles sm_100a without a GPU
    return _lib.load()


def test_header_symbols_exported(lib):
    from fastf_b200 import _lib
    hdr = open(os.path.join(ROOT, "include", "fastf_gpu.h")).read()
    declared = sorted(set(re.findall(r"\b(fastf_[a-z0-9_]+)\s*\(", hdr)))
    assert len(declared) >= 35
    for name in declared:
        assert hasattr(lib, name), "libfastf_gpu.so does not export " + name
    assert sorted(_lib.EXPORTS) == declared, "ctypes binding and header disagree"
    assert lib.fastf_abi_version() == 1


def test_no_cpu_fallback(lib, tmp_path):
    """without a visible CUDA device (hidden by CUDA_VISIBLE_DEVICES on a machine that has one) every entry point refuses"""
    import subprocess
    import sys
    code = ("import sys; sys.path.insert(0, %r)\n"
            "import fastf_b200\n"
            "from fastf_b200 import _lib\n"
            "try:\n"
            "    _lib.Context(0)\n"
            "    raise SystemExit('a context was created without a device')\n"
            "except _lib.FastfError as e:\n"
            "    assert 'no CUDA device' in str(e), e\n"
            "assert fastf_b200.freq(%r, %r, 16, 12) == 1\n"
            "print('OK refused')\n") % (ROOT, os.path.join(ROOT, "tests", "golden", "freq", "synth.fastq.gz"), str(tmp_path))
    r = subprocess.run([sys.executable, "-c", code], env=dict(os.environ, CUDA_VISIBLE_DEVICES=""), stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=300)
    assert r.returncode == 0 and "OK refused" in r.stdout, r.stdout[-2000:]
    assert not os.path.exists(tmp_path / "whitelist.txt")


def test_keep_threshold_matches_reference_rule(lib, oracle):
    table = {0.1: 429496736, 0.2: 858993472, 0.3: 1288490240, 0.5: 2147483648, 0.9: 3865470464, 1.0: 4294967295}   # SURVEY.md Appendix A
    for r, T in table.items():
        assert lib.fastf_keep_threshold(C.c_float(r)) == T
    rng = np.random.default_rng(1)
    for r in list(rng.random(40).astype(np.float32)) + [0.0, 1.0, 1.5, -0.5, 1e-9, 0.99999994, float("nan"), float("inf"), -0.0]:   # NaN: `x >= NaN` is false, the reference drops nothing
        T = lib.fastf_keep_threshold(C.c_float(float(r)))
        for u in {0, 1, 0xFFFFFFFF, max(T - 1, 0), min(T, 0xFFFFFFFF), min(T + 1, 0xFFFFFFFF)}:
            assert oracle.depth_keep(u, float(r)) == (u < T), (r, u, T)


@pytest.mark.parametrize("n,rate,seed", [(1000, 0.5, 926), (1000, 1.0, 926), (10, 0.7, 1), (50000, 0.2, 926), (7, 0.0, 3), (1, 0.99, 5), (12345, 0.333, 99)])
def test_sample_cells_matches_oracle(lib, oracle, n, rate, seed):
    from fastf_b200 import _lib
    out = np.zeros(n, dtype=np.uint64)
    d0 = C.c_uint64()
    ns = lib.fastf_sample_cells(n, C.c_float(rate), seed, out.ctypes.data_as(_lib.c_u64p), C.byref(d0))
    ons, oidx, od0 = oracle.sample_cells(n, rate, seed)
    assert ns == ons and d0.value == od0 and np.array_equal(out[:ns], oidx)


def test_sample_cells_rejects_oversampling(lib):
    from fastf_b200 import _lib
    out = np.zeros(10, dtype=np.uint64)
    assert lib.fastf_sample_cells(10, C.c_float(1.5), 1, out.ctypes.data_as(_lib.c_u64p), None) == 2**64 - 1


def test_bgzf_index_host(lib):
    import bamgen
    from fastf_b200 import _lib
    payloads = [b"a" * 100, b"", bytes(range(256)) * 200, b"xyz"]
    img = bamgen.bgzf_file(payloads)
    buf = np.frombuffer(img, dtype=np.uint8)
    io, il, isz = np.zeros(16, np.uint64), np.zeros(16, np.uint32), np.zeros(16, np.uint32)
    used = C.c_size_t()
    nb = lib.fastf_bgzf_index_host(C.c_void_p(buf.ctypes.data), buf.size, io.ctypes.data_as(_lib.c_u64p), il.ctypes.data_as(_lib.c_u32p), isz.ctypes.data_as(_lib.c_u32p), 16, C.byref(used))
    assert nb == 5 and used.value == len(img)
    assert isz[:5].tolist() == [100, 0, 51200, 3, 0]
    import zlib
    for k in range(5):
        raw = zlib.decompress(img[int(io[k]):int(io[k]) + int(il[k])], -15)
        assert raw == (payloads + [b""])[k]
    # a cut inside the third block: two whole blocks, NEED_MORE is not an error
    cut = int(io[2]) + 10
    nb = lib.fastf_bgzf_index_host(C.c_void_p(buf.ctypes.data), cut, io.ctypes.data_as(_lib.c_u64p), il.ctypes.data_as(_lib.c_u32p), isz.ctypes.data_as(_lib.c_u32p), 16, C.byref(used))
    assert nb == 2 and used.value == int(io[2]) - 18
    bad = np.frombuffer(b"\x1f\x8b\x08\x00" + b"\0" * 40, dtype=np.uint8)   # gzip without the BGZF extra field
    assert lib.fastf_bgzf_index_host(C.c_void_p(bad.ctypes.data), bad.size, io.ctypes.data_as(_lib.c_u64p), il.ctypes.data_as(_lib.c_u32p), isz.ctypes.data_as(_lib.c_u32p), 16, C.byref(used)) == -1


def _bst_preorder(first):
    """the reference's insert_tree / print_tree order, literally: insert keys (identified by rank) in order of first occurrence"""
    import sys
    n = len(first)
    order_in = np.argsort(first, kind="stable")
    left, right = [-1] * n, [-1] * n
    root = -1
    for k in order_in.tolist():
        if root < 0:
            root = k
            continue
        cur = root
        while True:
            if k < cur:
                if left[cur] < 0:
                    left[cur] = k
                    break
                cur = left[cur]
            else:
                if right[cur] < 0:
                    right[cur] = k
                    break
                cur = right[cur]
    out, stack = [], [root] if root >= 0 else []
    while stack:
        v = stack.pop()
        out.append(v)
        if right[v] >= 0:
            stack.append(right[v])
        if left[v] >= 0:
            stack.append(left[v])
    return out


@pytest.mark.parametrize("n,seed", [(1, 0), (2, 1), (17, 2), (1000, 3), (5000, 4)])
def test_cartesian_preorder_equals_bst_preorder(lib, n, seed):
    from fastf_b200 import _lib
    rng = np.random.default_rng(seed)
    first = rng.permutation(n * 3)[:n].astype(np.uint32)
    order = np.zeros(n, dtype=np.uint64)
    assert lib.fastf_cartesian_preorder(first.ctypes.data_as(_lib.c_u32p), n, order.ctypes.data_as(_lib.c_u64p)) == 0
    assert order.tolist() == _bst_preorder(first)
    # sorted / reverse-sorted insertion orders (degenerate trees, deep recursion in the reference)
    for f in (np.arange(n, dtype=np.uint32), np.arange(n, dtype=np.uint32)[::-1].copy()):
        assert lib.fastf_cartesian_preorder(f.ctypes.data_as(_lib.c_u32p), n, order.ctypes.data_as(_lib.c_u64p)) == 0
        assert order.tolist() == _bst_preorder(f)


def test_host_readers_mirror_reference_quirks(tmp_path, lib):
    """gzgets 1023-byte chunks, strcspn cut at \\n\\r\\t, strtok skipping empty fields, duplicate handling"""
    import gzip
    from fastf_b200 import bam2db_host as B
    assert B.gzgets_lines(b"ab\ncd") == [b"ab\n", b"cd"]
    assert [len(x) for x in B.gzgets_lines(b"x" * 2500 + b"\n")] == [1023, 1023, 455]
    bc = tmp_path / "b.tsv"
    bc.write_bytes(b"AAAA-1\r\nCCCC-1\textra\nAAAA-1\nGGGG-1\n")
    ft = tmp_path / "f.tsv.gz"
    with gzip.open(ft, "wb") as f:
        f.write(b"G1\tn1\tGene Expression\nG2\t\tn2\tGene Expression\tmore\nG1\tdup\tx\n")
    inp = B.Bam2dbInputs(lib, str(bc), str(ft), 1.0, 926)
    assert inp.n_cells == 4 and inp.d0 == 0
    assert inp.cells == [b"AAAA-1", b"CCCC-1"] and inp.duplicate_barcodes     # the duplicate stalls the index: GGGG-1 never matches
    assert [f[:4] for f in inp.features] == [(b"G1", b"G1", b"n1", b"Gene Expression"), (b"G2", b"G2", b"n2", b"Gene Expression")]
    assert inp.duplicate_features
