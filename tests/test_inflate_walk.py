"""Codes longer than the inflate kernel's primary table whose second-level tables do not fit: the canonical walk, with its range
limits and index offsets in the stream's global scratch (tests/walk_cases.py builds the image)."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import walk_cases

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_walk_image_overflows_the_subtables():
    assert walk_cases.subtable_entries(walk_cases.lit_lengths()) > walk_cases.SUB_CAPACITY
    img, want = walk_cases.image()
    assert len(want) > 40000 and len(img) < len(want) * 2


def test_emu_walk_limits_from_global_scratch(tmp_path):
    """the emulator build with role counters: byte equality with zlib, and the walk counter fired"""
    exe = str(tmp_path / "emu_walk")
    subprocess.run(["g++", "-O1", "-std=c++17", "-DFASTF_EMU", "-DFASTF_TPS_PROF=1", "-I" + os.path.join(ROOT, "tests", "emu"), "-o", exe,
                    os.path.join(ROOT, "tests", "emu", "emu_walk.cpp"), "-lz"], check=True)
    img, want = walk_cases.image()
    (tmp_path / "walk.bgzf").write_bytes(img)
    r = subprocess.run([exe, str(tmp_path / "walk.bgzf")], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=600)
    assert r.returncode == 0 and r.stdout.startswith("PASS"), r.stdout[-2000:]
    fields = dict(kv.split("=") for kv in r.stdout.split()[1:])
    assert int(fields["bytes"]) == len(want)
    # 80 % of the walk blocks' literals have 9-bit codes; each round of a decoder lane starts with at most one of them
    assert int(fields["walks"]) > 1000, r.stdout
    assert int(fields["walks"]) <= int(fields["long"])


@pytest.mark.gpu
@pytest.mark.parametrize("lanes", [0, 32])   # 0 = thread-per-stream kernel, 32 = lock-step kernel
def test_gpu_walk_limits_from_global_scratch(gpu_ctx, lanes):
    img, want = walk_cases.image()
    buf = np.frombuffer(img, dtype=np.uint8)
    out, n, ms = C.c_void_p(), C.c_size_t(), C.c_float()
    rc = gpu_ctx.lib.fastf_inflate_host(gpu_ctx.h, C.c_void_p(buf.ctypes.data), buf.size, lanes, C.byref(out), C.byref(n), C.byref(ms))
    assert rc == 0, gpu_ctx.lib.fastf_last_error(gpu_ctx.h)
    got = C.string_at(out, n.value)
    gpu_ctx.lib.fastf_free(out)
    assert got == want
