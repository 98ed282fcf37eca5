"""Stream set-up of the thread-per-stream inflate kernel under the SIMT emulator: the warp-parallel Huffman table build against a
serial build, and deflate blocks set up while the previous block's tokens are still in the ring (stored blocks then wait)."""
import os
import subprocess

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _emu(tmp_path, name, *flags, libs=()):
    exe = str(tmp_path / name)
    subprocess.run(["g++", "-O1", "-std=c++17", "-DFASTF_EMU", *flags, "-I" + os.path.join(ROOT, "tests", "emu"), "-o", exe,
                    os.path.join(ROOT, "tests", "emu", name + ".cpp"), *libs], check=True)
    r = subprocess.run([exe], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=600)
    assert r.returncode == 0 and r.stdout.startswith("PASS"), r.stdout[-2000:]
    return dict(kv.split("=") for kv in r.stdout.split()[1:])


def test_emu_parallel_table_build_matches_serial(tmp_path):
    """complete, over-subscribed, incomplete, single-code, empty and 15-bit codes for all three tables: same verdict, same tables"""
    f = _emu(tmp_path, "emu_build")
    assert int(f["invalid"]) > 500 and int(f["with-15-bit"]) > 100, f


def test_emu_setup_while_tokens_pending(tmp_path):
    """dynamic -> stored -> fixed -> dynamic deflate blocks in every BGZF block: byte equality with zlib's input, and the early
    set-up both ran and left stored blocks for the drained ring"""
    f = _emu(tmp_path, "emu_pending", "-DFASTF_TPS_PROF=1", libs=("-lz",))
    assert int(f["pending"]) > 0 and int(f["later"]) > 0, f
