#!/usr/bin/env python
"""A/B of inflate kernel builds: kernel ms (CUDA events inside fastf_inflate_host) and GB/s algorithmic on an image of exactly
ROUNDS x n_sm x streams-per-SM BGZF blocks of the synthetic 10x BAM (the persistent kernel keeps that many blocks in flight, so only
such a launch has no half-empty last round: a fixed image would favour whatever stream count divides it).  The library's CRC-32 pass
checks every inflated block against its BGZF trailer.

    python scripts/inflate_ab.py [--lanes L] [--reps R] [--rounds K]      # library = $FASTF_GPU_LIB or the in-tree build
"""
import argparse, ctypes as C, os, sys
import numpy as np
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))

ap = argparse.ArgumentParser()
ap.add_argument("--reads", type=int, default=12_300_000)   # > 2 x 148 x 256 BGZF blocks
ap.add_argument("--lanes", type=int, default=0)
ap.add_argument("--reps", type=int, default=3)
ap.add_argument("--rounds", type=int, default=2)
ap.add_argument("--cache", default="/tmp/fastf_ab_bam2")
a = ap.parse_args()

import synth_binding
from fastf_b200 import _lib
lib = _lib.load()
if os.path.exists(a.cache + ".npy"):
    bam, starts = np.load(a.cache + ".npy"), np.load(a.cache + "_starts.npy")
else:
    S = synth_binding.load()
    raw, st = S.bam(S.params(n_reads=a.reads, n_cells=10000, n_genes=36000, seed=11))
    bam = np.frombuffer(raw, dtype=np.uint8).copy()
    cap = int(st.n_blocks) + 8
    io, il, isz = np.zeros(cap, np.uint64), np.zeros(cap, np.uint32), np.zeros(cap, np.uint32)
    used = C.c_size_t()
    nb = lib.fastf_bgzf_index_host(C.c_void_p(bam.ctypes.data), bam.size, io.ctypes.data_as(_lib.c_u64p), il.ctypes.data_as(_lib.c_u32p), isz.ctypes.data_as(_lib.c_u32p), cap, C.byref(used))
    starts = np.concatenate([[0], (io[:nb] + il[:nb] + 8).astype(np.uint64)])   # block i starts where block i-1's trailer ends
    np.save(a.cache + ".npy", bam); np.save(a.cache + "_starts.npy", starts)
info = _lib.build_info()
shape = {0: None, 1: (8, 16), 2: (16, 24), 3: (16, 16), 4: (32, 28)}.get(a.lanes)
ctx = _lib.Context(0)
nblocks = min(a.rounds * 148 * int(info["streams"]), len(starts) - 2)
img = bam[: int(starts[nblocks])]
lanes = a.lanes | (0x200 if os.environ.get("FASTF_AB_NOCRC") else 0)
best = None
for r in range(a.reps):
    out, n, ms = C.c_void_p(), C.c_size_t(), C.c_float()
    rc = ctx.lib.fastf_inflate_host(ctx.h, C.c_void_p(img.ctypes.data), img.size, lanes, C.byref(out), C.byref(n), C.byref(ms))
    if rc:
        print("FAILED", ctx.lib.fastf_last_error(ctx.h).decode()); sys.exit(1)
    ctx.lib.fastf_free(out)
    best = ms.value if best is None else min(best, ms.value)
    if hasattr(ctx.lib, "fastf_debug_tps_prof") and r == a.reps - 1:
        # -DFASTF_TPS_PROF=1 build: role counters of the last launch (the ones before are discarded by the reset)
        pr = (C.c_ulonglong * 32)()   # FASTF_TPS_PROF_N
        ctx.lib.fastf_debug_tps_prof(pr, 1)
        (d, full, wait, npass, nempty, ccopy, csetup, cempty, nb_, ntok, ctot, nlong, nwalk, waitn, cwb, cwn, cdec, nbgzf, nhdr, cbuild,
         hob, nhob, hon, nhon, nearly, nlater) = [int(pr[i]) for i in range(26)]
        rounds = max(d + full + wait, 1)
        print("prof: decoder lane-rounds %d decoded, %d ring-full (%.1f%%), %d waiting for set-up (%.1f%%: BUILD %.1f%%, NEXT %.1f%%) | service passes %d, empty %.1f%%, batches %d (%.1f tokens), cycles: copy %.1f%% set-up %.1f%% empty passes %.1f%% of %.3g; per batch %.0f cycles | codes longer than the table %d, walks %d"
              % (d, full, 100.0 * full / rounds, wait, 100.0 * wait / rounds, 100.0 * (wait - waitn) / rounds, 100.0 * waitn / rounds, npass, 100.0 * nempty / max(npass, 1), nb_, ntok / max(nb_, 1),
                 100.0 * ccopy / max(ctot, 1), 100.0 * csetup / max(ctot, 1), 100.0 * cempty / max(ctot, 1), ctot, ccopy / max(nb_, 1), nlong, nwalk))
        print("prof-time: decoder cycles waiting for set-up %.1f%% (BUILD %.1f%%, NEXT %.1f%%) of %.3g | %d BGZF blocks, %.2f deflate blocks each | set-up cycles: headers + code lengths %.1f%%, table builds %.1f%% of %.3g (%.0f per deflate block) | hand-over to set-up start: BUILD %.0f cycles (%d), NEXT %.0f cycles (%d) | set-ups with tokens pending %d, %d of them left for later"
              % (100.0 * (cwb + cwn) / max(cdec, 1), 100.0 * cwb / max(cdec, 1), 100.0 * cwn / max(cdec, 1), cdec, nbgzf, nhdr / max(nbgzf, 1),
                 100.0 * (csetup - cbuild) / max(csetup, 1), 100.0 * cbuild / max(csetup, 1), csetup, csetup / max(nhdr, 1), hob / max(nhob, 1), nhob, hon / max(nhon, 1), nhon, nearly, nlater))
    elif hasattr(ctx.lib, "fastf_debug_tps_prof"):
        ctx.lib.fastf_debug_tps_prof(None, 1)
print("lib=%s %s lanes=%d blocks=%d ms=%.2f alg_GBps=%.1f out_GBps=%.1f %s" % (os.path.basename(os.environ.get("FASTF_GPU_LIB", "default")), " ".join(f"{k}={v}" for k, v in info.items() if k != "src"),
      a.lanes, nblocks, best, (img.size + n.value) / best / 1e6, n.value / best / 1e6, "nocrc" if os.environ.get("FASTF_AB_NOCRC") else "crc32-verified"))
