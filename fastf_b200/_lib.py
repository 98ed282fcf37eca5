"""ctypes binding of libfastf_gpu.so (include/fastf_gpu.h).  There is no CPU implementation behind this module:
if the CUDA library is missing, or no CUDA device is present, every entry point raises."""
import ctypes as C
import os

from . import build as _build

c_u8p = C.POINTER(C.c_uint8)
c_u32p = C.POINTER(C.c_uint32)
c_u64p = C.POINTER(C.c_uint64)


class Bam2dbParams(C.Structure):
    _fields_ = [("cell_keys", C.c_char_p), ("cell_off", c_u32p), ("n_cells", C.c_uint32),
                ("gene_keys", C.c_char_p), ("gene_off", c_u32p), ("n_genes", C.c_uint32),
                ("seed", C.c_uint32), ("d0", C.c_uint64), ("keep_threshold", C.c_uint64),
                ("umi_max_bytes", C.c_uint32), ("want_rows", C.c_uint32), ("inflate_lanes", C.c_uint32),
                ("chunk_inflated_bytes", C.c_uint64), ("headerless", C.c_uint32)]


class Bam2dbResult(C.Structure):
    _fields_ = [("total", C.c_uint64), ("cb_valid", C.c_uint64), ("sampled", C.c_uint64), ("valid", C.c_uint64),
                ("nnz", C.c_uint64), ("m_gene", c_u32p), ("m_cell", c_u32p), ("m_count", c_u32p),
                ("n_rows", C.c_uint64), ("row_keys", c_u64p),
                ("bits_cell", C.c_uint32), ("bits_gene", C.c_uint32), ("bits_umi", C.c_uint32), ("umi_max_bytes", C.c_uint32),
                ("n_blocks", C.c_uint64), ("compressed_bytes", C.c_uint64), ("inflated_bytes", C.c_uint64),
                ("status", C.c_uint32), ("n_launches", C.c_uint32), ("n_chunks", C.c_uint32),
                ("ms_inflate", C.c_float), ("ms_parse", C.c_float), ("ms_gather", C.c_float), ("ms_mt", C.c_float),
                ("ms_sample", C.c_float), ("ms_sort", C.c_float), ("ms_count", C.c_float), ("ms_device_total", C.c_float), ("ms_crc", C.c_float)]


SWEEP_MAX_RATES = 32   # FASTF_SWEEP_MAX_RATES


class Bam2dbSweepResult(C.Structure):
    _fields_ = [("n_rates", C.c_uint32), ("rate", Bam2dbResult * SWEEP_MAX_RATES),
                ("n_rows", C.c_uint64), ("row_keys", c_u64p), ("row_rate", c_u8p)]


class FreqResult(C.Structure):
    _fields_ = [("n_reads", C.c_uint64), ("n_keys", C.c_uint64), ("key", c_u64p), ("count", c_u32p), ("first", c_u32p),
                ("n_exceptions", C.c_uint64), ("exc_ordinal", c_u32p), ("exc_bytes", c_u8p), ("exc_stride", C.c_uint32),
                ("n_lines", C.c_uint64), ("last_byte_is_newline", C.c_uint8),
                ("n_blocks", C.c_uint64), ("compressed_bytes", C.c_uint64), ("inflated_bytes", C.c_uint64),
                ("status", C.c_uint32), ("n_launches", C.c_uint32),
                ("ms_inflate", C.c_float), ("ms_keys", C.c_float), ("ms_sort", C.c_float), ("ms_rle", C.c_float), ("ms_device_total", C.c_float)]


class TaghistResult(C.Structure):
    _fields_ = [("n_records", C.c_uint64), ("n_hits", C.c_uint64), ("n_groups", C.c_uint64), ("mode", C.c_uint32),
                ("first", c_u32p), ("count", c_u32p), ("ivalue", C.POINTER(C.c_int32)), ("a_off", c_u64p), ("a_len", c_u32p), ("b_len", c_u32p),
                ("strings", C.POINTER(C.c_char)), ("strings_bytes", C.c_uint64),
                ("n_blocks", C.c_uint64), ("compressed_bytes", C.c_uint64), ("inflated_bytes", C.c_uint64),
                ("status", C.c_uint32), ("n_launches", C.c_uint32), ("hash_rounds", C.c_uint32),
                ("ms_inflate", C.c_float), ("ms_tags", C.c_float), ("ms_sort", C.c_float), ("ms_rle", C.c_float), ("ms_device_total", C.c_float)]


_SIGS = {
    "fastf_abi_version": (C.c_int, []),
    "fastf_build_info": (C.c_char_p, []),
    "fastf_ctx_create": (C.c_int, [C.c_int, C.POINTER(C.c_void_p)]),
    "fastf_ctx_destroy": (None, [C.c_void_p]),
    "fastf_last_error": (C.c_char_p, [C.c_void_p]),
    "fastf_host_alloc": (C.c_int, [C.c_void_p, C.c_size_t, C.POINTER(C.c_void_p)]),
    "fastf_host_free": (None, [C.c_void_p, C.c_void_p]),
    "fastf_device_alloc": (C.c_int, [C.c_void_p, C.c_size_t, C.POINTER(C.c_void_p)]),
    "fastf_device_free": (None, [C.c_void_p, C.c_void_p]),
    "fastf_memcpy_h2d": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t]),
    "fastf_memcpy_d2h": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t]),
    "fastf_synchronize": (C.c_int, [C.c_void_p]),
    "fastf_ctx_trim": (None, [C.c_void_p]),
    "fastf_launch_count": (C.c_uint32, [C.c_void_p]),
    "fastf_compute_stream": (C.c_void_p, [C.c_void_p]),
    "fastf_keep_threshold": (C.c_uint64, [C.c_float]),
    "fastf_sample_cells": (C.c_uint64, [C.c_uint64, C.c_float, C.c_uint32, c_u64p, c_u64p]),
    "fastf_bgzf_index_host": (C.c_int64, [C.c_void_p, C.c_size_t, c_u64p, c_u32p, c_u32p, C.c_uint64, C.POINTER(C.c_size_t)]),
    "fastf_cartesian_preorder": (C.c_int, [c_u32p, C.c_uint64, c_u64p]),
    "fastf_bam2db_begin": (C.c_int, [C.c_void_p, C.POINTER(Bam2dbParams), C.POINTER(C.c_void_p)]),
    "fastf_bam2db_feed": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t]),
    "fastf_bam2db_feed_device": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t, c_u64p, c_u32p, c_u32p, C.c_uint64]),
    "fastf_bam2db_counts": (C.c_int, [C.c_void_p, c_u64p, c_u64p]),
    "fastf_bam2db_sample": (C.c_int, [C.c_void_p, C.c_uint64]),
    "fastf_bam2db_kept_device": (C.c_int, [C.c_void_p, C.POINTER(C.c_void_p), c_u64p]),
    "fastf_bam2db_sample_counts": (C.c_int, [C.c_void_p, c_u64p, c_u64p]),
    "fastf_bam2db_key_layout": (C.c_int, [C.c_void_p, c_u32p, c_u32p, c_u32p]),
    "fastf_bam2db_finish": (C.c_int, [C.c_void_p, C.POINTER(Bam2dbResult)]),
    "fastf_bam2db_finish_sweep": (C.c_int, [C.c_void_p, C.c_uint32, c_u64p, C.POINTER(Bam2dbSweepResult)]),
    "fastf_bam2db_sweep_result_free": (None, [C.POINTER(Bam2dbSweepResult)]),
    "fastf_bam2db_sample_sweep": (C.c_int, [C.c_void_p, C.c_uint64, C.c_uint32, c_u64p, c_u64p, c_u64p]),
    "fastf_bam2db_kept_sweep_device": (C.c_int, [C.c_void_p, C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), c_u64p]),
    "fastf_bam2db_stats": (C.c_int, [C.c_void_p, C.POINTER(Bam2dbResult)]),
    "fastf_bam2db_job_free": (None, [C.c_void_p]),
    "fastf_bam2db_result_free": (None, [C.POINTER(Bam2dbResult)]),
    "fastf_bam2db_run_sharded": (C.c_int, [C.c_int, C.POINTER(C.c_int), C.POINTER(Bam2dbParams), C.c_void_p, C.c_size_t, C.POINTER(Bam2dbResult)]),
    "fastf_bam2db_run_sharded_sweep": (C.c_int, [C.c_int, C.POINTER(C.c_int), C.POINTER(Bam2dbParams), C.c_void_p, C.c_size_t, C.c_uint32, c_u64p, C.POINTER(Bam2dbSweepResult)]),
    "fastf_sharded_last_error": (C.c_char_p, []),
    "fastf_sharded_exchanged": (C.c_uint64, []),
    "fastf_sort_u64_device": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint32]),
    "fastf_dedup_count_device": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint32, C.c_uint32, c_u64p, C.POINTER(c_u32p), C.POINTER(c_u32p), C.POINTER(c_u32p)]),
    "fastf_dedup_count_device_out": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint32, C.c_uint32, c_u64p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "fastf_unique_partition_device": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, C.c_void_p, c_u64p]),
    "fastf_unique_partition_rates_device": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p, c_u64p]),
    "fastf_sweep_count_device": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, c_u64p, C.POINTER(c_u32p), C.POINTER(c_u32p),
                                           C.POINTER(c_u32p)]),
    "fastf_free": (None, [C.c_void_p]),
    "fastf_inflate_host": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t, C.c_int, C.POINTER(C.c_void_p), C.POINTER(C.c_size_t), C.POINTER(C.c_float)]),
    "fastf_mt19937_host": (C.c_int, [C.c_void_p, C.c_uint32, C.c_uint64, c_u32p]),
    "fastf_mt19937_host_from": (C.c_int, [C.c_void_p, C.c_uint32, C.c_uint64, C.c_uint64, c_u32p]),
    "fastf_mt19937_keepbits_host": (C.c_int, [C.c_void_p, C.c_uint32, C.c_uint64, C.c_uint64, c_u32p]),
    "fastf_sort_u64_host": (C.c_int, [C.c_void_p, c_u64p, c_u32p, C.c_uint64, C.c_uint32]),
    "fastf_unique_counts_host": (C.c_int, [C.c_void_p, c_u64p, C.c_uint64, C.c_uint32, C.POINTER(c_u64p), C.POINTER(c_u32p), C.POINTER(C.c_uint64)]),
    "fastf_freq_gpu": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t, C.c_uint32, C.c_uint32, C.POINTER(FreqResult)]),
    "fastf_freq_gpu_device": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t, c_u64p, c_u32p, c_u32p, C.c_uint64, C.c_uint32, C.c_uint32, C.POINTER(FreqResult)]),
    "fastf_freq_result_free": (None, [C.POINTER(FreqResult)]),
    "fastf_taghist_gpu": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t, C.c_char_p, C.c_uint32, C.c_char_p, C.c_uint32, C.POINTER(TaghistResult)]),
    "fastf_taghist_result_free": (None, [C.POINTER(TaghistResult)]),
    "fastf_taghist_test_hooks": (None, [C.c_void_p, C.c_uint64, C.c_uint64]),
}
EXPORTS = sorted(_SIGS)

_lib = None


def library_path():
    return os.environ.get("FASTF_GPU_LIB") or _build.LIB


def load():
    """Loads libfastf_gpu.so; raises (never falls back) when it is missing."""
    global _lib
    if _lib is not None:
        return _lib
    path = library_path()
    if not os.path.exists(path):
        raise RuntimeError(f"{path} is missing: run `python -m fastf_b200.build` (nvcc, sm_100a). There is no CPU fallback.")

    def bind(p):
        lib = C.CDLL(p)
        for name, (res, args) in _SIGS.items():
            fn = getattr(lib, name)   # AttributeError if the library does not export a declared symbol
            fn.restype = res
            fn.argtypes = args
        return lib, dict(kv.split("=", 1) for kv in lib.fastf_build_info().decode().split())

    lib, info = bind(path)
    # A prebuilt binary that does not match the sources next to it is rebuilt (one rank at a time) or refused -- never used silently.
    # Variant builds named by FASTF_GPU_LIB opt out.
    if not os.environ.get("FASTF_GPU_LIB") and info.get("src") not in ("unknown", _build.source_hash()):
        import fcntl
        os.makedirs(_build.BUILD, exist_ok=True)
        with open(os.path.join(_build.BUILD, ".build.lock"), "w") as lock:
            fcntl.flock(lock, fcntl.LOCK_EX)
            try:
                # another rank may have rebuilt it while we waited; dlopen caches by path, so the fresh file is loaded under a new name
                fresh = os.path.join(_build.BUILD, "libfastf_gpu.%s.so" % _build.source_hash())
                if not os.path.exists(fresh):
                    _build.build_cuda(force=True)
                    import shutil
                    shutil.copyfile(path, fresh)
                lib, info = bind(fresh)
            finally:
                fcntl.flock(lock, fcntl.LOCK_UN)
        if info.get("src") != _build.source_hash():
            raise RuntimeError(f"{path} was built from other sources (src={info.get('src')}, tree={_build.source_hash()}) and could not be rebuilt: run `python -m fastf_b200.build`")
    _lib = lib
    return lib


def build_info():
    """dict of the loaded library's build parameters (streams per SM, kernel shape, source hash)"""
    return dict(kv.split("=", 1) for kv in load().fastf_build_info().decode().split())


class FastfError(RuntimeError):
    pass


class Context:
    """One CUDA device + its streams.  Creation fails without a GPU."""

    def __init__(self, device=0):
        self.lib = load()
        h = C.c_void_p()
        if self.lib.fastf_ctx_create(device, C.byref(h)) != 0:
            raise FastfError(self.lib.fastf_last_error(None).decode())
        self.h = h
        self.device = device

    def check(self, rc, what=""):
        if rc != 0:
            raise FastfError(f"{what}: {self.lib.fastf_last_error(self.h).decode()}")

    def close(self):
        if self.h:
            self.lib.fastf_ctx_destroy(self.h)
            self.h = None

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    @property
    def launches(self):
        return int(self.lib.fastf_launch_count(self.h))
