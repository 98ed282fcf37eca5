"""Host side of `fastF bam2db`, mirroring the reference operator

    int bam2db(char *bam_file, char *db_file, char *path_out, char *barcodes_file, char *features_file,
               float rate_cell, float rate_depth, unsigned int seed)          (reference src/bam2db_ds.h:62-70)

Same arguments, same return convention (0 ok / 1 failure + message on stderr), same stdout/stderr lines and the
same output files.  The per-read hot loop (reference src/bam2db_ds.c:360-438) and the sqlite aggregation
(src/bam2db_ds.c:480-483) run on the GPU through libfastf_gpu.so; this module only reads the two small list files,
draws the cell sample, and writes sqlite + .gz files from the device result.  No CPU implementation of the hot
path exists here."""
import ctypes as C
import gzip
import os
import sqlite3
import sys

import numpy as np

from . import _lib

_umi_copies_flag = 0   # reference global `_umi_copies_flag` (src/bam2db_ds.c:3), set by `-u`


def gzgets_lines(data, buflen=1024):
    """Lines as successive gzgets(fp, buf, buflen) calls return them (at most buflen-1 bytes each)."""
    out = []
    pos, n, lim = 0, len(data), buflen - 1
    while pos < n:
        nl = data.find(b"\n", pos, pos + lim)
        end = nl + 1 if nl >= 0 else min(pos + lim, n)
        out.append(data[pos:end])
        pos = end
    return out


def _read_maybe_gz(path):
    with open(path, "rb") as f:
        raw = f.read()
    return gzip.decompress(raw) if raw[:2] == b"\x1f\x8b" else raw   # gzopen reads plain files transparently too


def _cut(s, delims=b"\n\r\t"):
    for i, ch in enumerate(s):
        if ch in delims:
            return s[:i]
    return s


def _strtok3(line):
    """First three strtok(.., "\\t") tokens of a feature line + the hash key the reference uses (buffer up to its first NUL)."""
    line = line.split(b"\0", 1)[0]
    toks, i, n, key_end = [], 0, len(line), None
    while len(toks) < 3:
        while i < n and line[i] == 9:
            i += 1
        if i >= n:
            return None, None
        j = i
        while j < n and line[j] != 9:
            j += 1
        toks.append(line[i:j])
        if key_end is None:
            key_end = j
        i = j + 1
    return toks, line[:key_end]


class Bam2dbInputs:
    """Barcode sample + feature table exactly as the reference builds them (src/bam2db_ds.c:229-337)."""

    def __init__(self, lib, barcodes_file, features_file, rate_cell, seed):
        lines = gzgets_lines(_read_maybe_gz(barcodes_file))
        self.n_cells = len(lines)
        samp = np.zeros(max(self.n_cells, 1), dtype=np.uint64)
        d0 = C.c_uint64(0)
        ns = lib.fastf_sample_cells(self.n_cells, C.c_float(rate_cell), seed, samp.ctypes.data_as(_lib.c_u64p), C.byref(d0))
        if ns == 2**64 - 1:
            raise ValueError("Sample size must be smaller than population size when sampling without replacement.")
        self.n_cells_sampled = int(ns)
        self.d0 = int(d0.value)
        self.duplicate_barcodes = False
        cells, seen = [], set()
        cell_index = 1
        for nth, ln in enumerate(lines):
            if cell_index > ns:
                break
            if nth != int(samp[cell_index - 1]):
                continue
            bc = _cut(ln).split(b"\0", 1)[0]
            if bc not in seen:
                seen.add(bc)
                cells.append(bc)
                cell_index += 1
            else:
                self.duplicate_barcodes = True   # index not advanced: no later line can match (src/bam2db_ds.c:260,281-285)
        self.cells = cells
        feats, fseen = [], {}
        self.duplicate_features = False
        for ln in gzgets_lines(_read_maybe_gz(features_file)):
            toks, key = _strtok3(ln)
            if toks is None:
                raise ValueError("feature line with fewer than three tab-separated fields (the reference dereferences NULL here)")
            toks[2] = _cut(toks[2])
            if key not in fseen:
                fseen[key] = len(feats) + 1
                feats.append((key, toks[0], toks[1], toks[2]))
            else:
                self.duplicate_features = True
        self.features = feats


def _pack_table(keys):
    off = np.zeros(len(keys) + 1, dtype=np.uint32)
    if keys:
        off[1:] = np.cumsum([len(k) for k in keys], dtype=np.uint64).astype(np.uint32)
    blob = b"".join(keys) + b"\0"
    return blob, off


def decode_rows(row_keys, bits_gene, bits_umi, umi_max_bytes):
    """packed rows -> (cell, gene, blob_len or -1 for NULL, content as left-aligned integer of umi_max_bytes bytes)"""
    k = np.asarray(row_keys, dtype=np.uint64)
    code = k & np.uint64((1 << bits_umi) - 1)
    gene = ((k >> np.uint64(bits_umi)) & np.uint64((1 << bits_gene) - 1)).astype(np.uint32)
    cell = (k >> np.uint64(bits_umi + bits_gene)).astype(np.uint32)
    nn = (code >> np.uint64(bits_umi - 1)) & np.uint64(1)
    nbytes = (code & np.uint64(7)).astype(np.int64)
    content = (code >> np.uint64(3)) & np.uint64((1 << (8 * umi_max_bytes)) - 1)
    nbytes = np.where(nn == 1, nbytes, -1)
    return cell, gene, nbytes, content


BAM_STRADDLE = 0x400   # FASTF_BAM_STRADDLE (include/fastf_gpu.h)


def make_params(lib, inputs, rate_depth, seed, want_rows=True, inflate_lanes=0, chunk_inflated_bytes=0, umi_max_bytes=0, headerless=False):
    """fastf_bam2db_params for these inputs; the second value keeps the packed tables alive"""
    ckeys, coff = _pack_table(inputs.cells)
    gkeys, goff = _pack_table([f[0] for f in inputs.features])
    p = _lib.Bam2dbParams()
    p.cell_keys = ckeys
    p.cell_off = coff.ctypes.data_as(_lib.c_u32p)
    p.n_cells = len(inputs.cells)
    p.gene_keys = gkeys
    p.gene_off = goff.ctypes.data_as(_lib.c_u32p)
    p.n_genes = len(inputs.features)
    p.seed = seed
    p.d0 = inputs.d0
    p.keep_threshold = lib.fastf_keep_threshold(C.c_float(rate_depth))
    p.umi_max_bytes = umi_max_bytes
    p.want_rows = 1 if want_rows else 0
    p.inflate_lanes = inflate_lanes
    p.chunk_inflated_bytes = chunk_inflated_bytes
    p.headerless = 1 if headerless else 0
    return p, (ckeys, coff, gkeys, goff)


def _result_to_python(lib, res, want_rows):
    z32 = np.zeros(0, np.uint32)
    out = {
        "m_gene": np.ctypeslib.as_array(res.m_gene, (res.nnz,)).copy() if res.nnz else z32,
        "m_cell": np.ctypeslib.as_array(res.m_cell, (res.nnz,)).copy() if res.nnz else z32,
        "m_count": np.ctypeslib.as_array(res.m_count, (res.nnz,)).copy() if res.nnz else z32,
        "row_keys": np.ctypeslib.as_array(res.row_keys, (res.n_rows,)).copy() if (want_rows and res.n_rows) else np.zeros(0, np.uint64),
    }
    stats = {f: getattr(res, f) for f, _ in _lib.Bam2dbResult._fields_ if not f.startswith("m_") and f != "row_keys"}
    lib.fastf_bam2db_result_free(C.byref(res))
    return stats, out


def run_sharded(lib, bam_bytes, inputs, rate_depth, seed, n_devices, want_rows=True, devices=None, **kw):
    """bam2db over n_devices GPUs of this node in ONE process: the C driver fastf_bam2db_run_sharded (contexts, feeder threads and the
    NCCL all-to-all live in the library).  Returns (stats, arrays) like run_device; stats gains "exchanged_keys"."""
    p, keep = make_params(lib, inputs, rate_depth, seed, want_rows, **kw)
    buf = np.frombuffer(bam_bytes, dtype=np.uint8)
    res = _lib.Bam2dbResult()
    devs = (C.c_int * n_devices)(*devices) if devices else None
    if lib.fastf_bam2db_run_sharded(n_devices, devs, C.byref(p), C.c_void_p(buf.ctypes.data), buf.size, C.byref(res)) != 0:
        raise _lib.FastfError("bam2db_run_sharded: " + lib.fastf_sharded_last_error().decode())
    stats, out = _result_to_python(lib, res, want_rows)
    stats["exchanged_keys"] = int(lib.fastf_sharded_exchanged())
    del keep
    return stats, out


def _sweep_to_python(res, thr, want_rows):
    """[(stats, arrays)] per threshold (caller order) out of a filled Bam2dbSweepResult; rate i's rows are those whose rate's threshold is
    <= thr[i].  The caller frees res."""
    rows = np.ctypeslib.as_array(res.row_keys, (res.n_rows,)).copy() if (want_rows and res.n_rows) else np.zeros(0, np.uint64)
    row_rate = np.ctypeslib.as_array(res.row_rate, (res.n_rows,)).copy() if (want_rows and res.n_rows) else np.zeros(0, np.uint8)
    out = []
    for i in range(len(thr)):
        r = res.rate[i]
        z32 = np.zeros(0, np.uint32)
        arrays = {
            "m_gene": np.ctypeslib.as_array(r.m_gene, (r.nnz,)).copy() if r.nnz else z32,
            "m_cell": np.ctypeslib.as_array(r.m_cell, (r.nnz,)).copy() if r.nnz else z32,
            "m_count": np.ctypeslib.as_array(r.m_count, (r.nnz,)).copy() if r.nnz else z32,
            "row_keys": rows[thr[row_rate] <= thr[i]],
        }
        stats = {f: getattr(r, f) for f, _ in _lib.Bam2dbResult._fields_ if not f.startswith("m_") and f != "row_keys"}
        stats["n_rows"] = len(arrays["row_keys"])
        out.append((stats, arrays))
    return out


def _thresholds(lib, rates):
    return np.array([lib.fastf_keep_threshold(C.c_float(r)) for r in rates], dtype=np.uint64)


def run_sharded_sweep(lib, bam_bytes, inputs, rates, seed, n_devices, want_rows=True, devices=None, **kw):
    """The depth sweep over n_devices GPUs of this node in ONE process (fastf_bam2db_run_sharded_sweep).  Returns what
    Bam2dbJob.finish_sweep returns for one job over the whole file: [(stats, arrays)] in the order of `rates`; every stats gains
    "exchanged_keys"."""
    p, keep = make_params(lib, inputs, 0.0, seed, want_rows, **kw)
    thr = _thresholds(lib, rates)
    buf = np.frombuffer(bam_bytes, dtype=np.uint8)
    res = _lib.Bam2dbSweepResult()
    devs = (C.c_int * n_devices)(*devices) if devices else None
    try:
        if lib.fastf_bam2db_run_sharded_sweep(n_devices, devs, C.byref(p), C.c_void_p(buf.ctypes.data), buf.size, len(thr), thr.ctypes.data_as(_lib.c_u64p), C.byref(res)) != 0:
            raise _lib.FastfError("bam2db_run_sharded_sweep: " + lib.fastf_sharded_last_error().decode())
        out = _sweep_to_python(res, thr, want_rows)
    finally:
        lib.fastf_bam2db_sweep_result_free(C.byref(res))
    x = int(lib.fastf_sharded_exchanged())
    for stats, _ in out:
        stats["exchanged_keys"] = x
    del keep
    return out


class Bam2dbJob:
    """One streaming bam2db job on one GPU: begin -> feed*/feed_device* -> (counts -> sample(base)) -> finish."""

    def __init__(self, ctx, inputs, rate_depth, seed, want_rows=True, inflate_lanes=0, chunk_inflated_bytes=0, umi_max_bytes=0, headerless=False):
        self.ctx, self.lib = ctx, ctx.lib
        p, self._keep = make_params(self.lib, inputs, rate_depth, seed, want_rows, inflate_lanes, chunk_inflated_bytes, umi_max_bytes, headerless)
        self.want_rows = want_rows
        self.job = C.c_void_p()
        ctx.check(self.lib.fastf_bam2db_begin(ctx.h, C.byref(p), C.byref(self.job)), "bam2db_begin")

    def feed(self, host_ptr, nbytes):
        self.ctx.check(self.lib.fastf_bam2db_feed(self.job, C.c_void_p(host_ptr), nbytes), "bam2db_feed")

    def feed_device(self, dev_ptr, nbytes, in_off, in_len, isize):
        self.ctx.check(self.lib.fastf_bam2db_feed_device(self.job, C.c_void_p(dev_ptr), nbytes, in_off.ctypes.data_as(_lib.c_u64p), in_len.ctypes.data_as(_lib.c_u32p),
                                                         isize.ctypes.data_as(_lib.c_u32p), len(in_off)), "bam2db_feed_device")

    def counts(self):
        a, b = C.c_uint64(), C.c_uint64()
        self.ctx.check(self.lib.fastf_bam2db_counts(self.job, C.byref(a), C.byref(b)), "bam2db_counts")
        return a.value, b.value

    def sample(self, ordinal_base=0):
        self.ctx.check(self.lib.fastf_bam2db_sample(self.job, ordinal_base), "bam2db_sample")

    def sample_counts(self):
        a, b = C.c_uint64(), C.c_uint64()
        self.ctx.check(self.lib.fastf_bam2db_sample_counts(self.job, C.byref(a), C.byref(b)), "bam2db_sample_counts")
        return a.value, b.value

    def kept_device(self):
        p, n = C.c_void_p(), C.c_uint64()
        self.ctx.check(self.lib.fastf_bam2db_kept_device(self.job, C.byref(p), C.byref(n)), "bam2db_kept_device")
        return p.value, n.value

    def key_layout(self):
        a, b, c = C.c_uint32(), C.c_uint32(), C.c_uint32()
        self.lib.fastf_bam2db_key_layout(self.job, C.byref(a), C.byref(b), C.byref(c))
        return a.value, b.value, c.value

    def finish(self, copy=True):
        res = _lib.Bam2dbResult()
        self.ctx.check(self.lib.fastf_bam2db_finish(self.job, C.byref(res)), "bam2db_finish")
        out = None
        if copy:
            z32 = np.zeros(0, np.uint32)
            out = {
                "m_gene": np.ctypeslib.as_array(res.m_gene, (res.nnz,)).copy() if res.nnz else z32,
                "m_cell": np.ctypeslib.as_array(res.m_cell, (res.nnz,)).copy() if res.nnz else z32,
                "m_count": np.ctypeslib.as_array(res.m_count, (res.nnz,)).copy() if res.nnz else z32,
                "row_keys": np.ctypeslib.as_array(res.row_keys, (res.n_rows,)).copy() if (self.want_rows and res.n_rows) else np.zeros(0, np.uint64),
            }
        stats = {f: getattr(res, f) for f, _ in _lib.Bam2dbResult._fields_ if not f.startswith("m_") and f != "row_keys"}
        self.lib.fastf_bam2db_result_free(C.byref(res))
        return stats, out

    def finish_sweep(self, rates):
        """The depth sweep instead of finish(): one result per depth rate, in the order given.  Returns [(stats, arrays)], each
        what finish() returns for a job begun with that rate (counters, COO, that rate's rows and n_rows with want_rows); the stage
        clocks are the sweep job's, the same for every rate."""
        thr = _thresholds(self.lib, rates)
        res = _lib.Bam2dbSweepResult()
        try:
            self.ctx.check(self.lib.fastf_bam2db_finish_sweep(self.job, len(thr), thr.ctypes.data_as(_lib.c_u64p), C.byref(res)), "bam2db_finish_sweep")
            return _sweep_to_python(res, thr, self.want_rows)
        finally:
            self.lib.fastf_bam2db_sweep_result_free(C.byref(res))

    def stats(self):
        res = _lib.Bam2dbResult()
        self.ctx.check(self.lib.fastf_bam2db_stats(self.job, C.byref(res)), "bam2db_stats")
        return {f: getattr(res, f) for f, _ in _lib.Bam2dbResult._fields_ if not f.startswith("m_") and f != "row_keys"}

    def close(self):
        if self.job:
            self.lib.fastf_bam2db_job_free(self.job)
            self.job = None

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()


def _feed_all(job, bam_bytes, feed_piece):
    buf = np.frombuffer(bam_bytes, dtype=np.uint8)
    n = buf.size
    step = feed_piece if feed_piece else max(n, 1)
    for lo in range(0, n, step):
        hi = min(n, lo + step)
        job.feed(buf.ctypes.data + lo, hi - lo)


def run_device(ctx, bam_bytes, inputs, rate_depth, seed, want_rows=True, inflate_lanes=0, chunk_inflated_bytes=0, feed_piece=0, umi_max_bytes=0):
    """The C-ABI call sequence for one BAM image in host memory.  Returns (stats dict, dict of numpy result arrays)."""
    with Bam2dbJob(ctx, inputs, rate_depth, seed, want_rows, inflate_lanes, chunk_inflated_bytes, umi_max_bytes) as job:
        _feed_all(job, bam_bytes, feed_piece)
        return job.finish()


def run_device_sweep(ctx, bam_bytes, inputs, rates, seed, want_rows=True, inflate_lanes=0, chunk_inflated_bytes=0, feed_piece=0, umi_max_bytes=0):
    """run_device for several depth rates out of one job: [(stats, arrays)] in the order of `rates`."""
    with Bam2dbJob(ctx, inputs, 0.0, seed, want_rows, inflate_lanes, chunk_inflated_bytes, umi_max_bytes) as job:
        _feed_all(job, bam_bytes, feed_piece)
        return job.finish_sweep(rates)


def matrix_header(bam_file, rate_cell, rate_depth, total, sampled, valid):
    # "%%%M" in the reference's format string prints "%%M" with glibc (src/bam2db_ds.c:500)
    return ("%%%%MatrixMarket matrix coordinate integer general\n%%metadata_json: \n%%{\n%%\t\"software_version\": \"fastF-1.0.0\",\n"
            "%%\t\"format_version\": 1,\n%%\t\"parent_bam\": \"%s\",\n%%\t\"rate_cell\": %.3f,\n%%\t\"rate_depth\": %.3f,\n"
            "%%\t\"total_n_FastQ\": %d,\n%%\t\"sampled_n_FastQ\": %d,\n%%\t\"sampled_valid_n_FastQ\": %d\n%%}\n") % (
        bam_file, float(np.float32(rate_cell)), float(np.float32(rate_depth)), total, sampled, valid)


def _lines_u32(cols, sep):
    """vectorised "a<sep>b<sep>c\\n" formatting of u32 columns"""
    if len(cols[0]) == 0:
        return b""
    parts = []
    for i, c in enumerate(cols):
        parts.append(np.char.mod("%d", c))
    s = parts[0]
    for p_ in parts[1:]:
        s = np.char.add(np.char.add(s, sep), p_)
    return ("\n".join(s.tolist()) + "\n").encode()


def decode_dna10(blob_content, umi_max_bytes):
    """decode_DNA(blob, 10): the first 10 bases of the 2-bit blob (reference src/bam2db_ds.c:53-93, called at :629)"""
    out = []
    for k in range(10):
        bitpos = 8 * umi_max_bytes - 2 * (k + 1)
        code = (blob_content >> bitpos) & 3 if bitpos >= 0 else 0
        out.append("ACGT"[code])
    return "".join(out)


def open_database(db_file, bam_file, barcodes_file, features_file):
    """the reference's opening sequence with its stderr lines (src/bam2db_ds.c:127-210); returns the sqlite connection or None"""
    try:
        db = sqlite3.connect(db_file, isolation_level=None)
    except sqlite3.Error as e:
        sys.stderr.write("Can't open database: %s\n" % e)
        return None
    sys.stderr.write("Opened database successfully\n")
    for path, what in ((bam_file, "BAM"), (barcodes_file, "cell barcode"), (features_file, "feature name")):
        if not os.path.exists(path):
            sys.stderr.write("Can't open %s file %s\n" % (what, path))
            return None
        sys.stderr.write("Opened %s file %s successfully\n" % (what, path))
    db.execute("CREATE TABLE cell (cell_barcode TEXT);")
    db.execute("CREATE TABLE feature (feature_id TEXT, feature_name TEXT, feature_type);")
    db.execute("CREATE TABLE umi (cell_index INTEGER, feature_index INTEGER, encoded_umi TEXT);")
    return db


def insert_lists(db, inputs):
    db.execute("BEGIN TRANSACTION")
    db.executemany("INSERT INTO cell VALUES (?);", ((c.decode("latin-1"),) for c in inputs.cells))
    db.execute("END TRANSACTION")
    db.execute("BEGIN TRANSACTION")
    db.executemany("INSERT INTO feature VALUES (?, ?, ?);", ((f[1].decode("latin-1"), f[2].decode("latin-1"), f[3].decode("latin-1")) for f in inputs.features))
    db.execute("END TRANSACTION")


def load_lists(db, lib, barcodes_file, features_file, rate_cell, seed):
    inputs = Bam2dbInputs(lib, barcodes_file, features_file, rate_cell, seed)
    print("Total number of cells: %d" % inputs.n_cells)
    print("Actual number of sampled cell barcodes: %d" % inputs.n_cells_sampled)
    if inputs.duplicate_barcodes:
        print("Warning: Duplicate cell barcodes were found in %s!" % barcodes_file)
    if inputs.duplicate_features:
        print("Warning: Duplicate feature names were found in %s!" % features_file)
    if db is not None:
        insert_lists(db, inputs)
    return inputs


def unique_counts(ctx, keys, key_bits):
    """distinct keys (ascending) and their multiplicities through the device sort + run-length (fastf_unique_counts_host)"""
    keys = np.ascontiguousarray(keys, dtype=np.uint64)
    ok, oc, nu = _lib.c_u64p(), _lib.c_u32p(), C.c_uint64()
    ctx.check(ctx.lib.fastf_unique_counts_host(ctx.h, keys.ctypes.data_as(_lib.c_u64p), keys.size, key_bits, C.byref(ok), C.byref(oc), C.byref(nu)), "unique_counts")
    n = nu.value
    try:
        uniq = np.ctypeslib.as_array(ok, shape=(n,)).copy() if n else np.zeros(0, np.uint64)
        counts = np.ctypeslib.as_array(oc, shape=(n,)).copy() if n else np.zeros(0, np.uint32)
    finally:
        ctx.lib.fastf_free(C.cast(ok, C.c_void_p))
        ctx.lib.fastf_free(C.cast(oc, C.c_void_p))
    return uniq, counts


def write_outputs(db, bam_file, path_out, inputs, rate_cell, rate_depth, stats, out, ctx=None):
    """sqlite tables umi / mtx (/ numi) and the 10x .gz files from the device result (reference src/bam2db_ds.c:351-567)"""
    cell, gene, nbytes, content = decode_rows(out["row_keys"], stats["bits_gene"], stats["bits_umi"], stats["umi_max_bytes"])
    mb = stats["umi_max_bytes"]

    def rows():
        for c, g, nb, ct in zip(cell.tolist(), gene.tolist(), nbytes.tolist(), content.tolist()):
            yield (c, g, None if nb < 0 else ct.to_bytes(mb, "big")[:nb])
    db.execute("BEGIN TRANSACTION")
    db.executemany("INSERT INTO umi VALUES (?, ?, ?);", rows())
    db.execute("END TRANSACTION")
    print("In %s, total fastQ reads: %d" % (bam_file, stats["total"]))
    print("In %s, sampled fastQ reads: %d" % (bam_file, stats["sampled"]))
    print("In %s, sampled and valid fastQ reads: %d" % (bam_file, stats["valid"]))
    # table mtx from the device COO, with the schema text sqlite gives `CREATE TABLE mtx AS SELECT ...` (src/bam2db_ds.c:480-483)
    db.execute("CREATE TABLE mtx(\n  feature_index INT,\n  cell_index INT,\n  expression_level\n)")
    db.execute("BEGIN TRANSACTION")
    db.executemany("INSERT INTO mtx VALUES (?, ?, ?);", zip(out["m_gene"].tolist(), out["m_cell"].tolist(), out["m_count"].tolist()))
    db.execute("END TRANSACTION")
    try:
        fb = gzip.open(os.path.join(path_out, "barcodes.tsv.gz"), "wb")
        ff = gzip.open(os.path.join(path_out, "features.tsv.gz"), "wb")
        fm = gzip.open(os.path.join(path_out, "matrix.mtx.gz"), "wb")
    except OSError as e:
        sys.stderr.write("\x1b[31mError:\x1b[0m can not open file %s\n" % e.filename)
        return 1
    fm.write(matrix_header(bam_file, rate_cell, rate_depth, stats["total"], stats["sampled"], stats["valid"]).encode("latin-1"))
    fm.write(b"%d %d %d\n" % (len(inputs.features), len(inputs.cells), stats["nnz"]))
    fm.write(_lines_u32([out["m_gene"], out["m_cell"], out["m_count"]], " "))
    fm.close()
    print("matrix.mtx.gz is generated.")
    fb.write(b"".join(c + b"\n" for c in inputs.cells))
    fb.close()
    print("barcodes.tsv.gz is generated.")
    ff.write(b"".join(f[1] + b"\t" + f[2] + b"\t" + f[3] + b"\n" for f in inputs.features))
    ff.close()
    print("features.tsv.gz is generated.")
    if _umi_copies_flag:
        # numi = copies per distinct (cell, gene, umi): GROUP BY cell_index, feature_index, encoded_umi (src/bam2db_ds.c:539-543)
        # (sorted and run-length encoded on the device; without a context -- tests of the writers alone -- numpy does the same)
        if ctx is not None:
            uniq, counts = unique_counts(ctx, out["row_keys"], stats["bits_cell"] + stats["bits_gene"] + stats["bits_umi"])
        else:
            uniq, counts = np.unique(out["row_keys"], return_counts=True)
        c2, g2, nb2, ct2 = decode_rows(uniq, stats["bits_gene"], stats["bits_umi"], stats["umi_max_bytes"])
        db.execute("CREATE TABLE numi(\n  feature_index INT,\n  cell_index INT,\n  encoded_umi TEXT,\n  n_copy\n)")
        db.execute("BEGIN TRANSACTION")
        db.executemany("INSERT INTO numi VALUES (?, ?, ?, ?);",
                       ((g, c, None if nb < 0 else ct.to_bytes(mb, "big")[:nb], n) for c, g, nb, ct, n in zip(c2.tolist(), g2.tolist(), nb2.tolist(), ct2.tolist(), counts.tolist())))
        db.execute("END TRANSACTION")
        with gzip.open(os.path.join(path_out, "umi.tsv.gz"), "wb") as fu:
            for c, g, nb, ct, n in zip(c2.tolist(), g2.tolist(), nb2.tolist(), ct2.tolist(), counts.tolist()):
                fu.write(("%d\t%d\t%s\t%d\n" % (g, c, "NULL" if nb < 0 else decode_dna10(ct, mb), n)).encode())
        print("umi.tsv.gz is generated.")
    return 0


def _run_with_retries(run):
    """run(umi_max_bytes, inflate_lanes), retried the way the reference's inputs need it"""
    flags, umi_bytes = 0, 3   # 10x UMIs: 10 or 12 bases; room for 16 on demand
    while True:
        try:
            return run(umi_bytes, flags)
        except _lib.FastfError as e:
            if "umi-too-long" in str(e) and umi_bytes == 3:
                umi_bytes = 4
            elif "record-straddles-bgzf-block" in str(e) and not flags:
                flags = BAM_STRADDLE   # not an htslib-written file: guess and verify the record starts per block (one chunk)
            else:
                raise


def bam2db(bam_file, db_file, path_out, barcodes_file, features_file, rate_cell, rate_depth, seed=926, device=0, ctx=None):
    own = ctx is None
    try:
        if own:
            ctx = _lib.Context(device)
        db = open_database(db_file, bam_file, barcodes_file, features_file)
        if db is None:
            return 1
        inputs = load_lists(db, ctx.lib, barcodes_file, features_file, rate_cell, seed)
        print("Start to convert bam file to sqlite3 database...")
        sys.stdout.flush()
        bam_bytes = np.fromfile(bam_file, dtype=np.uint8)
        stats, out = _run_with_retries(lambda mb, fl: run_device(ctx, bam_bytes, inputs, rate_depth, seed, want_rows=True, umi_max_bytes=mb, inflate_lanes=fl))
        rc = write_outputs(db, bam_file, path_out, inputs, rate_cell, rate_depth, stats, out, ctx=ctx)
        db.close()
        return rc
    except (_lib.FastfError, ValueError, OSError, sqlite3.Error) as e:
        sys.stderr.write("bam2db: %s\n" % e)
        return 1
    finally:
        if own and ctx is not None:
            ctx.close()


def sweep_layout(db_name, path_out, rates):
    """(name, float32 value, output directory, database) per rate: rate r writes into path_out/depth_<r as given>/, its database
    is that directory's <basename of db_name>.  Raises ValueError on what the sweep refuses."""
    if not 1 <= len(rates) <= _lib.SWEEP_MAX_RATES:
        raise ValueError("the depth sweep takes 1..%d rates" % _lib.SWEEP_MAX_RATES)
    out, seen = [], set()
    for r in rates:
        name = r if isinstance(r, str) else str(r)
        val = np.float32(float(r))
        if name in seen or val.tobytes() in seen:
            raise ValueError("the rate %s is listed twice" % name)
        seen.update((name, val.tobytes()))
        d = os.path.join(path_out, "depth_" + name)
        out.append((name, float(val), d, os.path.join(d, os.path.basename(db_name))))
    for _, _, _, db in out:
        if os.path.exists(db):
            raise ValueError("database: %s already exists, change the name of database in -d argument!" % db)
    return out


def bam2db_sweep(bam_file, db_name, path_out, barcodes_file, features_file, rate_cell, rates, seed=926, device=0, ctx=None, gpus=1):
    """bam2db at several depth rates out of one pass over the BAM.  Rate r's output set is exactly what
    bam2db(bam_file, <its database>, <its directory>, ..., rate_cell, r, seed) writes; see sweep_layout for where it goes.
    gpus > 1 shards the BAM over devices 0..gpus-1 of this node (fastf_bam2db_run_sharded_sweep); `ctx` / `device` then only count
    the copies of -u (umi.tsv, table numi).
    Returns 0 / 1 like bam2db."""
    own = ctx is None
    dbs = []
    try:
        layout = sweep_layout(db_name, path_out, rates)
        if gpus < 1:
            raise ValueError("gpus must be >= 1")
        if own and gpus == 1:
            ctx = _lib.Context(device)
        lib = ctx.lib if ctx is not None else _lib.load()   # gpus > 1: the driver opens one context per device itself
        for _, _, d, dbf in layout:
            os.makedirs(d, exist_ok=True)
            db = open_database(dbf, bam_file, barcodes_file, features_file)
            if db is None:
                return 1
            dbs.append(db)
        inputs = load_lists(None, lib, barcodes_file, features_file, rate_cell, seed)
        for db in dbs:
            insert_lists(db, inputs)
        print("Start to convert bam file to sqlite3 database...")
        sys.stdout.flush()
        bam_bytes = np.fromfile(bam_file, dtype=np.uint8)
        vals = [v for _, v, _, _ in layout]
        if gpus > 1:
            # a BAM whose records straddle blocks fails here: the straddle mode (BAM_STRADDLE) needs the whole file in one job
            results = _run_with_retries(lambda mb, fl: run_sharded_sweep(lib, bam_bytes, inputs, vals, seed, gpus, want_rows=True, umi_max_bytes=mb, inflate_lanes=fl))
        else:
            results = _run_with_retries(lambda mb, fl: run_device_sweep(ctx, bam_bytes, inputs, vals, seed, want_rows=True, umi_max_bytes=mb, inflate_lanes=fl))
        if ctx is None and _umi_copies_flag:
            ctx = _lib.Context(device)   # numi / umi.tsv: the copies of every distinct key are counted on one device
        for (name, val, d, _), db, (stats, out) in zip(layout, dbs, results):
            print("Depth rate %s -> %s" % (name, d))
            if write_outputs(db, bam_file, d, inputs, rate_cell, val, stats, out, ctx=ctx):
                return 1
        return 0
    except (_lib.FastfError, ValueError, OSError, sqlite3.Error) as e:
        sys.stderr.write("bam2db: %s\n" % e)
        return 1
    finally:
        for db in dbs:
            db.close()
        if own and ctx is not None:
            ctx.close()
