/* fastf_gpu.h -- C-ABI of the B200-native bam2db / freq hot path (libfastf_gpu.so).
 *
 * This is the drop-in seam for yuw444/fastF.  The reference has no plugin API; the seam is the pair
 * of plain C calls its CLI makes:
 *     int   bam2db(char*,char*,char*,char*,char*,float,float,unsigned)   reference src/bam2db_ds.h:62-70
 *     node *cell_counts(gzFile, size_t, size_t)                          reference src/count.h:6
 * Inside bam2db() the part replaced by this library is the hot loop and the sqlite aggregation
 *     while (sam_read1(...) >= 0) { CB / draw / xf / GX / UB / INSERT }  reference src/bam2db_ds.c:360-438
 *     CREATE TABLE mtx AS SELECT ... COUNT(DISTINCT encoded_umi) ... GROUP BY cell_index, feature_index
 *                                                                        reference src/bam2db_ds.c:480-483
 * and inside cell_counts() the whole read/insert loop                    reference src/count.c:7-18.
 * Everything else (option parsing, reading the barcode/feature lists, SampleInt on <= 10^5 cells,
 * the sqlite file and the .gz writers) stays host C (fastf_b200/host/), fed from these results.
 *
 * Conventions: extern "C", plain pointers and sizes, no C++/torch types.  Every function returns 0 on
 * success and non-zero on failure; fastf_last_error() returns the message.  There is no CPU fallback:
 * without a CUDA device fastf_ctx_create fails.
 */
#ifndef FASTF_GPU_H
#define FASTF_GPU_H
#include <stddef.h>
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

/* OR this into any `inflate_lanes` argument to inflate with the B200 hardware decompression engine (driver API
 * cuMemBatchDecompressAsync, DEFLATE) instead of the hand-written SM kernel.  Fails loudly where the engine is absent. */
#define FASTF_INFLATE_HW_ENGINE 0x100u
/* OR this in to skip the CRC-32 check of every inflated block against its BGZF trailer (htslib bgzf_read_block does the same check
 * for the reference, src/bam2db_ds.c:360).  On by default: a mismatch fails the job with "bgzf-crc32-mismatch". */
#define FASTF_INFLATE_NO_CRC 0x200u
/* OR this in for BAM files whose records cross BGZF block boundaries (writers other than htslib, e.g. htsjdk or STAR).  Without it such
 * a file fails with "record-straddles-bgzf-block"; with it every block's first record start is guessed and the per-block kernels verify
 * the guesses (a wrong one fails the job, never the result).  The mode keeps the whole file in one chunk: the inflated bytes must fit HBM. */
#define FASTF_BAM_STRADDLE 0x400u

typedef struct fastf_ctx fastf_ctx;
typedef struct fastf_bam2db_job fastf_bam2db_job;

int fastf_abi_version(void);
/* how this binary was built: "streams=<BGZF blocks in flight per SM> lanes=.. svc=.. lbits=.. dbits=.. ring=.. staged=.. src=<hash of the kernel sources>";
 * hosts compare src with the sources they ship (fastf_b200/_lib.py refuses a stale library) */
const char *fastf_build_info(void);
int fastf_ctx_create(int device, fastf_ctx **out);
void fastf_ctx_destroy(fastf_ctx *ctx);
const char *fastf_last_error(const fastf_ctx *ctx);
/* pinned host memory for inputs that are fed repeatedly (bench end-to-end leg) */
int fastf_host_alloc(fastf_ctx *ctx, size_t bytes, void **out);
void fastf_host_free(fastf_ctx *ctx, void *p);
int fastf_device_alloc(fastf_ctx *ctx, size_t bytes, void **out);
void fastf_device_free(fastf_ctx *ctx, void *p);
int fastf_memcpy_h2d(fastf_ctx *ctx, void *dst_dev, const void *src_host, size_t bytes);
int fastf_memcpy_d2h(fastf_ctx *ctx, void *dst_host, const void *src_dev, size_t bytes);
int fastf_synchronize(fastf_ctx *ctx);
/* device and pinned buffers of finished jobs are cached in the context; this returns them to the driver */
void fastf_ctx_trim(fastf_ctx *ctx);
/* kernels launched through this context so far (bench.py: gpu_launches) */
uint32_t fastf_launch_count(const fastf_ctx *ctx);
/* the cudaStream_t all hot-path kernels are launched on (for external CUDA-event timing) */
void *fastf_compute_stream(const fastf_ctx *ctx);

/* ---- host helpers that define the sampling contract (reference src/utils.c:29-75, src/mt19937ar.c:149-153) ---- */
/* keep  <=>  genrand_int32()*(1.0/4294967295.0) < (double)rate_depth  <=>  u < T ;  T in [0, 2^32] */
uint64_t fastf_keep_threshold(float rate_depth);
/* n_cells_sampled = (size_t)((float)n_cells * rate_cell); fills out[0..ns) with the sorted sampled line indices and
 * *d0 with the number of MT19937 draws SampleInt consumed (0 when ns == n_cells). Returns ns, or UINT64_MAX if ns > n_cells. */
uint64_t fastf_sample_cells(uint64_t n_cells, float rate_cell, uint32_t seed, uint64_t *out, uint64_t *d0);
/* BGZF block index of a byte range (SAMv1 4.1); arrays are caller-allocated with capacity cap. Returns the number of
 * complete blocks (or -1 on a malformed block); *consumed = bytes covered by them. */
int64_t fastf_bgzf_index_host(const void *buf, size_t n, uint64_t *in_off, uint32_t *in_len, uint32_t *isize, uint64_t cap, size_t *consumed);

/* pre-order of the reference's histogram BST (insert_tree src/filter.c:105-124, print_tree src/filter.c:139-148) from the
 * first-occurrence ordinals of the distinct keys listed in ascending strcmp order: order_out[k] = index of the k-th printed key */
int fastf_cartesian_preorder(const uint32_t *first, uint64_t n, uint64_t *order_out);

/* ---- bam2db hot path ---- */
typedef struct {
    const char *cell_keys;      /* concatenated sampled barcodes, string i = [cell_off[i], cell_off[i+1]) -> cell_index i+1 */
    const uint32_t *cell_off;   /* n_cells + 1 offsets */
    uint32_t n_cells;
    const char *gene_keys;      /* feature ids, same layout -> feature_index i+1 */
    const uint32_t *gene_off;
    uint32_t n_genes;
    uint32_t seed;              /* init_genrand(seed) */
    uint64_t d0;                /* MT draws consumed by cell sampling */
    uint64_t keep_threshold;    /* fastf_keep_threshold(rate_depth) */
    uint32_t umi_max_bytes;     /* 0 = 3 (UMIs up to 12 bases); up to 4 */
    uint32_t want_rows;         /* also return the kept rows in read order (the sqlite `umi` table) */
    uint32_t inflate_lanes;     /* inflate kernel: 0 = default (thread-per-stream), 1..4 = shapes of it, 32/16/8 = lock-step kernel with that many
                                 * lanes per BGZF block; | FASTF_INFLATE_HW_ENGINE = hardware decompression engine */
    uint64_t chunk_inflated_bytes; /* 0 = default streaming chunk size */
    uint32_t headerless;        /* 1: the fed blocks start at an alignment record (a later shard of a BAM; the BAM header went to another job) */
} fastf_bam2db_params;

typedef struct {
    uint64_t total;             /* total_reads_counts            reference src/bam2db_ds.c:363 */
    uint64_t cb_valid;          /* reads that consumed a draw    reference src/bam2db_ds.c:385 */
    uint64_t sampled;           /* sampled_reads_counts          reference src/bam2db_ds.c:392 */
    uint64_t valid;             /* sampled_valid_reads_counts    reference src/bam2db_ds.c:435 */
    uint64_t nnz;               /* rows of table mtx, ascending (cell, gene) */
    uint32_t *m_gene, *m_cell, *m_count;   /* host arrays (library-owned until fastf_bam2db_result_free) */
    uint64_t n_rows;            /* == valid when want_rows */
    uint64_t *row_keys;         /* packed rows in read order: cell << (bits_gene+bits_umi) | gene << bits_umi | umi_code */
    uint32_t bits_cell, bits_gene, bits_umi, umi_max_bytes;
    uint64_t n_blocks, compressed_bytes, inflated_bytes;
    uint32_t status;            /* OR of FASTF_ST_* bits seen (0 = clean) */
    uint32_t n_launches;        /* kernels launched for this job */
    uint32_t n_chunks;          /* inflate (= parse) launches: one per streamed chunk */
    /* device time, CUDA events on the launching stream, milliseconds */
    float ms_inflate, ms_parse, ms_gather, ms_mt, ms_sample, ms_sort, ms_count, ms_device_total;
    float ms_crc;               /* CRC-32 verification of the inflated blocks */
} fastf_bam2db_result;

/* umi_code layout inside row_keys: bit (bits_umi-1) = non-NULL flag, then 8*umi_max_bytes content bits
 * (2 bits per base, MSB first, zero padded: reference encode_DNA src/bam2db_ds.c:22-51), then 3 bits = blob length in bytes. */

int fastf_bam2db_begin(fastf_ctx *ctx, const fastf_bam2db_params *p, fastf_bam2db_job **job);
/* compressed BGZF bytes in host memory; any split (partial blocks are carried to the next call) */
int fastf_bam2db_feed(fastf_bam2db_job *job, const void *host_bytes, size_t n);
/* compressed bytes already resident in HBM + their host-side block index (payload offsets relative to dev_bytes).  Blocks are launched in
 * chunks of a fixed number of blocks and may wait for the blocks of the NEXT feed to fill a chunk: dev_bytes must stay valid and unchanged
 * until fastf_bam2db_counts / _sample / _finish has returned.  (fastf_bam2db_feed copies its bytes before it returns.) */
int fastf_bam2db_feed_device(fastf_bam2db_job *job, const void *dev_bytes, size_t nbytes, const uint64_t *in_off, const uint32_t *in_len, const uint32_t *isize, uint64_t nblocks);
/* after the last feed: records and CB-valid reads seen by THIS job (multi-GPU: all-gather these to get ordinal bases) */
int fastf_bam2db_counts(fastf_bam2db_job *job, uint64_t *n_records, uint64_t *n_cb_valid);
/* depth sampling with the global ordinal of this job's first CB-valid read; leaves the kept keys (read order) on device */
int fastf_bam2db_sample(fastf_bam2db_job *job, uint64_t ordinal_base);
int fastf_bam2db_kept_device(fastf_bam2db_job *job, uint64_t **dev_keys, uint64_t *n);
/* after fastf_bam2db_sample: this job's sampled_reads_counts and sampled_valid_reads_counts (reference src/bam2db_ds.c:392,435) */
int fastf_bam2db_sample_counts(fastf_bam2db_job *job, uint64_t *sampled, uint64_t *valid);
int fastf_bam2db_key_layout(fastf_bam2db_job *job, uint32_t *bits_cell, uint32_t *bits_gene, uint32_t *bits_umi);
/* single-GPU tail: (sample if not done) + sort + dedup + count + copy back */
int fastf_bam2db_finish(fastf_bam2db_job *job, fastf_bam2db_result *res);
/* ---- depth sweep: one job, the outputs of several depth rates (single GPU) ----
 * For one -c / -s every read meets the same MT19937 draw u whatever the depth rate, and a larger threshold keeps a superset of the
 * reads a smaller one keeps.  So one inflate + parse + draw pass yields the exact result of every rate: rate[i] equals what
 * fastf_bam2db_finish returns for a job begun with keep_threshold = keep_thresholds[i].  The stage clocks are the job's, the same
 * in every rate[i]: ms_sample covers the per-rate histograms and the (key, rate index) compaction, ms_sort the one sort plus the
 * compaction of the distinct keys with their smallest rate index, ms_count the sum of the K per-rate count passes. */
#define FASTF_SWEEP_MAX_RATES 32
typedef struct {
    uint32_t n_rates;
    fastf_bam2db_result rate[FASTF_SWEEP_MAX_RATES]; /* rate[i] as fastf_bam2db_finish fills it for keep_thresholds[i]; row_keys NULL, n_rows 0 */
    uint64_t n_rows;      /* valid rows kept by the largest threshold, file order (0 unless the job was begun with want_rows) */
    uint64_t *row_keys;
    uint8_t *row_rate;    /* per row: index into keep_thresholds of the smallest threshold that keeps it (the first such index on ties);
                           * row r belongs to rate i's table umi <=> keep_thresholds[row_rate[r]] <= keep_thresholds[i] */
} fastf_bam2db_sweep_result;
/* instead of fastf_bam2db_finish (and of fastf_bam2db_sample, which must not have been called); keep_thresholds in caller order,
 * 1..FASTF_SWEEP_MAX_RATES of them, each <= 2^32 (fastf_keep_threshold); p->keep_threshold of the job is ignored */
int fastf_bam2db_finish_sweep(fastf_bam2db_job *job, uint32_t n_rates, const uint64_t *keep_thresholds, fastf_bam2db_sweep_result *res);
void fastf_bam2db_sweep_result_free(fastf_bam2db_sweep_result *res);
/* The depth sweep's per-shard building blocks (multi-GPU driver).  Unlike fastf_bam2db_finish_sweep these take the thresholds already
 * sorted, non-decreasing (1..FASTF_SWEEP_MAX_RATES of them, each <= 2^32): the caller sorts once and keeps the map to its own order.
 * The RATE INDEX of a row is its position p in that sorted list: the smallest p with u < sorted_thresholds[p] for the row's draw u,
 * so the row belongs to the output of every rate q >= p.  Device rate arrays hold it as a u32 per key.
 * fastf_bam2db_sample_sweep: instead of fastf_bam2db_sample (the job's CB-valid reads meet draws d0 + ordinal_base + k); sampled[p] /
 * valid[p] (host, n_rates each) = this job's sampled_reads_counts / sampled_valid_reads_counts at sorted rate p. */
int fastf_bam2db_sample_sweep(fastf_bam2db_job *job, uint64_t ordinal_base, uint32_t n_rates, const uint64_t *sorted_thresholds, uint64_t *sampled, uint64_t *valid);
/* after fastf_bam2db_sample_sweep: the valid rows kept by the largest threshold (file order) and their rate indices, owned by the job */
int fastf_bam2db_kept_sweep_device(fastf_bam2db_job *job, uint64_t **dev_keys, uint32_t **dev_rates, uint64_t *n);
/* ---- cell-rate grid: one job, the outputs of several cell rates x several depth rates (single GPU) ----
 * Each cell rate -c samples its own cell table and skips its own number of draws d0 (fastf_sample_cells), so the depth sweep's subset
 * argument does not hold across cell rates.  Inflate, CRC, record framing, the aux walk, the GX lookup and the UMI packing do not depend
 * on the cell table, though: a grid job parses the BAM once against the UNION of the cell tables (p->cell_keys / cell_off / n_cells;
 * p->d0 and p->keep_threshold are ignored) and keeps the cell of every CB-valid read, insertable or not.  Per cell rate it then rebuilds
 * on the device, in file order, exactly the candidate array a job begun with that rate's table would have gathered (the reads whose
 * cell the table holds, with the table's cell index) and runs the depth sweep over it at the rate's d0.
 * The union is the union of the tables' barcodes, not the sampled lines of the largest rate: the host stops a table at its first
 * duplicate barcode, so a smaller rate's table can hold a barcode that a larger rate's table lacks.
 * After begin_grid the job is fed as any other and finished with fastf_bam2db_finish_grid only: fastf_bam2db_finish / _finish_sweep /
 * _sample / _sample_sweep / _kept_device refuse a grid job, and finish_grid refuses any other job.  fastf_bam2db_counts on a grid job
 * reports the union table's CB-valid reads.  FASTF_BAM_STRADDLE works as for one job.  The job sees every read of every table, so it
 * fails with umi-too-long exactly where a single job begun with the union table would: retry with a larger umi_max_bytes as there. */
#define FASTF_GRID_MAX_CELL_RATES 32
typedef struct {
    const uint32_t *cell_index;   /* p->n_cells entries: cell_index[u - 1] = 1-based index in this rate's table of union cell u, 0 = not in it */
    uint32_t n_cells;             /* cells of this rate's table (its nonzero cell_index values are 1..n_cells, each once) */
    uint64_t d0;                  /* MT draws consumed by this rate's cell sampling */
} fastf_bam2db_cell_rate;
int fastf_bam2db_begin_grid(fastf_ctx *ctx, const fastf_bam2db_params *p, fastf_bam2db_job **job);
/* res[i] (n_cell_rates of them, caller order) is what fastf_bam2db_finish_sweep(n_rates, keep_thresholds) returns for a job begun with
 * cell rate i's table and d0: every depth rate's counters (cb_valid = that table's CB-valid reads) and COO, bits_cell of that table, and
 * the rows with their rate index when p->want_rows.  Stage clocks: ms_inflate / ms_crc / ms_parse / ms_gather are the shared pass's;
 * ms_mt, ms_sample (including the remap), ms_sort and ms_count are cell rate i's own.  ms_device_total and n_launches count from the
 * start of the job: for cell rate i they cover the shared pass and cell rates 0..i.  1..FASTF_GRID_MAX_CELL_RATES cell rates and
 * 1..FASTF_SWEEP_MAX_RATES depth thresholds (validated as in finish_sweep).  res[0..min(n_cell_rates, FASTF_GRID_MAX_CELL_RATES)) is
 * zeroed before anything is checked; free every res[i] with fastf_bam2db_sweep_result_free, also after a failure. */
int fastf_bam2db_finish_grid(fastf_bam2db_job *job, uint32_t n_cell_rates, const fastf_bam2db_cell_rate *cell_rates, uint32_t n_rates, const uint64_t *keep_thresholds,
                             fastf_bam2db_sweep_result *res);
/* counters, sizes and per-stage device clocks so far, without finishing (multi-GPU driver); no arrays are allocated */
int fastf_bam2db_stats(fastf_bam2db_job *job, fastf_bam2db_result *res);
void fastf_bam2db_job_free(fastf_bam2db_job *job);
void fastf_bam2db_result_free(fastf_bam2db_result *res);

/* ---- bam2db over several GPUs of one node, driven by ONE host process (fastf_b200/csrc/sharded.cu; SURVEY.md 8e) ----
 * The whole BGZF file image (host memory; an mmap of the file will do) is cut into contiguous block shards, one per device; every
 * device runs the single-GPU streaming path on its shard, the shards agree on the global MT19937 draw ordinals, exchange their
 * locally deduplicated keys with an NCCL all-to-all (ncclSend / ncclRecv over NVLink) partitioned by cell, and count locally.
 * res is laid out exactly like fastf_bam2db_finish's and is identical to the single-GPU result (and to the reference's tables:
 * src/bam2db_ds.c:360-438,480-483).  devices == NULL means 0..n_devices-1.  p->want_rows / umi_max_bytes / inflate_lanes as in
 * fastf_bam2db_begin (FASTF_BAM_STRADDLE is single-GPU only).  Stage clocks: the maximum over devices; ms_sort = the local unique +
 * partition, ms_count = the receiving-side sort + count including the copy of the COO piece to the host (CUDA events on
 * fastf_compute_stream around each call).  Returns 0, or 1 with fastf_sharded_last_error(). */
int fastf_bam2db_run_sharded(int n_devices, const int *devices, const fastf_bam2db_params *p, const void *bgzf_bytes, size_t n_bytes, fastf_bam2db_result *res);
/* The depth sweep over the same shards: res equals what fastf_bam2db_finish_sweep returns for one job over the whole file with these
 * keep_thresholds (caller order, validated as there): every rate[i]'s counters and COO, and n_rows / row_keys / row_rate in file order.
 * Each shard samples its reads at all rates at once (fastf_bam2db_sample_sweep), keeps every distinct key once with its smallest rate
 * index, and sends the rate index beside the key in the same all-to-all; the receiving device counts every rate
 * (fastf_sweep_count_device).  Stage clocks as in fastf_bam2db_run_sharded, ms_count over every rate's count and COO copy; the same
 * in every rate[i]. */
int fastf_bam2db_run_sharded_sweep(int n_devices, const int *devices, const fastf_bam2db_params *p, const void *bgzf_bytes, size_t n_bytes, uint32_t n_rates,
                                   const uint64_t *keep_thresholds, fastf_bam2db_sweep_result *res);
const char *fastf_sharded_last_error(void);
uint64_t fastf_sharded_exchanged(void);   /* keys that crossed the all-to-all in the last call (diagnostic) */

/* ---- device-level building blocks (multi-GPU driver, unit tests) ---- */
/* in-place stable LSD radix sort of n u64 keys on device over key_bits low bits (vals optional, may be NULL) */
int fastf_sort_u64_device(fastf_ctx *ctx, uint64_t *dev_keys, uint32_t *dev_vals, uint64_t n, uint32_t key_bits);
/* sorted packed keys on device -> COO (host arrays, library-owned: free with fastf_free) */
int fastf_dedup_count_device(fastf_ctx *ctx, const uint64_t *dev_sorted_keys, uint64_t n, uint32_t bits_gene, uint32_t bits_umi,
                             uint64_t *nnz, uint32_t **m_gene, uint32_t **m_cell, uint32_t **m_count);
/* same with the COO left on the device in caller-provided arrays of capacity >= n */
int fastf_dedup_count_device_out(fastf_ctx *ctx, const uint64_t *dev_sorted_keys, uint64_t n, uint32_t bits_gene, uint32_t bits_umi,
                                 uint64_t *nnz, uint32_t *dev_gene, uint32_t *dev_cell, uint32_t *dev_count);
/* locally sort + unique kept keys and partition them by destination rank = (cell_index-1)*nparts/n_cells (an order-preserving
 * partition of the cell index): out_keys (device, capacity n) holds the unique keys grouped by destination, each group
 * ascending; part_counts[nparts] (host) their sizes */
int fastf_unique_partition_device(fastf_ctx *ctx, uint64_t *dev_keys, uint64_t n, uint32_t key_bits, uint32_t bits_gene, uint32_t bits_umi,
                                  uint32_t n_cells, uint32_t nparts, uint64_t *dev_out_keys, uint64_t *part_counts);
/* the same carrying a rate index (fastf_bam2db_sample_sweep) per key: every distinct key leaves once, with the smallest rate index of
 * its copies in dev_out_rates (device, capacity n); dev_keys and dev_rates are overwritten */
int fastf_unique_partition_rates_device(fastf_ctx *ctx, uint64_t *dev_keys, uint32_t *dev_rates, uint64_t n, uint32_t key_bits, uint32_t bits_gene, uint32_t bits_umi,
                                        uint32_t n_cells, uint32_t nparts, uint64_t *dev_out_keys, uint32_t *dev_out_rates, uint64_t *part_counts);
/* the depth sweep's count over (key, rate index) rows on device, in any order, repeated keys allowed (each key counts at its smallest
 * rate index); sorts dev_keys / dev_rates in place.  Per sorted rate p < n_rates: nnz[p] rows of table mtx, ascending (cell, gene), in
 * host arrays m_gene[p] / m_cell[p] / m_count[p] (library-owned: free with fastf_free).  Only one rate's COO is on the device at a time. */
int fastf_sweep_count_device(fastf_ctx *ctx, uint64_t *dev_keys, uint32_t *dev_rates, uint64_t n, uint32_t key_bits, uint32_t bits_gene, uint32_t bits_umi, uint32_t n_rates,
                             uint64_t *nnz, uint32_t **m_gene, uint32_t **m_cell, uint32_t **m_count);
void fastf_free(void *p);

/* host-buffer wrappers around single kernels (tests, smoke) */
int fastf_inflate_host(fastf_ctx *ctx, const void *bgzf_bytes, size_t n, int lanes, void **out, size_t *out_n, float *ms);
int fastf_mt19937_host(fastf_ctx *ctx, uint32_t seed, uint64_t n, uint32_t *out_words);
/* the n outputs starting at stream index `first` (GF(2) jump-ahead to `first`, then the normal twist): what a later shard of a
 * multi-GPU job does instead of generating every draw in front of its own */
int fastf_mt19937_host_from(fastf_ctx *ctx, uint32_t seed, uint64_t first, uint64_t n, uint32_t *out_words);
int fastf_mt19937_keepbits_host(fastf_ctx *ctx, uint32_t seed, uint64_t n, uint64_t threshold, uint32_t *out_bits /* ceil(n/32) words */);
int fastf_sort_u64_host(fastf_ctx *ctx, uint64_t *keys, uint32_t *vals, uint64_t n, uint32_t key_bits);
/* distinct keys (ascending) and their multiplicities: device sort + run-length heads.  Replaces `SELECT ..., COUNT(*) ... GROUP BY
 * cell_index, feature_index, encoded_umi` of -u/--umicopies (reference src/bam2db_ds.c:527-530).  *out_keys / *out_counts are
 * malloc'ed by the library: free() them. */
int fastf_unique_counts_host(fastf_ctx *ctx, const uint64_t *keys, uint64_t n, uint32_t key_bits, uint64_t **out_keys, uint32_t **out_counts, uint64_t *n_unique);

/* ---- freq hot path (reference src/count.c:3-21) ---- */
typedef struct {
    uint64_t n_reads;           /* FASTQ records seen */
    uint64_t n_keys;            /* distinct pure-ACGT keys */
    uint64_t *key;              /* 2 bits per base, first base most significant; ascending == strcmp order */
    uint32_t *count;
    uint32_t *first;            /* read ordinal of the first occurrence (insertion time into the reference's BST) */
    uint64_t n_exceptions;      /* reads whose key holds a non-ACGT byte: raw bytes for the host merge */
    uint32_t *exc_ordinal;
    uint8_t *exc_bytes;         /* FASTF_FREQ_EXC_STRIDE (32) raw bytes each, from the start of the sequence line */
    uint32_t exc_stride;
    uint64_t n_lines;
    uint8_t last_byte_is_newline;
    uint64_t n_blocks, compressed_bytes, inflated_bytes;
    uint32_t status, n_launches;
    float ms_inflate, ms_keys, ms_sort, ms_rle, ms_device_total;
} fastf_freq_result;
/* bytes = whole R1 file image (BGZF, or plain uncompressed text); key_len = len_cellbarcode + len_umi (<= 31) */
int fastf_freq_gpu(fastf_ctx *ctx, const void *host_bytes, size_t n, uint32_t key_len, uint32_t inflate_lanes, fastf_freq_result *res);
/* same with the compressed bytes + block index already resident on the device (bench `value` leg) */
int fastf_freq_gpu_device(fastf_ctx *ctx, const void *dev_bytes, size_t nbytes, const uint64_t *in_off, const uint32_t *in_len, const uint32_t *isize, uint64_t nblocks,
                          uint32_t key_len, uint32_t inflate_lanes, fastf_freq_result *res);
void fastf_freq_result_free(fastf_freq_result *res);

/* ---- crb / extract: the reference's other two per-record BAM histograms -----------------------------------------------------
 * Replaces read_bam() (reference src/extract.c:64-133, called from cmd_crb src/main.c:272) and the record loop of extract_bam()
 * (src/extract.c:135-199, called from cmd_extract src/main.c:399): for every record that carries tag A, count its value -- a string
 * (bam_aux2Z), the pair (A, B) of two strings (crb: A = "CB", B = "CR"), or an integer (bam_aux2i printed with "%d").  The host
 * turns (value, count, first occurrence) into the pre-order of the reference's BSTs (insert_tree / insert_CB_node).  Where the
 * reference dereferences NULL (string mode on a non-string tag, CB present without CR) the call fails with "tag-not-a-string". */
#define FASTF_TAG_STRING 0u
#define FASTF_TAG_INT 1u
typedef struct {
    uint64_t n_records;         /* BAM records in the file (crb: read_count; extract: total_count / 2, src/extract.c:162,164) */
    uint64_t n_hits;            /* records carrying tag A (extract: valid_count) */
    uint64_t n_groups;          /* distinct values / pairs; the per-group arrays below are in no particular order */
    uint32_t mode;
    uint32_t *first;            /* ordinal among the hits (file order) of the group's first occurrence */
    uint32_t *count;
    int32_t *ivalue;            /* FASTF_TAG_INT: the value */
    uint64_t *a_off;            /* FASTF_TAG_STRING: value A = strings[a_off, a_off + a_len), value B follows it (b_len bytes); no NULs */
    uint32_t *a_len, *b_len;
    char *strings;
    uint64_t strings_bytes;
    uint64_t n_blocks, compressed_bytes, inflated_bytes;
    uint32_t status, n_launches;
    uint32_t hash_rounds;       /* 1 unless two different values shared a 64-bit hash (detected byte for byte, re-run with another seed) */
    float ms_inflate, ms_tags, ms_sort, ms_rle, ms_device_total;
} fastf_taghist_result;
/* bgzf_bytes: the whole BAM file in host memory; tag_b = NULL for a single tag.  The file streams through HBM in chunks of whole
 * blocks; each chunk is grouped on the device and the per-chunk groups are merged on the host. */
int fastf_taghist_gpu(fastf_ctx *ctx, const void *bgzf_bytes, size_t n, const char *tag_a, uint32_t mode, const char *tag_b, uint32_t inflate_lanes, fastf_taghist_result *res);
void fastf_taghist_result_free(fastf_taghist_result *res);
/* test hooks (0, 0 = production): blocks per streaming chunk, and a mask ANDed onto the first round's hash keys to force collisions */
void fastf_taghist_test_hooks(fastf_ctx *ctx, uint64_t chunk_blocks, uint64_t round0_key_mask);

#ifdef __cplusplus
}
#endif
#endif
