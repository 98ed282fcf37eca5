/* Host side of the operators, with the reference's own signatures (yuw444/fastF):
 *   int bam2db(char *bam_file, char *db_file, char *path_out, char *barcodes_file, char *features_file,
 *              float rate_cell, float rate_depth, unsigned int seed);            reference src/bam2db_ds.h:62-70
 *   freq: cell_counts(gzFile, l, u) + print_tree(node*, FILE*)                   reference src/count.h:6, src/filter.h:77
 * The per-read loop and the aggregation run on the GPU through include/fastf_gpu.h; nothing here has a CPU fallback. */
#ifndef FASTF_HOST_H
#define FASTF_HOST_H
#include <stddef.h>
#include <stdint.h>
#include <stdio.h>
#include <sys/types.h>
#include <zlib.h>
extern int _umi_copies_flag;   /* reference src/bam2db_ds.h:23 */
extern int fastf_device;       /* CUDA device ordinal (env FASTF_DEVICE, default 0) */
extern int fastf_gpus;         /* bam2db over this many GPUs of the node (env FASTF_GPUS or --gpus N, default 1) */
int bam2db(char *bam_file, char *db_file, char *path_out, char *barcodes_file, char *features_file, float rate_cell, float rate_depth, unsigned int seed);
/* bam2db over several output sets out of one device job (not a reference entry point; bam2db() is its one-set call).  The cell axis
 * is n_cell_rates cell rates (1..32, cell_names[i] names rate i on stdout), or with n_cell_rates = 0 the one rate cell_rates[0] and
 * no union table.  The depth axis is n_rates depth rates (1..32, named by rate_names[j]), or with n_rates = 0 the one rate rates[0]
 * (cell rates need n_rates >= 1).  Set (i, j) = what bam2db(..., cell_rates[i], rates[j], seed) writes, into out_dirs[i * K + j]
 * with database db_files[i * K + j], K = max(n_rates, 1).  Several cell or depth rates run on one GPU. */
int bam2db_run(char *bam_file, char **db_files, char **out_dirs, char *barcodes_file, char *features_file, uint32_t n_cell_rates, const char *const *cell_names,
               const float *cell_rates, uint32_t n_rates, const char *const *rate_names, const float *rates, unsigned int seed);
/* cell_counts + print_tree in one call: histogram of the first l+u bases of every read of R1 (BGZF or plain text), written to fp
 * in the reference's BST pre-order.  Returns 0 / 1. */
int freq_whitelist(const char *r1_path, size_t len_cellbarcode, size_t len_umi, FILE *fp);
/* reference extract_bam(bam_file, tag, type) (src/extract.h, src/extract.c:135-216): histogram of one aux tag -> ./tag_summary.csv; type 0 = string, 1 = integer.
 * Returns 0 / 1 (the reference returns void and exits on errors). */
int extract_bam(char *bam_file, const char *tag, int type);
/* reference read_bam() + print_CB_node() (src/extract.c:47-133): per cell barcode, its raw barcodes (CR) with counts, one gz line each */
int crb_write(char *bam_file, gzFile out);

/* ---- host writers / readers that keep up with the device (sqlite_bulk.c, fast_writers.c) ---- */
typedef struct fastf_sqlite_bulk fastf_sqlite_bulk;
/* direct table b-tree loader: the table (created through sqlite, still empty, connection closed) gets rows with rowids 1..n */
fastf_sqlite_bulk *fastf_sqlite_bulk_begin(const char *db_file, unsigned root_page);
int fastf_sqlite_bulk_row(fastf_sqlite_bulk *b, const int64_t *ints, unsigned n_int, int has_tail, const void *tail_blob_or_null, unsigned tail_len);
int fastf_sqlite_bulk_row4(fastf_sqlite_bulk *b, const int64_t head[2], const void *blob_or_null, unsigned blob_len, int64_t last);
/* row i of a bulk load -> record: ncol serial types (< 128 each) and their nb body bytes (see sqlite_bulk.c) */
typedef void (*fastf_row_encoder)(void *ctx, uint64_t i, uint8_t *types, unsigned *ncol, uint8_t *body, unsigned *nb);
int fastf_sqlite_bulk_rows_parallel(fastf_sqlite_bulk *b, uint64_t n, fastf_row_encoder enc, void *ctx);
unsigned fastf_sqlite_int_col(int64_t v, uint8_t *type, uint8_t *body);   /* minimal-width integer column; returns the body bytes */
int fastf_sqlite_bulk_end(fastf_sqlite_bulk *b);
typedef struct { char *p; size_t n, cap; } fastf_textbuf;
void fastf_textbuf_reserve(fastf_textbuf *b, size_t extra);
void fastf_textbuf_free(fastf_textbuf *b);
unsigned fastf_fmt_u64(char *p, uint64_t v);
unsigned fastf_fmt_i64(char *p, int64_t v);
int fastf_gz_write_parallel(const char *path, const char *text, size_t n);
#define FASTF_LINE_MAX 96
typedef unsigned (*fastf_line_fmt)(void *ctx, uint64_t i, char *p);   /* writes the line of row i (<= FASTF_LINE_MAX bytes), returns its length */
int fastf_gz_write_lines_parallel(const char *path, const char *head, size_t head_n, uint64_t n_rows, fastf_line_fmt fmt, void *ctx);
ssize_t fastf_pread_parallel(int fd, void *dst, size_t n, off_t off);
int fastf_host_threads(void);
#endif
