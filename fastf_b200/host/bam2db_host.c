/* bam2db(): drop-in for reference src/bam2db_ds.c:106-573.  Same arguments, return value, stdout/stderr lines and output files;
 * the BAM loop (reference :360-438) and the GROUP BY (:480-483) are replaced by the device job of include/fastf_gpu.h. */
#include "fastf_host.h"
#include "../../include/fastf_gpu.h"
#include "sqlite3_decl.h"
#include <stdint.h>
#include <stdlib.h>
#include <string.h>
#include <zlib.h>
#include <fcntl.h>
#include <sys/mman.h>
#include <sys/stat.h>
#include <unistd.h>

int _umi_copies_flag = 0;
int fastf_device = 0;
int fastf_gpus = 1;     /* > 1: the one-process multi-GPU driver of the library (FASTF_GPUS / --gpus) */

typedef struct { char *buf; uint32_t *off; uint32_t n, cap; size_t len, bcap; } strlist;
static void sl_push(strlist *l, const char *s, size_t n)
{
    if (l->n + 2 > l->cap) { l->cap = l->cap ? l->cap * 2 : 1024; l->off = (uint32_t *)realloc(l->off, sizeof(uint32_t) * l->cap); }
    if (l->len + n + 1 > l->bcap) { l->bcap = (l->bcap ? l->bcap * 2 : 65536) + n; l->buf = (char *)realloc(l->buf, l->bcap); }
    if (l->n == 0) l->off[0] = 0;
    memcpy(l->buf + l->len, s, n);
    l->len += n;
    l->off[++l->n] = (uint32_t)l->len;
}
static void sl_free(strlist *l) { free(l->buf); free(l->off); memset(l, 0, sizeof *l); }
/* open-addressing string set for the duplicate checks of the two list files (reference hash_table_insert refuses duplicates) */
typedef struct { uint32_t *slot; uint32_t mask; const strlist *l; } strset;
static uint32_t djb2(const char *s, size_t n) { uint32_t h = 5381; for (size_t i = 0; i < n; i++) h = h * 33u + (unsigned char)s[i]; return h; }
static void ss_init(strset *s, const strlist *l, size_t expect) { uint32_t c = 64; while (c < expect * 2 + 8) c <<= 1; s->slot = (uint32_t *)calloc(c, 4); s->mask = c - 1; s->l = l; }
/* 1 + the string's index in the list, 0 when absent */
static uint32_t ss_has(const strset *s, const char *k, size_t n)
{
    for (uint32_t i = djb2(k, n) & s->mask; s->slot[i]; i = (i + 1) & s->mask) {
        uint32_t id = s->slot[i] - 1;
        if (s->l->off[id + 1] - s->l->off[id] == n && !memcmp(s->l->buf + s->l->off[id], k, n)) return id + 1;
    }
    return 0;
}
static void ss_add(strset *s, const char *k, size_t n, uint32_t id) { uint32_t i = djb2(k, n) & s->mask; while (s->slot[i]) i = (i + 1) & s->mask; s->slot[i] = id + 1; }

static int exec_sql(sqlite3 *db, const char *sql)
{
    char *err = NULL;
    if (sqlite3_exec(db, sql, NULL, 0, &err) != SQLITE_OK) { fprintf(stderr, "SQL error: %s\n", err ? err : "?"); sqlite3_free(err); return 1; }
    return 0;
}

/* FASTF_HOST_TIMING=1: wall clock of the host phases on stderr (where does a run spend its time next to the device job?) */
#include <time.h>
static double now_s(void) { struct timespec t; clock_gettime(CLOCK_MONOTONIC, &t); return (double)t.tv_sec + 1e-9 * (double)t.tv_nsec; }
static double g_t_last = 0;
static void phase(const char *what)
{
    static int on = -1;
    if (on < 0) on = getenv("FASTF_HOST_TIMING") != NULL;
    const double t = now_s();
    if (on && g_t_last > 0) fprintf(stderr, "[host timing] %-34s %8.3f s\n", what, t - g_t_last);
    g_t_last = t;
}

/* root page of a table (sqlite_master.rootpage); 0 when absent */
static unsigned table_root(sqlite3 *db, const char *name)
{
    sqlite3_stmt *st = NULL;
    unsigned root = 0;
    if (sqlite3_prepare_v2(db, "SELECT rootpage FROM sqlite_master WHERE type='table' AND name=?1;", -1, &st, NULL) != SQLITE_OK) return 0;
    sqlite3_bind_text(st, 1, name, -1, SQLITE_TRANSIENT);
    if (sqlite3_step(st) == SQLITE_ROW) root = (unsigned)sqlite3_column_int(st, 0);
    sqlite3_finalize(st);
    return root;
}

/* packed row key -> cell, gene, UMI blob (NULL UMI: returns -1 as the blob length) */
static inline int key_fields(uint64_t k, uint32_t bu, uint32_t bg, uint32_t mb, int64_t *cell, int64_t *gene, uint8_t blob[8], uint64_t *content_out)
{
    const uint64_t code = k & ((1ull << bu) - 1);
    *gene = (int64_t)((k >> bu) & ((1ull << bg) - 1));
    *cell = (int64_t)(k >> (bu + bg));
    if (!((code >> (bu - 1)) & 1)) return -1;
    const uint64_t content = (code >> 3) & ((1ull << (8 * mb)) - 1);
    for (uint32_t b = 0; b < mb; b++) blob[b] = (uint8_t)(content >> (8 * (mb - 1 - b)));
    if (content_out) *content_out = content;
    return (int)(code & 7);
}

typedef struct { const uint64_t *keys; uint32_t bu, bg, mb; } umi_rows;
static void umi_row_enc(void *c, uint64_t i, uint8_t *types, unsigned *ncol, uint8_t *body, unsigned *nb)
{
    const umi_rows *R = (const umi_rows *)c;
    int64_t cell, gene;
    uint8_t blob[8];
    const int bl = key_fields(R->keys[i], R->bu, R->bg, R->mb, &cell, &gene, blob, NULL);
    unsigned n = fastf_sqlite_int_col(cell, &types[0], body);
    n += fastf_sqlite_int_col(gene, &types[1], body + n);
    types[2] = bl < 0 ? 0 : (uint8_t)(12 + 2 * bl);   /* NULL, or a blob of bl bytes */
    if (bl > 0) { memcpy(body + n, blob, (size_t)bl); n += (unsigned)bl; }
    *ncol = 3; *nb = n;
}
typedef struct { const uint32_t *gene, *cell, *count; } mtx_rows;
static void mtx_row_enc(void *c, uint64_t i, uint8_t *types, unsigned *ncol, uint8_t *body, unsigned *nb)
{
    const mtx_rows *M = (const mtx_rows *)c;
    unsigned n = fastf_sqlite_int_col((int)M->gene[i], &types[0], body);
    n += fastf_sqlite_int_col((int)M->cell[i], &types[1], body + n);
    n += fastf_sqlite_int_col((int)M->count[i], &types[2], body + n);
    *ncol = 3; *nb = n;
}
static unsigned mtx_line_fmt(void *c, uint64_t i, char *p)
{
    const mtx_rows *M = (const mtx_rows *)c;
    char *q = p;
    q += fastf_fmt_i64(q, (int)M->gene[i]); *q++ = ' ';
    q += fastf_fmt_i64(q, (int)M->cell[i]); *q++ = ' ';
    q += fastf_fmt_i64(q, (int)M->count[i]); *q++ = '\n';
    return (unsigned)(q - p);
}

/* The writing half of bam2db(), one call per output set: tables umi (read order, reference :351-435), mtx (:480-483) and numi
 * (:527-530) of db_file (opened as *dbp, tables cell / feature / umi already filled or created; closed here), the three count
 * lines, and the 10x files under path_out.  res holds the counters and the COO; rows are the table umi's packed keys. */
static int write_outputs(sqlite3 **dbp, const char *db_file, const char *bam_file, const char *path_out, float rate_cell, float rate_depth, const fastf_bam2db_result *res,
                         const uint64_t *rows, uint64_t n_rows, const strlist *cells, const strlist *fkeys, const strlist *fid, const strlist *fname, const strlist *ftype, fastf_ctx *ctx)
{
    int rc = 1;
    sqlite3 *db = *dbp;
    gzFile file_barcode = NULL, file_feature = NULL;
    char path[2048];
    /* sqlite creates the empty tables; the rows are then laid out directly as b-tree pages (sqlite_bulk.c): at 10^8 rows a
     * sqlite3_step() per row costs minutes behind a device job of seconds. */
    if (exec_sql(db, "CREATE TABLE mtx(\n  feature_index INT,\n  cell_index INT,\n  expression_level\n)")) goto done;
    if (_umi_copies_flag && exec_sql(db, "CREATE TABLE numi(\n  feature_index INT,\n  cell_index INT,\n  encoded_umi TEXT,\n  n_copy\n)")) goto done;
    const unsigned root_umi = table_root(db, "umi"), root_mtx = table_root(db, "mtx"), root_numi = _umi_copies_flag ? table_root(db, "numi") : 0;
    if (!root_umi || !root_mtx || (_umi_copies_flag && !root_numi)) { fprintf(stderr, "SQL error: table root pages not found\n"); goto done; }
    if (sqlite3_close(db) != SQLITE_OK) { fprintf(stderr, "SQL error: %s\n", sqlite3_errmsg(db)); goto done; }
    *dbp = db = NULL;
    const uint32_t bu = res->bits_umi, bg = res->bits_gene, mb = res->umi_max_bytes;
    {
        fastf_sqlite_bulk *bulk = fastf_sqlite_bulk_begin(db_file, root_umi);
        if (!bulk) { fprintf(stderr, "SQL error: cannot append to table umi of %s\n", db_file); goto done; }
        umi_rows R = {rows, bu, bg, mb};
        fastf_sqlite_bulk_rows_parallel(bulk, n_rows, umi_row_enc, &R);
        if (fastf_sqlite_bulk_end(bulk)) { fprintf(stderr, "SQL error: writing table umi of %s failed\n", db_file); goto done; }
    }
    phase("table umi (direct b-tree)");
    printf("In %s, total fastQ reads: %zu\n", bam_file, (size_t)res->total);
    printf("In %s, sampled fastQ reads: %zu\n", bam_file, (size_t)res->sampled);
    printf("In %s, sampled and valid fastQ reads: %zu\n", bam_file, (size_t)res->valid);

    /* ---- 10x output (reference :447-567) ---- */
    snprintf(path, sizeof path, "%s/barcodes.tsv.gz", path_out);
    if (!(file_barcode = gzopen(path, "wb"))) { fprintf(stderr, "\x1b[31mError:\x1b[0m can not open file %s\n", path); goto done; }
    snprintf(path, sizeof path, "%s/features.tsv.gz", path_out);
    if (!(file_feature = gzopen(path, "wb"))) { fprintf(stderr, "\x1b[31mError:\x1b[0m can not open file %s\n", path); goto done; }
    {
        /* table mtx = the device COO */
        fastf_sqlite_bulk *bulk = fastf_sqlite_bulk_begin(db_file, root_mtx);
        if (!bulk) { fprintf(stderr, "SQL error: cannot append to table mtx of %s\n", db_file); goto done; }
        mtx_rows M = {res->m_gene, res->m_cell, res->m_count};
        fastf_sqlite_bulk_rows_parallel(bulk, res->nnz, mtx_row_enc, &M);
        if (fastf_sqlite_bulk_end(bulk)) { fprintf(stderr, "SQL error: writing table mtx of %s failed\n", db_file); goto done; }
    }
    {
        /* matrix.mtx.gz: header (the reference's "%%%M" prints "%%M" with glibc, src/bam2db_ds.c:500), dimensions, one line per entry */
        fastf_textbuf tb = {0};
        fastf_textbuf_reserve(&tb, 4096 + strlen(bam_file));
        tb.n += (size_t)snprintf(tb.p, tb.cap,
             "%%%%MatrixMarket matrix coordinate integer general\n%%metadata_json: \n%%{\n%%\t\"software_version\": \"fastF-1.0.0\",\n%%\t\"format_version\": 1,\n"
             "%%\t\"parent_bam\": \"%s\",\n%%\t\"rate_cell\": %.3f,\n%%\t\"rate_depth\": %.3f,\n%%\t\"total_n_FastQ\": %zu,\n%%\t\"sampled_n_FastQ\": %zu,\n"
             "%%\t\"sampled_valid_n_FastQ\": %zu\n%%}\n%zu %zu %zu\n",
             bam_file, rate_cell, rate_depth, (size_t)res->total, (size_t)res->sampled, (size_t)res->valid, (size_t)fkeys->n, (size_t)cells->n, (size_t)res->nnz);
        snprintf(path, sizeof path, "%s/matrix.mtx.gz", path_out);
        mtx_rows M = {res->m_gene, res->m_cell, res->m_count};
        const int wrc = fastf_gz_write_lines_parallel(path, tb.p, tb.n, res->nnz, mtx_line_fmt, &M);
        fastf_textbuf_free(&tb);
        if (wrc) { fprintf(stderr, "\x1b[31mError:\x1b[0m can not open file %s\n", path); goto done; }
    }
    phase("table mtx + matrix.mtx.gz");
    printf("matrix.mtx.gz is generated.\n");
    for (uint32_t i = 0; i < cells->n; i++) { gzwrite(file_barcode, cells->buf + cells->off[i], cells->off[i + 1] - cells->off[i]); gzputc(file_barcode, '\n'); }
    printf("barcodes.tsv.gz is generated.\n");
    for (uint32_t i = 0; i < fid->n; i++) {
        gzwrite(file_feature, fid->buf + fid->off[i], fid->off[i + 1] - fid->off[i]); gzputc(file_feature, '\t');
        gzwrite(file_feature, fname->buf + fname->off[i], fname->off[i + 1] - fname->off[i]); gzputc(file_feature, '\t');
        gzwrite(file_feature, ftype->buf + ftype->off[i], ftype->off[i + 1] - ftype->off[i]); gzputc(file_feature, '\n');
    }
    printf("features.tsv.gz is generated.\n");
    if (_umi_copies_flag) {
        /* numi: copies per distinct (cell, gene, umi) in (cell, gene, umi) order, NULL first (reference :527-556); decode_DNA(blob, 10) at :629.
         * The device sorts the rows and takes the run lengths (fastf_unique_counts_host); here the table and the text are laid out. */
        uint64_t nu = 0, *k = NULL;
        uint32_t *copies_of = NULL;
        if (fastf_unique_counts_host(ctx, rows, n_rows, res->bits_cell + res->bits_gene + res->bits_umi, &k, &copies_of, &nu)) { fprintf(stderr, "\x1b[31mError:\x1b[0m %s\n", fastf_last_error(ctx)); goto done; }
        fastf_sqlite_bulk *bulk = fastf_sqlite_bulk_begin(db_file, root_numi);
        if (!bulk) { free(k); free(copies_of); fprintf(stderr, "SQL error: cannot append to table numi of %s\n", db_file); goto done; }
        fastf_textbuf tb = {0};
        for (uint64_t i = 0; i < nu; i++) {
            int64_t cell, gene;
            uint8_t blob[8];
            uint64_t content = 0;
            const int nb = key_fields(k[i], bu, bg, mb, &cell, &gene, blob, &content);
            const int64_t copies = (int64_t)copies_of[i];
            /* columns: feature_index, cell_index, encoded_umi, n_copy -- the blob sits in the middle, so the row is laid out by hand */
            {
                const int64_t head[2] = {gene, cell};
                if (fastf_sqlite_bulk_row4(bulk, head, nb < 0 ? NULL : blob, nb < 0 ? 0u : (unsigned)nb, copies)) break;
            }
            char dec[16] = "NULL";
            if (nb >= 0) {
                for (int b = 0; b < 10; b++) { int sh = (int)(8 * mb) - 2 * (b + 1); dec[b] = "ACGT"[sh >= 0 ? (content >> sh) & 3 : 0]; }
                dec[10] = 0;
            }
            fastf_textbuf_reserve(&tb, 96);
            char *q = tb.p + tb.n;
            q += fastf_fmt_i64(q, gene); *q++ = '\t';
            q += fastf_fmt_i64(q, cell); *q++ = '\t';
            size_t dl = strlen(dec); memcpy(q, dec, dl); q += dl; *q++ = '\t';
            q += fastf_fmt_i64(q, copies); *q++ = '\n';
            tb.n = (size_t)(q - tb.p);
        }
        free(k);
        free(copies_of);
        if (fastf_sqlite_bulk_end(bulk)) { fastf_textbuf_free(&tb); fprintf(stderr, "SQL error: writing table numi of %s failed\n", db_file); goto done; }
        snprintf(path, sizeof path, "%s/umi.tsv.gz", path_out);
        const int wrc = fastf_gz_write_parallel(path, tb.p, tb.n);
        fastf_textbuf_free(&tb);
        if (wrc) { fprintf(stderr, "\x1b[31mError:\x1b[0m can not open file %s\n", path); goto done; }
        printf("umi.tsv.gz is generated.\n");
    }
    phase("barcodes / features (/ umi.tsv) gz");
    rc = 0;
done:
    if (file_barcode) gzclose(file_barcode);
    if (file_feature) gzclose(file_feature);
    return rc;
}

/* One cell table exactly as the reference builds it (reference :229-289): the sampled lines in order, the index stalling at the first
 * duplicate barcode.  gb is rewound first; returns 0, or 1 when fastf_sample_cells refuses the rate. */
static int sample_cell_table(gzFile gb, size_t n_cells, float rate_cell, unsigned seed, const char *barcodes_file, strlist *cells, uint64_t *d0)
{
    uint64_t *samp = (uint64_t *)malloc(sizeof(uint64_t) * (n_cells ? n_cells : 1));
    const uint64_t ns = samp ? fastf_sample_cells(n_cells, rate_cell, seed, samp, d0) : UINT64_MAX;
    if (ns == UINT64_MAX) { free(samp); printf("Sample size must be smaller than population size when sampling without replacement."); return 1; }
    printf("Actual number of sampled cell barcodes: %zu\n", (size_t)ns);
    gzrewind(gb);
    strset cset = {0};
    ss_init(&cset, cells, ns);
    char line[1024];
    size_t cell_index = 1, nth = 0;
    while (gzgets(gb, line, 1024) != NULL && cell_index <= ns) {
        nth++;
        if (nth - 1 != samp[cell_index - 1]) continue;
        line[strcspn(line, "\n\r\t")] = '\0';
        size_t n = strlen(line);
        if (!ss_has(&cset, line, n)) {
            sl_push(cells, line, n);
            ss_add(&cset, line, n, cells->n - 1);
            cell_index++;
        } else {
            printf("Warning: Duplicate cell barcodes were found in %s!\n", barcodes_file);
        }
    }
    free(cset.slot);
    free(samp);
    return 0;
}

/* tables cell and feature of one output set (reference :229-337) */
static int insert_lists(sqlite3 *db, const strlist *cells, const strlist *fid, const strlist *fname, const strlist *ftype)
{
    sqlite3_stmt *st = NULL;
    int rc = 1;
    exec_sql(db, "BEGIN TRANSACTION");
    sqlite3_prepare_v2(db, "INSERT INTO cell VALUES (?1);", -1, &st, NULL);
    for (uint32_t i = 0; i < cells->n; i++) {
        sqlite3_bind_text(st, 1, cells->buf + cells->off[i], (int)(cells->off[i + 1] - cells->off[i]), SQLITE_TRANSIENT);
        if (sqlite3_step(st) != SQLITE_DONE) { fprintf(stderr, "SQL error: %s\n", sqlite3_errmsg(db)); goto done; }
        sqlite3_reset(st);
    }
    exec_sql(db, "END TRANSACTION");
    sqlite3_finalize(st);
    st = NULL;
    exec_sql(db, "BEGIN TRANSACTION");
    sqlite3_prepare_v2(db, "INSERT INTO feature VALUES (?1, ?2, ?3);", -1, &st, NULL);
    for (uint32_t i = 0; i < fid->n; i++) {
        sqlite3_bind_text(st, 1, fid->buf + fid->off[i], (int)(fid->off[i + 1] - fid->off[i]), SQLITE_TRANSIENT);
        sqlite3_bind_text(st, 2, fname->buf + fname->off[i], (int)(fname->off[i + 1] - fname->off[i]), SQLITE_TRANSIENT);
        sqlite3_bind_text(st, 3, ftype->buf + ftype->off[i], (int)(ftype->off[i + 1] - ftype->off[i]), SQLITE_TRANSIENT);
        if (sqlite3_step(st) != SQLITE_DONE) { fprintf(stderr, "SQL error: %s\n", sqlite3_errmsg(db)); goto done; }
        sqlite3_reset(st);
    }
    exec_sql(db, "END TRANSACTION");
    rc = 0;
done:
    if (st) sqlite3_finalize(st);
    return rc;
}

/* the job's parameters: the cell table it parses against, the feature keys, and the sampling of the first rate (ignored by the sweep,
 * and d0 by the grid) */
static fastf_bam2db_params job_params(const strlist *cells, const strlist *fkeys, unsigned seed, uint64_t d0, float rate, uint32_t umi_bytes, uint32_t flags)
{
    static const uint32_t zero_off[1] = {0};
    fastf_bam2db_params p;
    memset(&p, 0, sizeof p);
    p.cell_keys = cells->buf ? cells->buf : ""; p.cell_off = cells->off ? cells->off : zero_off; p.n_cells = cells->n;
    p.gene_keys = fkeys->buf ? fkeys->buf : ""; p.gene_off = fkeys->off ? fkeys->off : zero_off; p.n_genes = fkeys->n;
    p.seed = seed; p.d0 = d0; p.keep_threshold = fastf_keep_threshold(rate);
    p.umi_max_bytes = umi_bytes;
    p.want_rows = 1;
    p.inflate_lanes = flags;
    return p;
}

int bam2db_run(char *bam_file, char **db_files, char **out_dirs, char *barcodes_file, char *features_file, uint32_t n_cell_rates, const char *const *cell_names,
               const float *cell_rates, uint32_t n_rates, const char *const *rate_names, const float *rates, unsigned int seed)
{
    int rc = 1;
    const int grid = n_cell_rates > 0, sweep = n_rates > 0;
    const uint32_t M = grid ? n_cell_rates : 1, K = sweep ? n_rates : 1, NS = M * K;   /* cell tables, depth rates, output sets */
    sqlite3 **dbs = (sqlite3 **)calloc(NS ? NS : 1, sizeof *dbs);
    fastf_ctx *ctx = NULL;
    fastf_bam2db_job *job = NULL;
    fastf_bam2db_result res;
    memset(&res, 0, sizeof res);
    fastf_bam2db_sweep_result *sres = sweep ? (fastf_bam2db_sweep_result *)calloc(M, sizeof *sres) : NULL;
    uint64_t *rate_rows = NULL, thr[FASTF_SWEEP_MAX_RATES];
    strlist *cells = (strlist *)calloc(M, sizeof *cells);
    strlist ucells = {0}, fkeys = {0}, fid = {0}, fname = {0}, ftype = {0};
    strset uset = {0}, fset = {0};
    uint64_t d0s[FASTF_GRID_MAX_CELL_RATES] = {0};
    uint32_t *remap = NULL;
    fastf_bam2db_cell_rate crs[FASTF_GRID_MAX_CELL_RATES];
    void *pin[2] = {NULL, NULL}, *map = MAP_FAILED;
    size_t map_n = 0;
    int bam = -1;
    gzFile gb = NULL, gf = NULL;
    char line[1024];
    {   /* also honoured when the reference's own main() is the caller (INTEGRATION.md section B) */
        const char *e = getenv("FASTF_GPUS");
        if (e && atoi(e) > 0) fastf_gpus = atoi(e);
        if ((e = getenv("FASTF_DEVICE")) != NULL) fastf_device = atoi(e);
    }
    if (!dbs || !cells || (sweep && !sres)) { fprintf(stderr, "\x1b[31mError:\x1b[0m out of host memory\n"); goto done; }
    if (grid && (!sweep || n_cell_rates > FASTF_GRID_MAX_CELL_RATES || fastf_gpus > 1)) {
        fprintf(stderr, "\x1b[31mError:\x1b[0m the cell-rate grid takes 1..%d cell rates and 1..%d depth rates on one GPU\n", FASTF_GRID_MAX_CELL_RATES, FASTF_SWEEP_MAX_RATES);
        goto done;
    }
    if (sweep && (n_rates > FASTF_SWEEP_MAX_RATES || fastf_gpus > 1)) { fprintf(stderr, "\x1b[31mError:\x1b[0m the depth sweep takes 1..%d rates on one GPU\n", FASTF_SWEEP_MAX_RATES); goto done; }
    for (uint32_t r = 0; r < K; r++) thr[r] = fastf_keep_threshold(rates[r]);

    g_t_last = 0;
    phase("start");
    for (uint32_t r = 0; r < NS; r++) {
        if (sqlite3_open(db_files[r], &dbs[r])) { fprintf(stderr, "Can't open database: %s\n", sqlite3_errmsg(dbs[r])); goto done; }
        fprintf(stderr, "Opened database successfully\n");
    }
    bam = open(bam_file, O_RDONLY);
    if (bam < 0) { fprintf(stderr, "Can't open BAM file %s\n", bam_file); goto done; }
    fprintf(stderr, "Opened BAM file %s successfully\n", bam_file);
    gb = gzopen(barcodes_file, "r");
    if (!gb) { fprintf(stderr, "Can't open cell barcode file %s\n", barcodes_file); goto done; }
    fprintf(stderr, "Opened cell barcode file %s successfully\n", barcodes_file);
    gf = gzopen(features_file, "r");
    if (!gf) { fprintf(stderr, "Can't open feature name file %s\n", features_file); goto done; }
    fprintf(stderr, "Opened feature name file %s successfully\n", features_file);
    for (uint32_t r = 0; r < NS; r++)
        if (exec_sql(dbs[r], "CREATE TABLE cell (cell_barcode TEXT);") || exec_sql(dbs[r], "CREATE TABLE feature (feature_id TEXT, feature_name TEXT, feature_type);") ||
            exec_sql(dbs[r], "CREATE TABLE umi (cell_index INTEGER, feature_index INTEGER, encoded_umi TEXT);")) goto done;

    /* ---- barcodes: count, then per cell rate sample + second pass (reference :229-289) ---- */
    size_t n_cells = 0;
    while (gzgets(gb, line, 1024) != NULL) n_cells++;
    printf("Total number of cells: %zu\n", n_cells);
    for (uint32_t i = 0; i < M; i++) {
        if (grid) printf("Cell rate %s:\n", cell_names[i]);
        if (sample_cell_table(gb, n_cells, cell_rates[i], seed, barcodes_file, &cells[i], &d0s[i])) goto done;
    }

    /* ---- features (reference :296-337): strtok on tabs, key = buffer up to its first NUL ---- */
    {
        size_t nlines = 0;
        while (gzgets(gf, line, 1024) != NULL) nlines++;
        gzrewind(gf);
        ss_init(&fset, &fkeys, nlines);
    }
    while (gzgets(gf, line, 1024) != NULL) {
        char *id = strtok(line, "\t"), *name = strtok(NULL, "\t"), *type = strtok(NULL, "\t");
        if (!id || !name || !type) { fprintf(stderr, "\x1b[31mError:\x1b[0m feature line with fewer than three tab-separated fields in %s\n", features_file); goto done; }
        type[strcspn(type, "\n\r\t")] = '\0';
        size_t kn = strlen(line);
        if (!ss_has(&fset, line, kn)) {
            sl_push(&fkeys, line, kn);
            ss_add(&fset, line, kn, fkeys.n - 1);
            sl_push(&fid, id, strlen(id)); sl_push(&fname, name, strlen(name)); sl_push(&ftype, type, strlen(type));
        } else {
            printf("Warning: Duplicate feature names were found in %s!\n", features_file);
        }
    }
    for (uint32_t r = 0; r < NS; r++)
        if (insert_lists(dbs[r], &cells[r / K], &fid, &fname, &ftype)) goto done;

    /* the cell table the device job parses against: the one table, or the union of the grid's tables with a remap per cell rate */
    const strlist *jcells = &cells[0];
    if (grid) {
        size_t tot = 0;
        for (uint32_t i = 0; i < M; i++) tot += cells[i].n;
        ss_init(&uset, &ucells, tot);
        for (uint32_t i = 0; i < M; i++)
            for (uint32_t k = 0; k < cells[i].n; k++) {
                const char *c = cells[i].buf + cells[i].off[k];
                const size_t n = cells[i].off[k + 1] - cells[i].off[k];
                if (!ss_has(&uset, c, n)) { sl_push(&ucells, c, n); ss_add(&uset, c, n, ucells.n - 1); }
            }
        remap = (uint32_t *)calloc((size_t)M * (ucells.n ? ucells.n : 1), sizeof(uint32_t));
        if (!remap) { fprintf(stderr, "\x1b[31mError:\x1b[0m out of host memory\n"); goto done; }
        for (uint32_t i = 0; i < M; i++) {
            crs[i].cell_index = remap + (size_t)i * ucells.n;
            crs[i].n_cells = cells[i].n;
            crs[i].d0 = d0s[i];
            for (uint32_t k = 0; k < cells[i].n; k++)
                remap[(size_t)i * ucells.n + ss_has(&uset, cells[i].buf + cells[i].off[k], cells[i].off[k + 1] - cells[i].off[k]) - 1] = k + 1;
        }
        jcells = &ucells;
    }

    /* ---- the hot path: device job fed with the raw BGZF bytes ---- */
    printf("Start to convert bam file to sqlite3 database...\n");
    fflush(stdout);
    phase("lists + small tables");
    if (fastf_gpus > 1) {
        /* several GPUs of this node: contiguous block shards, global draw ordinals, NCCL all-to-all by cell (csrc/sharded.cu) */
        struct stat sb;
        if (fstat(bam, &sb) || sb.st_size <= 0) { fprintf(stderr, "\x1b[31mError:\x1b[0m cannot stat %s\n", bam_file); goto done; }
        map_n = (size_t)sb.st_size;
        if ((map = mmap(NULL, map_n, PROT_READ, MAP_PRIVATE, bam, 0)) == MAP_FAILED) { fprintf(stderr, "\x1b[31mError:\x1b[0m cannot map %s\n", bam_file); goto done; }
        madvise(map, map_n, MADV_SEQUENTIAL);
    } else if (fastf_ctx_create(fastf_device, &ctx)) { fprintf(stderr, "\x1b[31mError:\x1b[0m %s\n", fastf_last_error(NULL)); goto done; }
    /* 10x UMIs are 10 or 12 bases: retried once with room for 16.  Records that cross BGZF blocks (htsjdk / STAR writers): retried once
     * on one GPU with FASTF_BAM_STRADDLE, record starts guessed and verified per block (whole file in one chunk). */
    for (uint32_t umi_bytes = 3, flags = 0;;) {
        const fastf_bam2db_params p = job_params(jcells, &fkeys, seed, d0s[0], rates[0], umi_bytes, flags);
        int failed;
        if (fastf_gpus > 1) {
            failed = fastf_bam2db_run_sharded(fastf_gpus, NULL, &p, map, map_n, &res);
        } else if (!(failed = (grid ? fastf_bam2db_begin_grid : fastf_bam2db_begin)(ctx, &p, &job))) {
            const size_t PIECE = (size_t)256 << 20;
            if (!pin[0] && (fastf_host_alloc(ctx, PIECE, &pin[0]) || fastf_host_alloc(ctx, PIECE, &pin[1]))) { fprintf(stderr, "\x1b[31mError:\x1b[0m %s\n", fastf_last_error(ctx)); goto done; }
            ssize_t got;
            off_t at = 0;
            int which = 0;
            while (!failed && (got = fastf_pread_parallel(bam, pin[which], PIECE, at)) > 0) {   /* several readers: one fread() cannot feed PCIe */
                failed = fastf_bam2db_feed(job, pin[which], (size_t)got);
                at += got;
                which ^= 1;
            }
            if (!failed && got < 0) { fprintf(stderr, "\x1b[31mError:\x1b[0m reading %s failed\n", bam_file); goto done; }
            if (!failed && grid) failed = fastf_bam2db_finish_grid(job, M, crs, K, thr, sres);
            else if (!failed && sweep) failed = fastf_bam2db_finish_sweep(job, K, thr, sres);
            else if (!failed) failed = fastf_bam2db_finish(job, &res);
        }
        if (!failed) break;
        char err[1024];
        snprintf(err, sizeof err, "%s", fastf_gpus > 1 ? fastf_sharded_last_error() : fastf_last_error(ctx));
        if (job) { fastf_bam2db_job_free(job); job = NULL; }
        fastf_bam2db_result_free(&res);
        for (uint32_t i = 0; sweep && i < M; i++) fastf_bam2db_sweep_result_free(&sres[i]);
        if (umi_bytes == 3 && strstr(err, "umi-too-long")) { umi_bytes = 4; continue; }
        if (!flags && fastf_gpus == 1 && strstr(err, "record-straddles-bgzf-block")) { flags = FASTF_BAM_STRADDLE; continue; }
        fprintf(stderr, "\x1b[31mError:\x1b[0m %s\n", err);
        if (fastf_gpus > 1 && strstr(err, "record-straddles-bgzf-block")) fprintf(stderr, "(records cross BGZF blocks: not an htslib-written file; run it on one GPU, FASTF_GPUS=1)\n");
        goto done;
    }
    if (!ctx && _umi_copies_flag && fastf_ctx_create(fastf_device, &ctx)) { fprintf(stderr, "\x1b[31mError:\x1b[0m %s\n", fastf_last_error(NULL)); goto done; }

    /* ---- one output set per (cell rate i, depth rate r); a single-rate run is set (0, 0): the job's result and all its rows ---- */
    phase("device job (ctx, read, feed, finish)");
    for (uint32_t i = 0; i < M; i++) {
        const fastf_bam2db_sweep_result *sr = sweep ? &sres[i] : NULL;
        if (sr) {
            free(rate_rows);
            rate_rows = (uint64_t *)malloc(sizeof(uint64_t) * (sr->n_rows ? sr->n_rows : 1));
            if (!rate_rows) { fprintf(stderr, "\x1b[31mError:\x1b[0m out of host memory\n"); goto done; }
        }
        for (uint32_t r = 0; r < K; r++) {
            const fastf_bam2db_result *rr = &res;
            const uint64_t *rows = res.row_keys;
            uint64_t n = res.n_rows;
            if (sr) {   /* table umi of rate r: the rows whose smallest keeping threshold is <= its own, in file order */
                rr = &sr->rate[r];
                rows = rate_rows;
                n = 0;
                for (uint64_t k = 0; k < sr->n_rows; k++)
                    if (thr[sr->row_rate[k]] <= thr[r]) rate_rows[n++] = sr->row_keys[k];
            }
            if (grid) printf("Cell rate %s, depth rate %s -> %s\n", cell_names[i], rate_names[r], out_dirs[i * K + r]);
            else if (sweep) printf("Depth rate %s -> %s\n", rate_names[r], out_dirs[r]);
            if (write_outputs(&dbs[i * K + r], db_files[i * K + r], bam_file, out_dirs[i * K + r], cell_rates[i], rates[r], rr, rows, n, &cells[i], &fkeys, &fid, &fname, &ftype,
                              ctx)) goto done;
        }
    }
    rc = 0;
done:
    for (uint32_t r = 0; dbs && r < NS; r++)
        if (dbs[r]) sqlite3_close(dbs[r]);
    free(dbs);
    if (gb) gzclose(gb);
    if (gf) gzclose(gf);
    if (map != MAP_FAILED) munmap(map, map_n);
    if (bam >= 0) close(bam);
    fastf_bam2db_result_free(&res);
    if (sres) { for (uint32_t i = 0; i < M; i++) fastf_bam2db_sweep_result_free(&sres[i]); free(sres); }
    free(rate_rows);
    free(remap);
    if (job) fastf_bam2db_job_free(job);
    if (ctx) { fastf_host_free(ctx, pin[0]); fastf_host_free(ctx, pin[1]); fastf_ctx_destroy(ctx); }
    for (uint32_t i = 0; cells && i < M; i++) sl_free(&cells[i]);
    free(cells);
    free(uset.slot); free(fset.slot);
    sl_free(&ucells); sl_free(&fkeys); sl_free(&fid); sl_free(&fname); sl_free(&ftype);
    return rc;
}

int bam2db(char *bam_file, char *db_file, char *path_out, char *barcodes_file, char *features_file, float rate_cell, float rate_depth, unsigned int seed)
{
    return bam2db_run(bam_file, &db_file, &path_out, barcodes_file, features_file, 0, NULL, &rate_cell, 0, NULL, &rate_depth, seed);
}
