/* fastF (B200 build): the reference's command line for the GPU subcommands (reference src/main.c:30-92, 231-402, 404-443).
 *   fastF bam2db  -b BAM -f FEATURES -a BARCODES -d DB -c RATE_CELL -r RATE_DEPTH [-o OUT] [-s SEED] [-u]
 *   fastF bam2db  -b BAM -f FEATURES -a BARCODES -d DB -c RATE_CELL --depths R1,R2,... [-o OUT] [-s SEED] [-u]
 *                 (the depth sweep, not a reference option: one pass, rate Ri written into OUT/depth_<Ri>/ with database OUT/depth_<Ri>/<basename of DB>)
 *   fastF bam2db  -b BAM -f FEATURES -a BARCODES -d DB --cells C1,C2,... (-r RATE_DEPTH | --depths R1,R2,...) [-o OUT] [-s SEED] [-u]
 *                 (the cell-rate grid, not a reference option: one pass, set (Ci, Rj) written into OUT/cell_<Ci>/ with -r, into
 *                 OUT/cell_<Ci>/depth_<Rj>/ with --depths; database <that directory>/<basename of DB>)
 *   fastF freq    -R R1 -o OUT [-l LEN] [-u UMI]
 *   fastF crb     -b BAM -o OUT.gz
 *   fastF extract -b BAM -t TAG [-T 0|1]
 * Long options (--bam --feature --barcode --dbname --cell --depth --out --seed --umicopies; --R1 --out --len --umi; --tag --type) as
 * in the reference.  filter is not part of this build (out of scope: see DESIGN.md). */
#include "fastf_host.h"
#include "../../include/fastf_gpu.h"
#include <errno.h>
#include <stdlib.h>
#include <string.h>
#include <sys/stat.h>
#include <unistd.h>
#include <zlib.h>

typedef struct { char s; const char *l; int has_arg; } optdef;
/* returns the option index or -1; *val gets the argument ("-x VAL", "-xVAL", "--long VAL", "--long=VAL") */
static int next_opt(int argc, const char **argv, int *i, const optdef *defs, int ndefs, const char **val)
{
    const char *a = argv[*i];
    *val = NULL;
    if (a[0] != '-' || !a[1]) { fprintf(stderr, "error: unknown option `%s`\n", a); exit(1); }
    for (int k = 0; k < ndefs; k++) {
        if (a[1] == '-') {
            size_t n = strlen(defs[k].l);
            if (strncmp(a + 2, defs[k].l, n) || (a[2 + n] && a[2 + n] != '=')) continue;
            if (defs[k].has_arg) {
                if (a[2 + n] == '=') *val = a + 3 + n;
                else if (*i + 1 < argc) *val = argv[++*i];
                else { fprintf(stderr, "error: option `--%s` requires a value\n", defs[k].l); exit(1); }
            }
            return k;
        }
        if (a[1] == defs[k].s) {
            if (defs[k].has_arg) {
                if (a[2]) *val = a + 2;
                else if (*i + 1 < argc) *val = argv[++*i];
                else { fprintf(stderr, "error: option `-%c` requires a value\n", defs[k].s); exit(1); }
            }
            return k;
        }
    }
    fprintf(stderr, "error: unknown option `%s`\n", a);
    exit(1);
}

static int cmd_freq(int argc, const char **argv)
{
    const char *r1 = NULL, *out = NULL;
    size_t l = 16, u = 10;   /* reference src/main.c:35-36 */
    static const optdef defs[] = {{'R', "R1", 1}, {'o', "out", 1}, {'l', "len", 1}, {'u', "umi", 1}, {'h', "help", 0}};
    for (int i = 1; i < argc; i++) {
        const char *v;
        switch (next_opt(argc, argv, &i, defs, 5, &v)) {
        case 0: r1 = v; break;
        case 1: out = v; break;
        case 2: l = (size_t)(int)strtol(v, NULL, 0); break;   /* argparse OPT_INTEGER stores through an int* (src/argparse.c:85-100) */
        case 3: u = (size_t)(int)strtol(v, NULL, 0); break;
        default: printf("Usage: fastF freq -R R1.fastq.gz -o OUTDIR [-l 16] [-u 10]\n\nFind all the cell barcode whitelist and their frequencies.\n"); exit(0);
        }
    }
    if (!r1) { fprintf(stderr, "Please specify the path to R1 fastq files.\n"); exit(1); }
    if (access(r1, F_OK) == -1) { fprintf(stderr, "Cannot open file %s \n", r1); exit(1); }
    char path[2048];
    snprintf(path, sizeof path, "%s/whitelist.txt", out ? out : "(null)");
    FILE *fp = fopen(path, "w");
    if (!fp) { fprintf(stderr, "Cannot open file %s \n", path); exit(1); }
    int rc = freq_whitelist(r1, l, u, fp);
    fclose(fp);
    return rc;
}

#define MAX_DEPTHS 32   /* FASTF_SWEEP_MAX_RATES = FASTF_GRID_MAX_CELL_RATES */

/* "R1,R2,..." of option `opt` -> names (pointers into *copy, strdup'ed) and float values as -r / -c read them; exits on what is refused */
static uint32_t parse_rates(const char *list, const char *opt, char **copy, char **names, float *rates)
{
    uint32_t n = 0;
    *copy = strdup(list);
    for (char *save = NULL, *t = strtok_r(*copy, ",", &save); t; t = strtok_r(NULL, ",", &save)) {
        if (n == MAX_DEPTHS) { fprintf(stderr, "\x1b[31mError:\x1b[0m %s takes at most %d rates.\n", opt, MAX_DEPTHS); exit(1); }
        names[n] = t;
        rates[n] = strtof(t, NULL);
        for (uint32_t k = 0; k < n; k++)
            if (!strcmp(names[k], t) || !memcmp(&rates[k], &rates[n], sizeof(float))) { fprintf(stderr, "\x1b[31mError:\x1b[0m %s lists the rate %s twice.\n", opt, t); exit(1); }
        n++;
    }
    if (!n) { fprintf(stderr, "\x1b[31mError:\x1b[0m %s needs at least one rate.\n", opt); exit(1); }
    return n;
}

/* bam2db() lets FASTF_GPUS override --gpus: refuse either before any directory is made */
static void one_gpu_only(const char *opt)
{
    const char *e = getenv("FASTF_GPUS");
    if (fastf_gpus > 1 || (e && atoi(e) > 1)) { fprintf(stderr, "\x1b[31mError:\x1b[0m %s runs on one GPU (--gpus 1, FASTF_GPUS unset or 1).\n", opt); exit(1); }
}

/* <dir>/<basename of db>: exits when it exists */
static char *fresh_db(const char *dir, const char *db)
{
    const char *base = strrchr(db, '/') ? strrchr(db, '/') + 1 : db;
    char *p = (char *)malloc(strlen(dir) + strlen(base) + 2);
    sprintf(p, "%s/%s", dir, base);
    if (access(p, F_OK) != -1) { fprintf(stderr, "\x1b[31mError:\x1b[0m database: %s already exists, change the name of database in -d argument!\n", p); exit(1); }
    return p;
}

static char *subdir(const char *parent, const char *prefix, const char *name)
{
    char *p = (char *)malloc(strlen(parent) + strlen(prefix) + strlen(name) + 2);
    sprintf(p, "%s/%s%s", parent, prefix, name);
    return p;
}

/* --depths and/or --cells: one device pass, one output set per (cell rate, depth rate) (bam2db_run).  The cell axis is the --cells list
 * (cell_list) or the one -c rate, the depth axis the --depths list (depth_list) or the one -r rate.  Set (Ci, Rj) goes to
 * OUT[/cell_<Ci>][/depth_<Rj>]/, a level for each list.  Everything refused is refused before any directory is made. */
static int rate_sets(const char *bam, const char *feat, const char *bc, const char *db, const char *out, const char *cell_list, float rate_cell, const char *rate_cell_text,
                     const char *depth_list, float rate_depth, const char *rate_depth_text, unsigned seed)
{
    char *cnames[MAX_DEPTHS], *dnames[MAX_DEPTHS], *ccopy = NULL, *dcopy = NULL;
    float crates[MAX_DEPTHS], drates[MAX_DEPTHS];
    uint32_t m = 1, k = 1;
    if (cell_list) m = parse_rates(cell_list, "--cells", &ccopy, cnames, crates);
    else { cnames[0] = (char *)rate_cell_text; crates[0] = rate_cell; }
    if (depth_list) k = parse_rates(depth_list, "--depths", &dcopy, dnames, drates);
    else { dnames[0] = (char *)rate_depth_text; drates[0] = rate_depth; }
    one_gpu_only(cell_list ? "--cells" : "--depths");
    {   /* a cell rate the reference's SampleInt refuses */
        gzFile g = gzopen(bc, "r");
        char line[1024];
        size_t n_cells = 0;
        while (g && gzgets(g, line, 1024) != NULL) n_cells++;
        if (g) gzclose(g);
        uint64_t *samp = (uint64_t *)malloc(sizeof(uint64_t) * (n_cells ? n_cells : 1)), d0 = 0;
        for (uint32_t i = 0; i < m; i++)
            if (fastf_sample_cells(n_cells, crates[i], seed, samp, &d0) == UINT64_MAX) {
                fprintf(stderr, "\x1b[31mError:\x1b[0m cell rate %s: Sample size must be smaller than population size when sampling without replacement.\n", cnames[i]);
                exit(1);
            }
        free(samp);
    }
    char **cdirs = (char **)malloc(sizeof(char *) * m), **dirs = (char **)malloc(sizeof(char *) * m * k), **dbs = (char **)malloc(sizeof(char *) * m * k);
    for (uint32_t i = 0; i < m; i++) {
        cdirs[i] = cell_list ? subdir(out, "cell_", cnames[i]) : strdup(out);
        for (uint32_t j = 0; j < k; j++) {
            dirs[i * k + j] = depth_list ? subdir(cdirs[i], "depth_", dnames[j]) : strdup(cdirs[i]);
            dbs[i * k + j] = fresh_db(dirs[i * k + j], db);
        }
    }
    for (uint32_t i = 0; i < m; i++) {
        if (cell_list && mkdir(cdirs[i], 0777) && errno != EEXIST) { fprintf(stderr, "\x1b[31mError:\x1b[0m can not create directory %s\n", cdirs[i]); exit(1); }
        for (uint32_t j = 0; j < k && depth_list; j++)
            if (mkdir(dirs[i * k + j], 0777) && errno != EEXIST) { fprintf(stderr, "\x1b[31mError:\x1b[0m can not create directory %s\n", dirs[i * k + j]); exit(1); }
    }
    const int rc = bam2db_run((char *)bam, dbs, dirs, (char *)bc, (char *)feat, cell_list ? m : 0, (const char *const *)cnames, crates, k, (const char *const *)dnames, drates, seed);
    for (uint32_t i = 0; i < m * k; i++) { free(dirs[i]); free(dbs[i]); }
    for (uint32_t i = 0; i < m; i++) free(cdirs[i]);
    free(cdirs); free(dirs); free(dbs); free(ccopy); free(dcopy);
    if (rc) { fprintf(stderr, "\x1b[31mError:\x1b[0m bam2db failed.\n"); return 1; }
    return 0;
}

static int cmd_bam2db(int argc, const char **argv)
{
    const char *bam = NULL, *feat = NULL, *bc = NULL, *db = NULL, *out = ".", *depths = NULL, *cells = NULL, *rate_cell_text = "0", *rate_depth_text = NULL;
    float rate_cell = 0.0f, rate_depth = 0.0f;   /* the reference leaves these uninitialised (src/main.c:293-294): pass -c and -r */
    int have_r = 0, have_c = 0;
    unsigned seed = 926;
    static const optdef defs[] = {{'b', "bam", 1}, {'f', "feature", 1}, {'a', "barcode", 1}, {'d', "dbname", 1}, {'c', "cell", 1}, {'r', "depth", 1}, {'o', "out", 1}, {'s', "seed", 1}, {'u', "umicopies", 0}, {'h', "help", 0}, {'g', "gpus", 1}, {0, "depths", 1}, {0, "cells", 1}};
    for (int i = 1; i < argc; i++) {
        const char *v;
        switch (next_opt(argc, argv, &i, defs, 13, &v)) {
        case 0: bam = v; break;
        case 1: feat = v; break;
        case 2: bc = v; break;
        case 3: db = v; break;
        case 4: rate_cell = strtof(v, NULL); rate_cell_text = v; have_c = 1; break;     /* OPT_FLOAT uses strtof (src/argparse.c:101-116) */
        case 5: rate_depth = strtof(v, NULL); rate_depth_text = v; have_r = 1; break;
        case 6: out = v; break;
        case 7: seed = (unsigned)(int)strtol(v, NULL, 0); break;
        case 8: _umi_copies_flag = 1; break;
        case 10: fastf_gpus = (int)strtol(v, NULL, 0); break;   /* not a reference option: GPUs of this node to shard the BAM over */
        case 11: depths = v; break;                              /* not a reference option: the depth sweep */
        case 12: cells = v; break;                               /* not a reference option: the cell-rate grid */
        default: printf("Usage: fastF bam2db -b BAM -f FEATURES -a BARCODES -d DB -c RATE_CELL -r RATE_DEPTH [-o OUT] [-s 926] [-u] [--gpus N]\n"
                        "       fastF bam2db -b BAM -f FEATURES -a BARCODES -d DB -c RATE_CELL --depths R1,R2,... [-o OUT] [-s 926] [-u]\n"
                        "       fastF bam2db -b BAM -f FEATURES -a BARCODES -d DB --cells C1,C2,... (-r RATE_DEPTH | --depths R1,R2,...) [-o OUT] [-s 926] [-u]\n\n"
                        "Filter bam file with desired cell proportion and read depth, then summarise it into UMI matrix.\n"
                        "--depths writes the result of every rate Ri (up to 32, one pass over the BAM) into OUT/depth_<Ri>/, database OUT/depth_<Ri>/<basename of DB>.\n"
                        "--cells writes the result of every cell rate Ci (up to 32, one pass over the BAM) into OUT/cell_<Ci>/ (with -r) or, for every depth\n"
                        "rate Rj, into OUT/cell_<Ci>/depth_<Rj>/ (with --depths); database <that directory>/<basename of DB>.\n"); exit(0);
        }
    }
    if (depths && have_r) { fprintf(stderr, "\x1b[31mError:\x1b[0m -r/--depth and --depths exclude each other.\n"); exit(1); }
    if (cells && have_c) { fprintf(stderr, "\x1b[31mError:\x1b[0m -c/--cell and --cells exclude each other.\n"); exit(1); }
    if (cells && !depths && !have_r) { fprintf(stderr, "\x1b[31mError:\x1b[0m --cells needs -r or --depths.\n"); exit(1); }
    if (!bam || access(bam, F_OK) == -1) { fprintf(stderr, "\x1b[31mError:\x1b[0m bam file: %s does not exist.\n", bam ? bam : "(null)"); exit(1); }
    if (!feat || access(feat, F_OK) == -1) { fprintf(stderr, "\x1b[31mError:\x1b[0m feature file: %s does not exist.\n", feat ? feat : "(null)"); exit(1); }
    if (!bc || access(bc, F_OK) == -1) { fprintf(stderr, "\x1b[31mError:\x1b[0m barcode file: %s does not exist.\n", bc ? bc : "(null)"); exit(1); }
    if (!db) { fprintf(stderr, "\x1b[31mError:\x1b[0m please name the database with -d.\n"); exit(1); }
    if (cells || depths) return rate_sets(bam, feat, bc, db, out, cells, rate_cell, rate_cell_text, depths, rate_depth, rate_depth_text, seed);
    if (access(db, F_OK) != -1) { fprintf(stderr, "\x1b[31mError:\x1b[0m database: %s already exists, change the name of database in -d argument!\n", db); exit(1); }
    if (bam2db((char *)bam, (char *)db, (char *)out, (char *)bc, (char *)feat, rate_cell, rate_depth, seed)) { fprintf(stderr, "\x1b[31mError:\x1b[0m bam2db failed.\n"); return 1; }
    return 0;
}

static int cmd_crb(int argc, const char **argv)
{
    const char *bam = NULL, *out = ".";   /* reference default (src/main.c:234): gzopen(".") fails */
    static const optdef defs[] = {{'b', "bam", 1}, {'o', "out", 1}, {'h', "help", 0}};
    for (int i = 1; i < argc; i++) {
        const char *v;
        switch (next_opt(argc, argv, &i, defs, 3, &v)) {
        case 0: bam = v; break;
        case 1: out = v; break;
        default: printf("Usage: fastF crb -b BAM -o OUT.gz\n\nExtract CR and CB tags from bam file and summarize them with frequencies to a tsv file.\n"); exit(0);
        }
    }
    if (!bam) { fprintf(stderr, "\x1b[31mError:\x1b[0m path to bam file can not been NULL while extracting .\n"); exit(1); }
    gzFile fo = gzopen(out, "w");
    if (!fo) { fprintf(stderr, "\x1b[31mError:\x1b[0m can not open file %s\n", out); exit(1); }
    int rc = crb_write((char *)bam, fo);
    gzclose(fo);
    if (!rc) printf("Done.\n");
    return rc;
}

static int cmd_extract(int argc, const char **argv)
{
    const char *bam = NULL, *tag = NULL;
    int type = 0;
    static const optdef defs[] = {{'b', "bam", 1}, {'t', "tag", 1}, {'T', "type", 1}, {'h', "help", 0}};
    for (int i = 1; i < argc; i++) {
        const char *v;
        switch (next_opt(argc, argv, &i, defs, 4, &v)) {
        case 0: bam = v; break;
        case 1: tag = v; break;
        case 2: type = (int)strtol(v, NULL, 0); break;
        default: printf("Usage: fastF extract -b BAM -t TAG [-T 0|1]\n\nExtract the tag of bam file.\n"); exit(0);
        }
    }
    if (!bam || access(bam, F_OK) == -1) { fprintf(stderr, "\x1b[31mError:\x1b[0m bam file: %s does not exist.\n", bam ? bam : "(null)"); exit(1); }
    if (!tag) { fprintf(stderr, "\x1b[31mError:\x1b[0m --tag is required.\n"); exit(1); }
    return extract_bam((char *)bam, tag, type);
}

static void leave(int rc)
{
    fflush(stdout);
    fflush(stderr);
    _exit(rc & 0xff);
}

int main(int argc, const char **argv)
{
    const char *dev = getenv("FASTF_DEVICE");
    if (dev) fastf_device = atoi(dev);
    const char *gpus = getenv("FASTF_GPUS");
    if (gpus) fastf_gpus = atoi(gpus);
    if (argc < 2 || !strcmp(argv[1], "-h") || !strcmp(argv[1], "--help")) {
        printf("Usage: fastF [-h] <command> [<args>]\n\nCommands (GPU build): freq, bam2db, crb, extract\n");
        return argc < 2 ? -1 : 0;
    }
    /* Every file is written and closed when a command returns.  Leaving through _exit() skips the CUDA runtime's exit handlers
     * (tearing the primary context down costs a few hundred ms to seconds of a run that takes a few seconds in all). */
    if (!strcmp(argv[1], "freq")) leave(cmd_freq(argc - 1, argv + 1));
    if (!strcmp(argv[1], "bam2db")) leave(cmd_bam2db(argc - 1, argv + 1));
    if (!strcmp(argv[1], "crb")) leave(cmd_crb(argc - 1, argv + 1));
    if (!strcmp(argv[1], "extract")) leave(cmd_extract(argc - 1, argv + 1));
    if (!strcmp(argv[1], "filter")) { fprintf(stderr, "fastF (B200 build): `%s` is not part of this build; use the reference binary.\n", argv[1]); return 1; }
    return 0;   /* the reference silently ignores unknown commands (src/main.c:437-442) */
}
