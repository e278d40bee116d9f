/*
 * wdpmcl_b200 - command-line host of the B200-native WDPM redistribution solver.
 *
 * Drop-in for the reference executable WDPMCL (/root/reference/src/WDPMCL.c): same
 * command line and parameter-file grammar (:308-531), same ESRI ASCII reader and
 * writer (:533-593, :1533-1599), same printed report (:1616-1857), same
 * 1000-iteration convergence cadence and stop tests (:1054-1377), same exit codes
 * (42 usage / missing water file, 1 set-up failure, 255 runtime device failure).
 * What changes is the solver: every block runs on the GPU through the C ABI of
 * libwdpm_b200 (include/wdpm_b200.h); grids are uploaded once and stay resident,
 * the water grid comes back only for a scratch file or the final output.
 *
 * The two backend selectors of the reference command line ("0 serial / 1 OpenCL",
 * "0 OpenCL CPU / 1 OpenCL GPU") are parsed at their positions; whatever they say,
 * the CUDA solver runs - there is no CPU path - and the report says so. The first
 * picks the arithmetic, as it does in the reference, where the two branches differ
 * in Subtract and Drain (DESIGN.md §4): "cpu" = 0 runs the serial branch's
 * (WDPM_SCHEDULE_SERIAL), any other value the OpenCL branch's (runoff.cl). The
 * second flag (OpenCL device kind) is ignored.
 *
 * Extension: `wdpmcl_b200 chain paramfile1 paramfile2 ...` runs several modules in ONE process (the
 * reference's validate_WDPM.sh:77-99 runs Add -> Drain -> Subtract as three). Each module prints its
 * usual report and writes its usual files; what is saved is the hand-over: a DEM named again is not
 * parsed again, and a water file that is the previous module's output is not read back - on one GPU
 * the grids go from solver to solver inside HBM (wdpm_copy_state) and the water gets the "%f"
 * quantisation a file would have given it (wdpm_quantize_water; include/wdpm_quantize.h), so every
 * output is byte-identical to what the separate runs write (tests/test_cli.py).
 *
 * Environment: WDPM_B200_DEVICE (first CUDA ordinal, default 0), WDPM_B200_KERNEL
 * (0 auto, 1 colour, 2 fused, 3 resident), WDPM_B200_GPUS (number of GPUs, default 1:
 * the DEM is cut into that many row stripes, one solver per GPU, halos exchanged over
 * NVLink by the library; results do not depend on the count).
 *
 * Extension, Drain modules only (chained ones too): WDPM_B200_OUTLETS replaces the reference's single outlet
 * (the lowest cell with dem > 0) by a set of outlets, each with its own drained total (wdpm_set_outlets):
 *   WDPM_B200_OUTLETS=rim     every cell with dem > nodata in the first or last row or column of the DEM;
 *   WDPM_B200_OUTLETS=<path>  an ESRI ASCII grid of the DEM's ncols and nrows: every cell whose value is > 0
 *                             and not the grid's NODATA value is an outlet.
 * Outlets are taken in row-major order. Fewer than one, more than WDPM_MAX_OUTLETS, an outlet on a cell with
 * dem <= nodata, a grid of another size, or a set of more than one outlet with cpu=0 (the serial branch drains
 * one outlet) print a message and exit with 1. Each total starts at max(water at its outlet, 0)
 * (wdpm_seed_outlet_drains, WDPMCL.c:1029 per outlet). The report prints "Drain outlets:" and the lowest
 * outlet elevation instead of the drain column, row and elevation; "Volume drained" is the sum of the totals
 * in outlet order. WDPM_B200_OUTLET_TOTALS=<path> also writes one CSV line per outlet at the end, in outlet
 * order: row,col,elevation_m,drained_m3 (1-based padded coordinates, values as %.17g).
 *
 * Extension, not under chain: exact checkpoints (wdpm_checkpoint_arm / wdpm_checkpoint_wait; file format at
 * ck_header). WDPM_B200_CHECKPOINT=<path> writes one every WDPM_B200_CHECKPOINT_EVERY blocks (default 1) and one at
 * the end; a "%d" in the path becomes the iteration count. Mid-run ones are captured at the start of the next block
 * and written by a thread while it runs; the thread is joined before the next capture, so checkpoints are never
 * skipped and a slow disk holds the run up. WDPM_B200_RESUME=<path> continues the run the file was written by, bit
 * for bit: water, outlet totals, iteration count, drained total and initial volume come from it, the add or
 * subtract step is skipped. A file that is missing, damaged or written by a run of another identity prints a
 * message and exits with 1 before any solver exists.
 */
#define _POSIX_C_SOURCE 200809L
#include <ctype.h>
#include <errno.h>
#include <fcntl.h>
#include <math.h>
#include <pthread.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <sys/stat.h>
#include <sys/time.h>
#include <unistd.h>

#ifdef _OPENMP
#include <omp.h>
#endif

#include "wdpm_b200.h"
#include "wdpm_quantize.h"

enum { BLOCK_ITERATIONS = 1000 }; /* IterationNum, WDPMCL.c:597 */
enum { EXIT_USAGE = 42 };

typedef struct {
    char module[32];
    char dem[512], water[512], output[512], scratch[512];
    double depth_mm;     /* add / subtract */
    double runoff_frac;  /* add */
    double eltol_mm;
    double drain_tol;    /* drain, m3 */
    int backend, device_kind; /* the reference's "cpu" and "gpu" flags */
    double thres_mm;
    int iter_limit;
} run_args;

typedef struct {
    char name[6][104];
    double value[6];
    int ncols, nrows;
    double cellsize, nodata;
} asc_header;

static int is_module(const char *s) { return !strcmp(s, "add") || !strcmp(s, "subtract") || !strcmp(s, "drain"); }
static void line(const char *s) { printf("%s\n", s); }

/* ---- usage texts (WDPMCL.c:1658-1745) ------------------------------------ */

static void usage_module(const char *module)
{
    line("                                          ");
    line("Program arguments in order of specification");
    if (!strcmp(module, "add")) line("Add module specified");
    else if (!strcmp(module, "subtract")) line("Subtract module specified");
    else if (!strcmp(module, "drain")) line("Drain module specified");
    line("DEM file name (string) ");
    line(!strcmp(module, "add") ? "Water file name (string) - Optional, Use NULL to omit" : "Water file name (string)");
    line("Output file name (string)");
    line("Scratch file name (string) - Optional, use NULL to omit");
    if (!strcmp(module, "add")) {
        line("Depth of water to add (mm) (real)");
        line("Water runoff fraction (real)");
        line("Elevation tolerance (mm) (real)");
    } else if (!strcmp(module, "subtract")) {
        line("Depth of water to remove (mm) (real)");
        line("Elevation tolerance (mm) (real)");
    } else if (!strcmp(module, "drain")) {
        line("Elevation tolerance (mm) (real)");
        line("Drain tolerance (m3) (real)");
    }
    line("Specify 0 for serial CPU and 1 for opencl ");
    line("Specify 0 for OpenCL CPU and 1 for opencl GPU ");
    line("Zero depth threshold (mm) (real)");
    line("Maximum number of iterations (integer) - Optional, Use 0 to omit ");
    line("                                          ");
}

static void usage_all(void)
{
    static const char *const add[] = {"Module name: add", "DEM file name (string)",
        "Water file name (string) - Optional, use --NULL-- to omit", "Output file name (string)",
        "Scratch file name (string) - Optional, use --NULL-- to omit", "Depth of water to add (mm) (real)",
        "Water runoff fraction (real)", "Elevation tolerance (mm) (real)", "Specify 0 for serial CPU and 1 for opencl ",
        "Specify 0 for OpenCL CPU and 1 for opencl GPU ", "Zero depth threshold (mm) (real) ",
        "Maximum number of iterations (integer) - Optional, Use 0 to omit", "                                          ",
        "                                          ", NULL};
    static const char *const sub[] = {"Module name: subtract", "Path and Name of Report file", "DEM file name (string)",
        "Water file name (string)", "Output file name (string)", "Scratch file name (string) - Optional, use --NULL-- to omit",
        "Depth of water to remove (mm) (real)", "Elevation tolerance (mm) (real)", "Specify 0 for serial CPU and 1 for opencl ",
        "Specify 0 for OpenCL CPU and 1 for opencl GPU ", "Zero depth threshold (mm) (real) ",
        "Maximum number of iterations (integer) - Optional, Use 0 to omit ", "                                          ",
        "                                          ", NULL};
    static const char *const drn[] = {"Module name: drain", "Path and Name of Report file", "DEM file name (string)",
        "Water file name (string) ", "Output file name (string)", "Scratch file name (string) - Optional, use --NULL-- to omit",
        "Elevation tolerance (mm) (real)", "Drain tolerance (m3) (real)", "Specify 0 for serial CPU and 1 for opencl ",
        "Specify 0 for OpenCL CPU and 1 for opencl GPU ", "Zero depth threshold (mm) (real) ",
        "Maximum number of iterations (integer) - Optional, Use 0 to omit", "                                          ", NULL};
    const char *const *sets[] = {add, sub, drn};
    for (int k = 0; k < 3; k++)
        for (const char *const *p = sets[k]; *p; p++) line(*p);
}

/* ---- banner and parameter echo (WDPMCL.c:1616-1655, :1748-1797) ----------- */

static void banner(const char *module)
{
    static const char blank[] = "                                                                   ";
    line(blank); line(blank);
    line("Wetland DEM Ponding Model version 2.0");
    line("Copyright (c) 2010, 2012, 2014, 2020 Kevin Shook, Centre for Hydrology");
    line("Developed by Oluwaseun Sharomi, Raymond Spiteri and Tonghe Liu");
    line("Numerical Simulation Laboratory, University of Saskatchewan.\n");
    line("--------------------------------------------------------------------");
    line(blank);
    line("This program is free software: you can redistribute it and/or modify");
    line("it under the terms of the GNU General Public License as published by");
    line("the Free Software Foundation, either version 3 of the License, or");
    line("(at your option) any later version.");
    line(blank);
    line("This program is distributed in the hope that it will be useful,");
    line("but WITHOUT ANY WARRANTY; without even the implied warranty of");
    line("MERCHANTABILITY or FITNESS FOR A PARTICULAR PURPOSE.  See the");
    line("GNU General Public License for more details.");
    line(blank);
    line("You should have received a copy of the GNU General Public License");
    line("along with this program.  If not, see <http://www.gnu.org/licenses/>.");
    line(blank);
    if (!strcmp(module, "add")) {
        line("This program adds water to an ArcGIS ASCII file of water runoff");
        line("and redistributes water over the DEM");
    } else if (!strcmp(module, "subtract")) {
        line("This program removes a depth water to an ArcGIS ASCII file of water depths");
        line("and redistributes water over the DEM");
    } else if (!strcmp(module, "drain")) {
        line("This program drains an ArcGIS ASCII file of water runoff");
        line("from the lowest point in the DEM, which acts as a drain");
    }
    line("From the algorithm of Shapiro, M., & Westervelt, J. (1992). ");
    line("An Algebra for GIS and Image Processing (pp. 1-22).");
    line(blank); line(blank);
}

static void echo_args(const run_args *a)
{
    printf("%30s\n", "WDPM Parameters");
    printf("%30s %s\n", "Function used:", a->module);
    printf("%30s %s\n", "DEM file:", a->dem);
    printf("%30s %s\n", "Water file:", a->water);
    printf("%30s %s\n", "Output file:", a->output);
    printf("%30s %s\n", "Scratch file:", a->scratch);
    if (!strcmp(a->module, "add")) {
        printf("%30s %0.4f %s\n", "Water added:", a->depth_mm, "mm");
        printf("%30s %0.4f\n", "Runoff fraction:", a->runoff_frac);
    }
    if (!strcmp(a->module, "subtract")) printf("%30s %0.4f %s\n", "Water subtracted:", a->depth_mm, "mm");
    printf("%30s %0.4f %s\n", "Elevation tolerance:", a->eltol_mm, "mm");
    if (!strcmp(a->module, "drain")) printf("%30s %0.4f %s\n", "Drain tolerance:", a->drain_tol, "m3");
    printf("%30s %0.4f %s\n", "Zero depth threshold:", a->thres_mm, "mm");
    if (a->iter_limit == 0) printf("%30s\n", "No iteration limitation is set");
    else printf("%30s %d\n", "Maximum number of iterations:", a->iter_limit);
    line("               ");
    /* the reference prints which OpenCL/serial backend the two flags select (:1781-1796);
     * here the first one selects the arithmetic only */
    printf("%41s\n", "Using CUDA (sm_100a) for Computation");
    if (a->backend == 0) printf("%40s\n", "serial-branch arithmetic on CUDA");
    else printf("%40s\n", "backend flags accepted and ignored");
}

/* ---- arguments: positional argv or a whitespace-token parameter file ------- */

static int tokens_from_file(const char *path, char tok[][512], int max)
{
    FILE *f = fopen(path, "r");
    if (!f) return -1;
    int n = 0;
    while (n < max && fscanf(f, "%511s", tok[n]) == 1) n++;
    fclose(f);
    return n;
}

/* v[0] = module, v[1..] = its arguments in the reference's order */
static int fill_args(run_args *a, int n, char v[][512])
{
    memset(a, 0, sizeof *a);
    snprintf(a->module, sizeof a->module, "%s", v[0]);
    const int need = !strcmp(a->module, "add") ? 12 : 11;
    if (!is_module(a->module) || n < need) return -1;
    int k = 1;
    snprintf(a->dem, sizeof a->dem, "%s", v[k++]);
    snprintf(a->water, sizeof a->water, "%s", v[k++]);
    snprintf(a->output, sizeof a->output, "%s", v[k++]);
    snprintf(a->scratch, sizeof a->scratch, "%s", v[k++]);
    if (!strcmp(a->module, "add")) {
        a->depth_mm = atof(v[k++]);
        a->runoff_frac = atof(v[k++]);
        a->eltol_mm = atof(v[k++]);
    } else if (!strcmp(a->module, "subtract")) {
        a->depth_mm = atof(v[k++]);
        a->eltol_mm = atof(v[k++]);
    } else {
        a->eltol_mm = atof(v[k++]);
        a->drain_tol = atof(v[k++]);
    }
    a->backend = (int)atof(v[k++]);
    a->device_kind = (int)atof(v[k++]);
    a->thres_mm = atof(v[k++]);
    a->iter_limit = (int)atof(v[k++]);
    return 0;
}

static int is_null_name(const char *s)
{
    return strlen(s) == 4 && toupper((unsigned char)s[0]) == 'N' && toupper((unsigned char)s[1]) == 'U' &&
           toupper((unsigned char)s[2]) == 'L' && toupper((unsigned char)s[3]) == 'L';
}

static int file_exists(const char *p) { struct stat st; return stat(p, &st) == 0; }

/* ---- ESRI ASCII grids ------------------------------------------------------ */

static char *slurp(const char *path, size_t *len)
{
    FILE *f = fopen(path, "rb");
    if (!f) return NULL;
    fseek(f, 0, SEEK_END);
    long n = ftell(f);
    rewind(f);
    char *buf = malloc((size_t)n + 1);
    if (!buf || fread(buf, 1, (size_t)n, f) != (size_t)n) { fclose(f); free(buf); return NULL; }
    fclose(f);
    buf[n] = 0;
    if (len) *len = (size_t)n;
    return buf;
}

/* six "name value" pairs, positional (WDPMCL.c:542-555); returns a pointer past them */
static const char *parse_header(const char *p, asc_header *h)
{
    for (int i = 0; i < 6; i++) {
        int used = 0;
        if (sscanf(p, " %100s%n", h->name[i], &used) != 1) return NULL;
        p += used;
        char *end;
        h->value[i] = strtod(p, &end);
        if (end == p) return NULL;
        p = end;
    }
    h->ncols = (int)h->value[0];
    h->nrows = (int)h->value[1];
    h->cellsize = h->value[4];
    h->nodata = h->value[5];
    return p;
}

/* Parallel text -> double. The data section is cut into one byte range per thread; a token belongs
 * to the range its first character lies in. Pass 1 counts tokens per range, a prefix sum gives each
 * range its output offset, pass 2 converts with strtod - the conversion fscanf("%lf") itself uses
 * (WDPMCL.c:1569-1574, :1592-1597), so every value is bit-identical to the reference's reader. */
static int is_space(char c) { return c == ' ' || c == '\n' || c == '\t' || c == '\r' || c == '\f' || c == '\v'; }

static size_t parse_values(const char *p, const char *end, double *g, size_t n)
{
    int nt = 1;
#ifdef _OPENMP
    nt = omp_get_max_threads();
#endif
    const size_t len = (size_t)(end - p);
    if (len < (size_t)1 << 16) nt = 1;
    size_t *count = calloc((size_t)nt + 1, sizeof *count);
    if (!count) return 0;
#pragma omp parallel num_threads(nt)
    {
        int t = 0;
#ifdef _OPENMP
        t = omp_get_thread_num();
#endif
        const char *lo = p + len * (size_t)t / (size_t)nt, *hi = p + len * (size_t)(t + 1) / (size_t)nt;
        size_t c = 0;
        for (const char *q = lo; q < hi; q++)
            if (!is_space(*q) && (q == p || is_space(q[-1]))) c++;
        count[t + 1] = c;
#pragma omp barrier
#pragma omp single
        for (int i = 0; i < nt; i++) count[i + 1] += count[i];
        size_t k = count[t];
        for (const char *q = lo; q < hi && k < n; q++) {
            if (!is_space(*q) && (q == p || is_space(q[-1]))) {
                char *stop;
                g[k++] = strtod(q, &stop);
                if (stop > q) q = stop - 1;
            }
        }
    }
    const size_t total = count[nt];
    free(count);
    return total < n ? total : n;
}

/* rows*cols values in row-major order after the header; missing values stay as `fill` */
static double *read_grid(const char *path, int rows, int cols, double fill, asc_header *hdr_out)
{
    size_t len = 0;
    char *buf = slurp(path, &len);
    if (!buf) return NULL;
    asc_header h;
    const char *p = parse_header(buf, &h);
    if (!p) { free(buf); return NULL; }
    if (hdr_out) *hdr_out = h;
    const size_t n = (size_t)rows * (size_t)cols;
    double *g = malloc(n * sizeof *g);
    if (!g) { free(buf); return NULL; }
    size_t k = parse_values(p, buf + len, g, n);
    for (; k < n; k++) g[k] = fill;
    free(buf);
    return g;
}

/* write_gis, WDPMCL.c:1533-1554: "%f " per value, header formats as there. Rows are formatted in
 * parallel into per-thread buffers (the same printf conversion, so the bytes are the reference's)
 * and written out in order. */
static int write_grid(const char *path, const asc_header *h, const double *g)
{
    FILE *f = fopen(path, "w");
    if (!f) return -1;
    fprintf(f, "%s %d\n", h->name[0], (int)h->value[0]);
    fprintf(f, "%s %d\n", h->name[1], (int)h->value[1]);
    fprintf(f, "%s %14.6f\n", h->name[2], h->value[2]);
    fprintf(f, "%s %14.6f\n", h->name[3], h->value[3]);
    fprintf(f, "%s %9.6f\n", h->name[4], h->value[4]);
    fprintf(f, "%s %14.6f\n", h->name[5], h->value[5]);
    int nt = 1;
#ifdef _OPENMP
    nt = omp_get_max_threads();
#endif
    if (h->nrows < nt) nt = h->nrows > 0 ? h->nrows : 1;
    char **bufs = calloc((size_t)nt, sizeof *bufs);
    size_t *used = calloc((size_t)nt, sizeof *used);
    int failed = !bufs || !used;
#pragma omp parallel num_threads(nt) if (!failed)
    {
        int t = 0;
#ifdef _OPENMP
        t = omp_get_thread_num();
#endif
        const int r0 = (int)((long long)h->nrows * t / nt), r1 = (int)((long long)h->nrows * (t + 1) / nt);
        size_t cap = (size_t)(r1 - r0) * ((size_t)h->ncols * 12 + 2) + 512, u = 0;
        char *b = malloc(cap);
        for (int r = r0; r < r1 && b; r++) {
            const double *row = g + (size_t)r * h->ncols;
            for (int c = 0; c < h->ncols; c++) {
                if (cap - u < 400) { /* "%f" of a huge double can take ~320 characters */
                    cap = cap * 2 + 1024;
                    char *nb = realloc(b, cap);
                    if (!nb) { free(b); b = NULL; break; }
                    b = nb;
                }
                u += (size_t)snprintf(b + u, cap - u, "%f ", row[c]);
            }
            if (b) b[u++] = '\n';
        }
        bufs[t] = b;
        used[t] = u;
        if (!b && r1 > r0) {
#pragma omp atomic write
            failed = 1;
        }
    }
    for (int t = 0; t < nt && !failed; t++)
        if (bufs[t] && fwrite(bufs[t], 1, used[t], f) != used[t]) failed = 1;
    if (bufs) for (int t = 0; t < nt; t++) free(bufs[t]);
    free(bufs);
    free(used);
    if (fclose(f) != 0) failed = 1;
    return failed ? -1 : 0;
}

/* ---- drain outlet sets (WDPM_B200_OUTLETS) ------------------------------------ */

typedef struct {
    int32_t n;
    int32_t *row, *col; /* 1-based padded coordinates, row-major order */
} outlet_set;

static void outlets_fail(const char *spec, const char *why)
{
    fprintf(stderr, "Couldn't use the drain outlets WDPM_B200_OUTLETS=%s: %s\n", spec, why);
    exit(1);
}

/* The set WDPM_B200_OUTLETS names, checked against the DEM before any solver exists. */
static void load_outlets(const char *spec, const double *dem, int rows, int cols, double nodata, outlet_set *os)
{
    const size_t n = (size_t)rows * (size_t)cols;
    unsigned char *is_out = calloc(n, 1);
    if (!is_out) outlets_fail(spec, "out of memory");
    if (!strcmp(spec, "rim")) {
        for (int i = 0; i < rows; i++)
            for (int j = 0; j < cols; j++)
                if (i == 0 || i == rows - 1 || j == 0 || j == cols - 1) is_out[(size_t)i * cols + j] = dem[(size_t)i * cols + j] > nodata;
    } else {
        char *hb = slurp(spec, NULL);
        asc_header h;
        if (!hb || !parse_header(hb, &h)) outlets_fail(spec, "not a readable ESRI ASCII grid");
        free(hb);
        if (h.ncols != cols || h.nrows != rows) outlets_fail(spec, "its ncols and nrows differ from the DEM's");
        double *g = read_grid(spec, rows, cols, 0.0, NULL);
        if (!g) outlets_fail(spec, "not a readable ESRI ASCII grid");
        for (size_t k = 0; k < n; k++) is_out[k] = g[k] > 0 && g[k] != h.nodata;
        free(g);
    }
    size_t cnt = 0;
    for (size_t k = 0; k < n; k++) {
        if (!is_out[k]) continue;
        if (!(dem[k] > nodata)) outlets_fail(spec, "an outlet lies on a cell with dem <= nodata");
        cnt++;
    }
    if (cnt == 0) outlets_fail(spec, "no outlet");
    if (cnt > WDPM_MAX_OUTLETS) outlets_fail(spec, "more outlets than WDPM_MAX_OUTLETS");
    os->n = (int32_t)cnt;
    os->row = malloc(cnt * sizeof *os->row);
    os->col = malloc(cnt * sizeof *os->col);
    if (!os->row || !os->col) outlets_fail(spec, "out of memory");
    cnt = 0;
    for (size_t k = 0; k < n; k++)
        if (is_out[k]) {
            os->row[cnt] = (int32_t)(k / (size_t)cols) + 1;
            os->col[cnt] = (int32_t)(k % (size_t)cols) + 1;
            cnt++;
        }
    free(is_out);
}

/* ---- run ------------------------------------------------------------------- */

static double seconds_since(const struct timeval *t0)
{
    struct timeval t;
    gettimeofday(&t, NULL);
    return (double)(t.tv_usec - t0->tv_usec) / 1000000 + (double)(t.tv_sec - t0->tv_sec);
}

static void die_solver(const char *what)
{
    printf("error: %s with CUDA solver error (%s)\n", what, wdpm_last_error());
    exit(-1); /* as exitOnFail, WDPMCL.c:225-232 */
}

/* ---- one solver, or one stripe solver per GPU ------------------------------- */

enum { MAX_GPUS = 16, ENQUEUE_CHUNK = 50, CK_HANDOVER_ITERATIONS = 200 };

typedef struct {
    int n;                       /* solvers (1 = plain solver, >1 = row stripes) */
    wdpm_solver *sv[MAX_GPUS];
    int32_t band_row0[MAX_GPUS], band_rows[MAX_GPUS], owned_row0[MAX_GPUS], owned_rows[MAX_GPUS];
} solver_set;

static void set_create(solver_set *ss, wdpm_config base, int want)
{
    const int rows = base.rows, padded = rows + 2, triples = (padded + 2) / 3;
    int n = want;
    if (n > MAX_GPUS) n = MAX_GPUS;
    if (n > wdpm_device_count() - base.device) n = wdpm_device_count() - base.device;
    while (n > 1 && padded < 9 * n) n--; /* a stripe needs at least 9 rows (3 * n triples are too few when the last is partial) */
    if (n < 1) n = 1;
    memset(ss, 0, sizeof *ss);
    ss->n = n;
    for (int g = 0; g < n; g++) {
        wdpm_config cfg = base;
        cfg.device = base.device + g;
        if (n > 1) { /* bands of padded rows starting at multiples of 3, as equal as possible */
            const int t0 = (int)((long long)triples * g / n), t1 = (int)((long long)triples * (g + 1) / n);
            cfg.stripe_row0 = 3 * t0;
            cfg.stripe_rows = (3 * t1 < padded ? 3 * t1 : padded) - 3 * t0;
            cfg.kernel = WDPM_KERNEL_FUSED;
        }
        if (wdpm_create(&cfg, &ss->sv[g]) != WDPM_OK) {
            fprintf(stderr, "Couldn't create the CUDA solver: %s\n", wdpm_last_error());
            exit(1);
        }
        if (n > 1) {
            if (wdpm_stripe_band(ss->sv[g], &ss->band_row0[g], &ss->band_rows[g], &ss->owned_row0[g], &ss->owned_rows[g]) != WDPM_OK)
                die_solver("query stripe band");
        } else {
            ss->band_rows[g] = ss->owned_rows[g] = rows;
        }
    }
    if (n > 1) {
        static wdpm_stripe_endpoint ep[MAX_GPUS];
        for (int g = 0; g < n; g++)
            if (wdpm_stripe_export(ss->sv[g], &ep[g]) != WDPM_OK) die_solver("export stripe");
        for (int g = 0; g < n; g++)
            if (wdpm_stripe_connect(ss->sv[g], g > 0 ? &ep[g - 1] : NULL, g + 1 < n ? &ep[g + 1] : NULL) != WDPM_OK)
                die_solver("connect stripes");
    }
}

static void set_upload(solver_set *ss, const double *dem, const double *water, int cols)
{
    for (int g = 0; g < ss->n; g++) {
        const size_t off = (size_t)ss->band_row0[g] * (size_t)cols;
        const int rc = ss->n == 1 ? wdpm_upload(ss->sv[g], dem, water)
                                  : wdpm_stripe_upload(ss->sv[g], dem + off, water + off, ss->band_row0[g], ss->band_rows[g]);
        if (rc != WDPM_OK) die_solver("upload grids");
    }
}

static void set_download(solver_set *ss, double *water, int cols)
{
    for (int g = 0; g < ss->n; g++)
        if (wdpm_download_water(ss->sv[g], water + (size_t)ss->owned_row0[g] * (size_t)cols) != WDPM_OK) die_solver("read water");
}

typedef struct ck_writer ck_writer;
static void ck_hand_over(solver_set *ss, ck_writer *cw);

/* One block of `iters` iterations on every stripe; results combined in stripe order. With `cw`, the solvers are
 * armed: their capture lands while the first CK_HANDOVER_ITERATIONS run, and the host waits for it and hands it to
 * the writer before feeding the rest. That many queued iterations keep every GPU busy during the wait (at 32768²
 * on one GPU they take 1.4 s, the capture of 8.6 GB lands in 0.17 s), and the writer still has most of the
 * block to write the file before the next capture is due. */
static void set_run_block(solver_set *ss, int iters, wdpm_block_result *out, ck_writer *cw)
{
    if (ss->n == 1 && !cw) {
        if (wdpm_run_block(ss->sv[0], iters, out) != WDPM_OK) die_solver("run block");
        return;
    }
    for (int g = 0; g < ss->n; g++)
        if (wdpm_block_begin(ss->sv[g]) != WDPM_OK) die_solver("begin block");
    int handed = !cw;
    for (int done = 0; done < iters;) { /* feed all GPUs round-robin: nothing here blocks */
        int nit = ss->n > 1 ? ENQUEUE_CHUNK : handed ? iters - done : CK_HANDOVER_ITERATIONS;
        if (nit > iters - done) nit = iters - done;
        for (int g = 0; g < ss->n; g++)
            if (wdpm_block_enqueue(ss->sv[g], nit) != WDPM_OK) die_solver("enqueue iterations");
        done += nit;
        if (!handed && (done >= CK_HANDOVER_ITERATIONS || done == iters)) {
            ck_hand_over(ss, cw);
            handed = 1;
        }
    }
    if (ss->n == 1) {
        if (wdpm_block_end(ss->sv[0], out) != WDPM_OK) die_solver("end block");
        return;
    }
    memset(out, 0, sizeof *out);
    for (int g = 0; g < ss->n; g++) {
        wdpm_block_result r;
        if (wdpm_block_end(ss->sv[g], &r) != WDPM_OK) die_solver("end block");
        if (r.max_diff > out->max_diff) out->max_diff = r.max_diff;
        out->masked_sum += r.masked_sum;
        out->total_drain += r.total_drain;
        out->wet_cells += r.wet_cells;
        out->launches += r.launches;
        out->iterations = r.iterations;
    }
}

/* Scratch (checkpoint) files are written by a background thread while the GPUs run the next block
 * (the reference writes them inline, WDPMCL.c:1290-1372). The thread owns its own copy of the grid. */
typedef struct {
    pthread_t thread;
    int running;
    char path[512];
    asc_header hdr;
    double *grid;
} scratch_writer;

static void *scratch_main(void *arg)
{
    scratch_writer *sw = arg;
    write_grid(sw->path, &sw->hdr, sw->grid);
    return NULL;
}

static void scratch_join(scratch_writer *sw)
{
    if (sw->running) {
        pthread_join(sw->thread, NULL);
        sw->running = 0;
    }
}

/* hands `grid` (n values) to the writer: copied, so the caller may overwrite it at once */
static void scratch_start(scratch_writer *sw, const char *path, const asc_header *h, const double *grid, size_t n)
{
    scratch_join(sw);
    if (!sw->grid) sw->grid = malloc(n * sizeof *sw->grid);
    if (!sw->grid) { write_grid(path, h, grid); return; }
    memcpy(sw->grid, grid, n * sizeof *grid);
    snprintf(sw->path, sizeof sw->path, "%s", path);
    sw->hdr = *h;
    if (pthread_create(&sw->thread, NULL, scratch_main, sw) == 0) sw->running = 1;
    else write_grid(path, h, grid);
}

/* what the scratch file and the Add output hold: water with NODATA cells marked (WDPMCL.c:1336-1344, :1386-1392) */
static void mark_nodata(double *w, const double *dem, size_t n, double nodata)
{
    for (size_t k = 0; k < n; k++)
        if (dem[k] <= nodata) w[k] = nodata;
}

/* ---- exact checkpoints (WDPM_B200_CHECKPOINT, WDPM_B200_RESUME) -----------------------------------------------
 * The only code that knows the file format. Little-endian, in this order:
 *   ck_header (128 bytes): magic, version, the run's identity, then where the run stands;
 *   n_totals doubles: every outlet's drained total (depth in m, as the solver keeps it) in outlet order;
 *   rows*cols doubles: the water, raw fp64 bits, row-major: the state the next block starts from;
 *   a uint64 trailer: the water's order-free checksum (wdpm_water_checksum's definition).
 * A checkpoint resumes only a run of the same identity: the DEM (size, nodata, georeference and a hash of its
 * values' bits), module, schedule ("cpu" flag), depth, runoff fraction, zero threshold and outlet set. The elevation
 * and drain tolerances, the iteration limit, paths, the GPU count and the kernel are free to change. */
#define CK_MAGIC "WDPMCKPT"
enum { CK_VERSION = 1 };

typedef struct {
    char magic[8];
    uint32_t version;
    int32_t module;                   /* WDPM_ADD / WDPM_SUBTRACT / WDPM_DRAIN */
    int32_t rows, cols;
    double nodata, cellsize, xll, yll;
    uint64_t dem_hash;                /* ck_checksum of the DEM's fp64 bits */
    int32_t schedule;                 /* WDPM_SCHEDULE_*, from the "cpu" flag */
    int32_t n_totals;                 /* Drain: outlets (1 for the reference's outlet); 0 otherwise */
    double depth, runoff_frac, thres; /* m, fraction, m */
    uint64_t outlet_hash;             /* 0: the reference's outlet, or not Drain */
    int64_t iterations;
    double initial_vol, total_drain;  /* m3; m (the report's old_drain of the next block) */
} ck_header;
_Static_assert(sizeof(ck_header) == 128, "checkpoint header layout");

/* sum of bits(g[k]) * (2 * (index0 + k) + 1) mod 2^64: equal sums over any partition of the same grid */
static uint64_t ck_checksum(const double *g, size_t n, size_t index0)
{
    uint64_t sum = 0;
#pragma omp parallel for reduction(+ : sum) schedule(static)
    for (long long k = 0; k < (long long)n; k++) {
        uint64_t b;
        memcpy(&b, &g[k], sizeof b);
        sum += b * (2 * ((uint64_t)index0 + (uint64_t)k) + 1);
    }
    return sum;
}

static uint64_t ck_outlet_hash(const outlet_set *os)
{
    if (os->n == 0) return 0;
    uint64_t h = 1469598103934665603ull; /* FNV-1a over the (row, col) pairs in outlet order */
    for (int32_t k = 0; k < os->n; k++) {
        const int32_t v[2] = {os->row[k], os->col[k]};
        const unsigned char *p = (const unsigned char *)v;
        for (size_t b = 0; b < sizeof v; b++) h = (h ^ p[b]) * 1099511628211ull;
    }
    return h ? h : 1;
}

static void ck_identity(ck_header *h, const asc_header *hdr, const double *dem, int module, int schedule, double depth,
                        double runoff_frac, double thres, const outlet_set *os)
{
    memset(h, 0, sizeof *h);
    memcpy(h->magic, CK_MAGIC, sizeof h->magic);
    h->version = CK_VERSION;
    h->module = module;
    h->rows = hdr->nrows;
    h->cols = hdr->ncols;
    h->nodata = hdr->nodata;
    h->cellsize = hdr->cellsize;
    h->xll = hdr->value[2];
    h->yll = hdr->value[3];
    h->dem_hash = ck_checksum(dem, (size_t)hdr->nrows * (size_t)hdr->ncols, 0);
    h->schedule = schedule;
    h->n_totals = module == WDPM_DRAIN ? (os->n > 0 ? os->n : 1) : 0;
    h->depth = depth;
    h->runoff_frac = runoff_frac;
    h->thres = thres;
    h->outlet_hash = ck_outlet_hash(os);
}

/* `pattern` with its first "%d" replaced by the iteration count */
static void ck_path(char *out, size_t cap, const char *pattern, long long k)
{
    const char *p = strstr(pattern, "%d");
    if (p) snprintf(out, cap, "%.*s%lld%s", (int)(p - pattern), pattern, k, p + 2);
    else snprintf(out, cap, "%s", pattern);
}

/* One checkpoint to write: the water arrives in pieces of whole rows (a stripe's owned rows each, straight from the
 * solvers' capture staging, or one piece for the whole grid) and each goes to its offset in the file. */
struct ck_writer {
    pthread_t thread;
    int running, failed; /* failed: the errno of a failed write */
    char path[1024];
    ck_header h;
    double *totals; /* h.n_totals */
    int n_pieces;
    const double *piece[MAX_GPUS];
    int32_t row0[MAX_GPUS], nrows[MAX_GPUS];
};

static int pwrite_all(int fd, const void *buf, size_t len, off_t off)
{
    const char *p = buf;
    while (len > 0) {
        const ssize_t w = pwrite(fd, p, len < ((size_t)1 << 30) ? len : ((size_t)1 << 30), off);
        if (w <= 0) {
            if (w == 0) errno = EIO; /* no progress: a full device reports ENOSPC on the next call, but do not spin */
            return -1;
        }
        p += w;
        len -= (size_t)w;
        off += w;
    }
    return 0;
}

/* A temporary file, fsync, then rename: the file at the path is always a complete checkpoint. Returns 0, or the
 * errno of the first call that failed. */
static int ck_write(ck_writer *cw)
{
    const ck_header *h = &cw->h;
    char tmp[1100];
    snprintf(tmp, sizeof tmp, "%s.tmp", cw->path);
    const int fd = open(tmp, O_WRONLY | O_CREAT | O_TRUNC, 0644);
    if (fd < 0) return errno ? errno : EIO;
    const off_t water_at = (off_t)sizeof *h + (off_t)h->n_totals * (off_t)sizeof(double);
    uint64_t sum = 0;
    int err = 0;
#define CK_CALL(ok) do { if (!err && !(ok)) err = errno ? errno : EIO; } while (0) /* later calls skipped once one fails */
    CK_CALL(pwrite_all(fd, h, sizeof *h, 0) == 0);
    CK_CALL(pwrite_all(fd, cw->totals, (size_t)h->n_totals * sizeof(double), (off_t)sizeof *h) == 0);
    for (int p = 0; p < cw->n_pieces && !err; p++) {
        const size_t cells = (size_t)cw->nrows[p] * (size_t)h->cols, first = (size_t)cw->row0[p] * (size_t)h->cols;
        CK_CALL(pwrite_all(fd, cw->piece[p], cells * sizeof(double), water_at + (off_t)(first * sizeof(double))) == 0);
        sum += ck_checksum(cw->piece[p], cells, first);
    }
    CK_CALL(pwrite_all(fd, &sum, sizeof sum, water_at + (off_t)((size_t)h->rows * (size_t)h->cols * sizeof(double))) == 0);
    CK_CALL(fsync(fd) == 0);
    if (close(fd) != 0 && !err) err = errno ? errno : EIO;
    CK_CALL(rename(tmp, cw->path) == 0);
#undef CK_CALL
    if (err) unlink(tmp);
    return err;
}

static void *ck_main(void *arg)
{
    ck_writer *cw = arg;
    cw->failed = ck_write(cw);
    return NULL;
}

/* Checkpoints are never skipped: a writer still busy when the next one is due holds the run up. */
static void ck_join(ck_writer *cw)
{
    if (cw->running) {
        pthread_join(cw->thread, NULL);
        cw->running = 0;
    }
    if (cw->failed) {
        fprintf(stderr, "Couldn't write the checkpoint %s: %s\n", cw->path, strerror(cw->failed));
        exit(1);
    }
}

static void ck_start(ck_writer *cw)
{
    if (pthread_create(&cw->thread, NULL, ck_main, cw) == 0) cw->running = 1;
    else ck_main(cw);
}

/* Every solver's capture has landed: the writer takes their staging as it is (each stripe's rows go to their offset)
 * and the totals added over the stripes (each lives on the stripe that owns its outlet and reads 0 on the others). */
static void ck_hand_over(solver_set *ss, ck_writer *cw)
{
    for (int32_t q = 0; q < cw->h.n_totals; q++) cw->totals[q] = 0.0;
    for (int g = 0; g < ss->n; g++) {
        const void *w;
        const double *t;
        int32_t nt;
        if (wdpm_checkpoint_wait(ss->sv[g], &w, &t, &nt) != WDPM_OK) die_solver("wait for the checkpoint capture");
        cw->piece[g] = w;
        cw->row0[g] = ss->owned_row0[g];
        cw->nrows[g] = ss->owned_rows[g];
        for (int32_t q = 0; q < cw->h.n_totals && q < nt; q++) cw->totals[q] += t[q];
    }
    cw->n_pieces = ss->n;
    ck_start(cw);
}

static void ck_fail(const char *path, const char *why)
{
    fprintf(stderr, "Couldn't resume from the checkpoint WDPM_B200_RESUME=%s: %s\n", path, why);
    exit(1);
}

/* Read the checkpoint at `path` into h, *totals (allocated) and water (rows*cols), refusing any file that is not a
 * complete, intact checkpoint of a run with the identity `want`. */
static void ck_read(const char *path, const ck_header *want, ck_header *h, double **totals, double *water)
{
    FILE *f = fopen(path, "rb");
    if (!f) ck_fail(path, strerror(errno));
    if (fread(h, sizeof *h, 1, f) != 1) ck_fail(path, "truncated file");
    if (memcmp(h->magic, CK_MAGIC, sizeof h->magic) != 0) ck_fail(path, "not a checkpoint file (wrong magic)");
    if (h->version != CK_VERSION) ck_fail(path, "unsupported checkpoint version");
#define CK_SAME(field) (memcmp(&h->field, &want->field, sizeof h->field) == 0)
    if (!CK_SAME(rows) || !CK_SAME(cols) || !CK_SAME(nodata) || !CK_SAME(cellsize) || !CK_SAME(xll) || !CK_SAME(yll) || !CK_SAME(dem_hash))
        ck_fail(path, "it was written for another DEM");
    if (!CK_SAME(module)) ck_fail(path, "it was written by another module");
    if (!CK_SAME(schedule)) ck_fail(path, "it was written with another cpu flag (update schedule)");
    if (!CK_SAME(depth) || !CK_SAME(runoff_frac)) ck_fail(path, "it was written with another depth or runoff fraction");
    if (!CK_SAME(thres)) ck_fail(path, "it was written with another zero depth threshold");
    if (!CK_SAME(n_totals) || !CK_SAME(outlet_hash)) ck_fail(path, "it was written with other drain outlets (WDPM_B200_OUTLETS)");
#undef CK_SAME
    if (h->iterations < 0 || h->iterations > INT32_MAX - 2 * BLOCK_ITERATIONS) ck_fail(path, "iteration count out of range");
    const size_t n = (size_t)h->rows * (size_t)h->cols;
    *totals = malloc(((size_t)h->n_totals + 1) * sizeof **totals);
    if (!*totals) ck_fail(path, "out of memory");
    uint64_t sum = 0;
    if (fread(*totals, sizeof **totals, (size_t)h->n_totals, f) != (size_t)h->n_totals || fread(water, sizeof *water, n, f) != n ||
        fread(&sum, sizeof sum, 1, f) != 1)
        ck_fail(path, "truncated file");
    if (fgetc(f) != EOF) ck_fail(path, "longer than a checkpoint");
    fclose(f);
    if (ck_checksum(water, n, 0) != sum) ck_fail(path, "checksum mismatch (the water grid is damaged)");
}

/* What a chained run carries from one module to the next (all of it owned here). */
typedef struct {
    int active;
    char dem_path[512];
    asc_header hdr;
    double *dem;
    char out_path[512];
    double *water;        /* the previous module's output as a file would give it back: "%f"-quantised */
    solver_set prev;      /* the previous module's solver(s), grids still in HBM */
    int have_prev;
} chain_state;

static int run_module(int ntok, char tok[][512], int argc, chain_state *cs);

/* Every outlet's total over the stripes (each total lives on the stripe that owns the outlet's row and reads 0
 * elsewhere, so the element-wise sum is exact) and their sum in outlet order, the single-GPU block total. */
static double set_outlet_totals(solver_set *ss, const outlet_set *os, double *totals)
{
    double *part = ss->n > 1 ? malloc((size_t)os->n * sizeof *part) : NULL;
    if (ss->n > 1 && !part) die_solver("allocate outlet totals");
    for (int g = 0; g < ss->n; g++) {
        if (wdpm_get_outlet_drains(ss->sv[g], g == 0 ? totals : part, os->n) != WDPM_OK) die_solver("read outlet totals");
        if (g > 0)
            for (int32_t k = 0; k < os->n; k++) totals[k] += part[k];
    }
    free(part);
    double t = totals[0];
    for (int32_t k = 1; k < os->n; k++) t = t + totals[k];
    return t;
}

int main(int argc, char **argv)
{
    setbuf(stdout, NULL);
    static char tok[16][512];
    int ntok = 0;
    if (argc == 1) {
        usage_all();
        return EXIT_USAGE;
    }
    if (argc == 4 && !strcmp(argv[1], "--asc-roundtrip")) { /* test hook: read a grid, write it back */
        char *hb0 = slurp(argv[2], NULL);
        asc_header h0;
        if (!hb0 || !parse_header(hb0, &h0)) return 1;
        free(hb0);
        double *g0 = read_grid(argv[2], h0.nrows, h0.ncols, 0.0, NULL);
        return (g0 && write_grid(argv[3], &h0, g0) == 0) ? 0 : 1;
    }
    if (argc >= 3 && !strcmp(argv[1], "chain")) { /* extension: several parameter files, one process */
        static chain_state cs;
        for (const char *const *v = (const char *const[]){"WDPM_B200_CHECKPOINT", "WDPM_B200_RESUME", NULL}; *v; v++)
            if (getenv(*v) && *getenv(*v)) {
                fprintf(stderr, "%s does not apply to chain: checkpoint and resume one module at a time\n", *v);
                return 1;
            }
        cs.active = 1;
        for (int f = 2; f < argc; f++) {
            ntok = tokens_from_file(argv[f], tok, 16);
            if (ntok < 1) {
                perror("Couldn't read the parameter file");
                return 1;
            }
            const int rc = run_module(ntok, tok, 2, &cs);
            if (rc != 0) return rc;
        }
        if (cs.have_prev)
            for (int g = 0; g < cs.prev.n; g++) wdpm_destroy(cs.prev.sv[g]);
        free(cs.dem);
        free(cs.water);
        return 0;
    }
    if (argc == 2) {
        if (is_module(argv[1])) {
            usage_module(argv[1]);
            return EXIT_USAGE;
        }
        ntok = tokens_from_file(argv[1], tok, 16);
        if (ntok < 1) {
            perror("Couldn't read the parameter file");
            return 1;
        }
    } else if (argc == 12 || argc == 13) {
        for (int i = 1; i < argc; i++) snprintf(tok[ntok++], 512, "%s", argv[i]);
    } else {
        usage_module(argv[1]);
        return EXIT_USAGE;
    }
    return run_module(ntok, tok, argc, NULL);
}

/* One module, start to finish (the body of the reference's main, WDPMCL.c:308-1486). */
static int run_module(int ntok, char tok[][512], int argc, chain_state *cs)
{
    banner(tok[0]);
    run_args a;
    if (fill_args(&a, ntok, tok) != 0 || (argc > 2 && argc != (!strcmp(tok[0], "add") ? 13 : 12))) {
        usage_module(tok[0]);
        return EXIT_USAGE;
    }
    echo_args(&a);
    const int is_add = !strcmp(a.module, "add"), is_sub = !strcmp(a.module, "subtract"), is_drain = !strcmp(a.module, "drain");
    /* mm -> m (WDPMCL.c:417-420, :473-476, :528-530) */
    const double eltol = a.eltol_mm / 1000.0;
    const double depth = is_add ? a.depth_mm / 1000.0 : a.depth_mm / 1000;
    const double thres = a.thres_mm / 1000;
    /* exact checkpoints: written every ck_every blocks and at the end (ck_spec), or a run resumed from one */
    const char *ck_spec = getenv("WDPM_B200_CHECKPOINT"), *resume_path = getenv("WDPM_B200_RESUME");
    if (ck_spec && !*ck_spec) ck_spec = NULL;
    if (resume_path && !*resume_path) resume_path = NULL;
    int ck_every = 1;
    if (getenv("WDPM_B200_CHECKPOINT_EVERY") && *getenv("WDPM_B200_CHECKPOINT_EVERY")) {
        ck_every = atoi(getenv("WDPM_B200_CHECKPOINT_EVERY"));
        if (ck_every < 1) {
            fprintf(stderr, "WDPM_B200_CHECKPOINT_EVERY must be a positive number of blocks\n");
            return 1;
        }
    }

    /* DEM header and data (a chained run keeps the DEM it parsed for the module before) */
    const int same_dem = cs && cs->dem && !strcmp(cs->dem_path, a.dem);
    asc_header hdr;
    if (same_dem) {
        hdr = cs->hdr;
    } else {
        char *hb = slurp(a.dem, NULL);
        if (!hb || !parse_header(hb, &hdr)) {
            perror("Couldn't read the DEM file");
            return 1;
        }
        free(hb);
    }
    line("                  ");
    printf("%30s\n", "ArcGIS file header");
    printf("%30s %d\n", hdr.name[0], hdr.ncols);
    printf("%30s %d\n", hdr.name[1], hdr.nrows);
    for (int i = 2; i < 6; i++) printf("%30s %9.1f\n", hdr.name[i], hdr.value[i]);
    const int rows = hdr.nrows, cols = hdr.ncols;
    const size_t n = (size_t)rows * (size_t)cols;
    const double nodata = hdr.nodata, cellarea = hdr.cellsize * hdr.cellsize;
    printf("%30s\n", "Setting array sizes");
    double *dem = same_dem ? cs->dem : read_grid(a.dem, rows, cols, 0.0, NULL);
    if (!dem) {
        perror("Couldn't read the DEM file");
        return 1;
    }
    if (cs && !same_dem) { /* a new DEM: whatever the chain carried belongs to the old one */
        free(cs->dem);
        free(cs->water);
        cs->water = NULL;
        cs->out_path[0] = 0;
        if (cs->have_prev)
            for (int g = 0; g < cs->prev.n; g++) wdpm_destroy(cs->prev.sv[g]);
        cs->have_prev = 0;
        cs->dem = dem;
        cs->hdr = hdr;
        snprintf(cs->dem_path, sizeof cs->dem_path, "%s", a.dem);
    }
    line("           ");
    line("           ");

    long basincount = 0;
    for (size_t k = 0; k < n; k++) basincount += dem[k] > nodata;

    /* water: scratch file (resume) > water file > zeros; the messages follow WDPMCL.c:666-989 */
    double *water = NULL;
    int resumed = 0, chained = 0; /* chained: the water file is the output the module before has just written */
    double initial_vol = 0.0;
    if (!resume_path && !is_null_name(a.scratch)) {
        if (file_exists(a.scratch)) {
            line("           ");
            printf("%30s\n", "Scratch file found");
            water = read_grid(a.scratch, rows, cols, 0.0, NULL);
            resumed = 1;
        } else {
            line("           ");
            printf("%30s\n", "No Scratch file found");
            line("           ");
            printf("%30s\n", is_sub ? "New Scratch will be saved." : "New Scratch will be saved");
            line("           ");
            printf("%30s\n", "Now proceeding with Waterfile checking");
            line("           ");
        }
    }
    if (resume_path) {
        water = malloc(n * sizeof *water); /* filled from the checkpoint once the outlets are known */
    } else if (!water) {
        const int named = is_drain || !is_null_name(a.water);
        if (named && file_exists(a.water)) {
            printf("%30s\n", "Existing water file found");
            if (cs && cs->water && !strcmp(cs->out_path, a.water)) {
                water = cs->water; /* what reading that file back would give */
                cs->water = NULL;
                chained = 1;
            } else {
                water = read_grid(a.water, rows, cols, 0.0, NULL);
            }
            if (!is_drain && !is_null_name(a.scratch)) { /* only this path recomputes the initial volume (:690-699, :846-855) */
                for (size_t k = 0; k < n; k++)
                    if (is_add ? dem[k] > nodata : dem[k] > 0) initial_vol += water[k];
                initial_vol *= cellarea;
            }
        } else if (is_drain) {
            printf("%30s\n", "Error water file missing");
            return EXIT_USAGE;
        } else {
            printf("%30s\n", named ? "Water file missing, will be created" : "Water file will be created");
            water = calloc(n, sizeof *water);
        }
    }
    if (!water) {
        perror("Couldn't read the water file");
        return 1;
    }
    if (is_drain && !resume_path) {
        initial_vol = 0.0;
        for (size_t k = 0; k < n; k++)
            if (dem[k] > nodata) initial_vol += water[k];
        initial_vol *= cellarea;
    }

    /* an outlet set replaces the reference's single outlet (Drain only); checked before any solver exists */
    outlet_set os = {0, NULL, NULL};
    const char *outlet_spec = getenv("WDPM_B200_OUTLETS");
    if (is_drain && outlet_spec && *outlet_spec) {
        load_outlets(outlet_spec, dem, rows, cols, nodata, &os);
        if (a.backend == 0 && os.n > 1) outlets_fail(outlet_spec, "cpu=0 (the serial branch) drains through one outlet");
    }
    double *outlet_totals = os.n > 0 ? malloc((size_t)os.n * sizeof *outlet_totals) : NULL;
    if (os.n > 0 && !outlet_totals) outlets_fail(outlet_spec, "out of memory");

    const int module = is_add ? WDPM_ADD : is_sub ? WDPM_SUBTRACT : WDPM_DRAIN;
    const int schedule = a.backend == 0 ? WDPM_SCHEDULE_SERIAL : WDPM_SCHEDULE_OPENCL;
    ck_header ident, ck_in;
    double *ck_totals = NULL;
    if (ck_spec || resume_path) ck_identity(&ident, &hdr, dem, module, schedule, is_drain ? 0.0 : depth, is_add ? a.runoff_frac : 0.0, thres, &os);
    if (resume_path) { /* checked in full before any solver exists */
        ck_read(resume_path, &ident, &ck_in, &ck_totals, water);
        initial_vol = ck_in.initial_vol;
        line("           ");
        printf("%30s\n", "Checkpoint found");
        printf("%30s %lld\n", "Resuming at iteration:", (long long)ck_in.iterations);
        line("           ");
    }

    /* solver */
    wdpm_config cfg;
    memset(&cfg, 0, sizeof cfg);
    cfg.struct_size = sizeof cfg;
    cfg.rows = rows;
    cfg.cols = cols;
    cfg.nodata = nodata;
    cfg.dtype = WDPM_F64;
    cfg.module = module;
    cfg.zero_threshold = thres;
    cfg.schedule = schedule;
    cfg.device = getenv("WDPM_B200_DEVICE") ? atoi(getenv("WDPM_B200_DEVICE")) : 0;
    cfg.kernel = getenv("WDPM_B200_KERNEL") ? atoi(getenv("WDPM_B200_KERNEL")) : WDPM_KERNEL_AUTO;
    solver_set ss;
    set_create(&ss, cfg, getenv("WDPM_B200_GPUS") ? atoi(getenv("WDPM_B200_GPUS")) : 1);
    if (cs && cs->have_prev && same_dem && ss.n == 1 && cs->prev.n == 1) {
        /* same DEM, one GPU: the grids never leave HBM */
        if (wdpm_copy_state(ss.sv[0], cs->prev.sv[0], WDPM_COPY_DEM | (chained ? WDPM_COPY_WATER : 0)) != WDPM_OK) die_solver("hand the grids on");
        if (chained) {
            if (wdpm_quantize_water(ss.sv[0]) != WDPM_OK) die_solver("quantise the water grid");
        } else if (wdpm_upload_water(ss.sv[0], water) != WDPM_OK) {
            die_solver("upload the water grid");
        }
    } else {
        set_upload(&ss, dem, water, cols);
    }
    if (cs && cs->have_prev) {
        for (int g = 0; g < cs->prev.n; g++) wdpm_destroy(cs->prev.sv[g]);
        cs->have_prev = 0;
    }
    if (!resumed && !resume_path) {
        for (int g = 0; g < ss.n; g++) {
            if (is_add && wdpm_apply_add(ss.sv[g], depth, a.runoff_frac) != WDPM_OK) die_solver("add water");
            if (is_sub && wdpm_apply_subtract(ss.sv[g], depth) != WDPM_OK) die_solver("subtract water");
        }
    }

    double total_drain = 0.0;
    if (is_drain && os.n > 0) {
        double minel = 0.0;
        for (int32_t k = 0; k < os.n; k++) {
            const double e = dem[(size_t)(os.row[k] - 1) * cols + (os.col[k] - 1)];
            if (k == 0 || e < minel) minel = e;
        }
        for (int g = 0; g < ss.n; g++) {
            if (wdpm_set_outlets(ss.sv[g], os.n, os.row, os.col) != WDPM_OK) die_solver("set the drain outlets");
            if (resume_path ? wdpm_set_outlet_drains(ss.sv[g], ck_totals, os.n) != WDPM_OK : wdpm_seed_outlet_drains(ss.sv[g]) != WDPM_OK)
                die_solver("seed the outlet totals");
        }
        total_drain = resume_path ? ck_in.total_drain : set_outlet_totals(&ss, &os, outlet_totals);
        line("               ");
        printf("%30s\n", "Basin summary");
        printf("%20s %10.4f %s\n", "Basin area:", (double)basincount * cellarea, "m2");
        printf("%20s %10.4f %s\n", "Initial volume:", initial_vol, "m3");
        printf("%20s %d\n", "Drain outlets:", os.n);
        printf("%20s %10.4f %s\n", "Min DEM elevation:", minel, "m");
    } else if (is_drain) {
        int32_t drow = 0, dcol = 0;
        double minel = 0.0, w_out = 0.0;
        int owner = -1;
        for (int g = 0; g < ss.n; g++) { /* every stripe's lowest cell; the lowest, first in row-major order, wins */
            int32_t r, c;
            double e;
            if (wdpm_find_outlet(ss.sv[g], &r, &c, &e) != WDPM_OK) continue; /* no cell above 0 in this stripe */
            if (owner < 0 || e < minel) { owner = g; drow = r; dcol = c; minel = e; }
        }
        if (owner < 0) die_solver("locate the drain");
        for (int g = 0; g < ss.n; g++)
            if (wdpm_set_outlet(ss.sv[g], drow, dcol) != WDPM_OK) die_solver("set the drain");
        if (resume_path) {
            total_drain = ck_in.total_drain;
            for (int g = 0; g < ss.n; g++)
                if (wdpm_set_outlet_drains(ss.sv[g], ck_totals, 1) != WDPM_OK) die_solver("set totaldrain");
        } else {
            if (wdpm_get_cell_water(ss.sv[owner], drow, dcol, &w_out) != WDPM_OK) die_solver("read the drain cell");
            total_drain = w_out > 0 ? w_out : 0; /* WDPMCL.c:1029 */
            for (int g = 0; g < ss.n; g++)
                if (wdpm_set_total_drain(ss.sv[g], g == owner ? total_drain : 0.0) != WDPM_OK) die_solver("set totaldrain");
        }
        line("               ");
        printf("%30s\n", "Basin summary");
        printf("%20s %10.4f %s\n", "Basin area:", (double)basincount * cellarea, "m2");
        printf("%20s %10.4f %s\n", "Initial volume:", initial_vol, "m3");
        printf("%20s %d\n", "Drain column:", dcol);
        printf("%20s %d\n", "Drain row:", drow);
        printf("%20s %10.4f %s\n", "Min DEM elevation:", minel, "m");
    }
    line("               ");
    printf("%30s\n", "Doing calculations");
    if (is_drain) {
        printf("%15s %15s %15s %15s %15s\n", "iterations", "max diff", "vol change", "water left", "run time");
        printf("%13s %14s %15s %16s %17s\n", " ", "(m)", "(m3)", "(m3)", "(s)");
    } else {
        printf("%15s %15s %15s\n", "iterations", "max diff", "run time");
        printf("%13s %14s %15s\n", " ", "(m)", "(s)");
    }

    /* blocks of 1000 iterations until a stop test fires (WDPMCL.c:1054-1377) */
    struct timeval t0;
    gettimeofday(&t0, NULL);
    int k = resume_path ? (int)ck_in.iterations : 0, done = 0, armed = 0;
    scratch_writer scratch;
    memset(&scratch, 0, sizeof scratch);
    static ck_writer ckw; /* large (per-GPU arrays); one module at a time */
    memset(&ckw, 0, sizeof ckw);
    if (ck_spec) {
        ckw.totals = malloc(((size_t)ident.n_totals + 1) * sizeof *ckw.totals);
        if (!ckw.totals) die_solver("allocate the checkpoint totals");
    }
    while (!done) {
        const double old_drain = total_drain;
        wdpm_block_result r;
        set_run_block(&ss, BLOCK_ITERATIONS, &r, armed ? &ckw : NULL);
        armed = 0;
        k += BLOCK_ITERATIONS;
        total_drain = (os.n > 0 && ss.n > 1) ? set_outlet_totals(&ss, &os, outlet_totals) : r.total_drain;
        double diffdrain = 0.0;
        if (is_drain) {
            diffdrain = fabs(total_drain - old_drain) * cellarea;
            printf("%7s %d %7s %8.3f %5s %10.1f %5s %12.1f %5s %8.2f\n", "", k, "", r.max_diff, "", diffdrain, "",
                   r.masked_sum * cellarea, "", seconds_since(&t0));
        } else {
            printf("%7s %d %7s %8.3f %5s %8.2f\n", "", k, "", r.max_diff, "", seconds_since(&t0));
        }
        done = r.max_diff <= eltol || (is_drain && diffdrain < a.drain_tol) || (a.iter_limit > 0 && k >= a.iter_limit);
        if (!done && !is_null_name(a.scratch)) {
            set_download(&ss, water, cols);
            if (is_add) mark_nodata(water, dem, n, nodata);
            scratch_start(&scratch, a.scratch, &hdr, water, n);
        }
        if (!done && ck_spec && (k / BLOCK_ITERATIONS) % ck_every == 0) { /* the next block captures the state at k */
            ck_join(&ckw); /* its staging is about to be reused */
            for (int g = 0; g < ss.n; g++)
                if (wdpm_checkpoint_arm(ss.sv[g]) != WDPM_OK) die_solver("arm the checkpoint capture");
            ckw.h = ident;
            ckw.h.iterations = k;
            ckw.h.initial_vol = initial_vol;
            ckw.h.total_drain = total_drain;
            ck_path(ckw.path, sizeof ckw.path, ck_spec, k);
            armed = 1;
        }
    }

    scratch_join(&scratch);

    /* final grid and statistics (WDPMCL.c:1379-1467) */
    set_download(&ss, water, cols);
    if (ck_spec) { /* the end of the run, from the grid downloaded for the output anyway */
        ck_join(&ckw);
        ckw.h = ident;
        ckw.h.iterations = k;
        ckw.h.initial_vol = initial_vol;
        ckw.h.total_drain = total_drain;
        if (os.n > 0) set_outlet_totals(&ss, &os, ckw.totals);
        else if (is_drain) ckw.totals[0] = total_drain;
        ckw.n_pieces = 1;
        ckw.piece[0] = water;
        ckw.row0[0] = 0;
        ckw.nrows[0] = rows;
        ck_path(ckw.path, sizeof ckw.path, ck_spec, k);
        ck_main(&ckw);
        ck_join(&ckw);
        free(ckw.totals);
    }
    mark_nodata(water, dem, n, nodata);
    /* The order-free statistics come from the device (wdpm_final_statistics: counts add and maxima combine over the
     * stripes); the volume is the reference's own sequential sum over the grid the output file needs anyway, so that
     * the printed digits are the reference's (WDPMCL.c:1394-1459). */
    long watercount = 0;
    double watertotal = 0.0, dev_maxdepth = 0.0;
    int64_t dev_valid = 0, dev_wet = 0;
    int have_dev_stats = 1;
    for (int g = 0; g < ss.n; g++) {
        int64_t nv = 0, nw = 0;
        double md = 0.0;
        if (wdpm_final_statistics(ss.sv[g], &nv, &nw, &md) != WDPM_OK) { have_dev_stats = 0; break; }
        if (nv > 0 && (dev_valid == 0 || md > dev_maxdepth)) dev_maxdepth = md;
        dev_valid += nv;
        dev_wet += nw;
    }
    for (size_t i = 0; i < n; i++)
        if (dem[i] > nodata) watertotal += water[i];
    if (have_dev_stats && dev_valid == basincount && basincount > 0) {
        watercount = (long)dev_wet;
    } else { /* no valid cell, or a DEM the device masks differently (NaN / infinite elevations): count here */
        have_dev_stats = 0;
        for (size_t i = 0; i < n; i++)
            if (dem[i] > nodata && water[i] > 0.001) watercount++;
    }
    const double final_vol = watertotal * cellarea;
    const double meanwater = watertotal / ((float)watercount);
    const double waterfrac = (float)watercount / (float)basincount;
    const double drainvol = total_drain * cellarea;
    const double draindepth = (drainvol / ((float)basincount * cellarea)) * 1000;
    double maxdepth = water[0]; /* the reference scans every cell, NODATA-valued ones included (:1451-1459) */
    if (have_dev_stats && nodata < 0 && dev_maxdepth >= maxdepth) {
        maxdepth = dev_maxdepth; /* valid cells hold >= 0, NODATA cells the (negative) NODATA value: the maximum is a valid cell's */
    } else {
        for (size_t i = 0; i < n; i++)
            if (water[i] > maxdepth) maxdepth = water[i];
    }
    maxdepth *= 1000;

    line("                     ");
    printf("%30s\n", "WDPM run summary");
    printf("%20s %10.2f %s\n", "Initial volume", initial_vol, "m3");
    printf("%20s %10.2f %s\n", "Final volume", final_vol, "m3");
    printf("%20s %10.2f %s\n", "Volume change", is_drain ? initial_vol - final_vol : final_vol - initial_vol, "m3");
    if (is_drain) printf("%20s %10.2f %s\n", "Volume drained", drainvol, "m3");
    printf("%20s %10.4f %s\n", "Final water coverage", waterfrac, "");
    printf("%20s %10.2f %s\n", "Mean water depth", meanwater * 1000., "mm");
    if (is_drain) printf("%20s %10.2f %s\n", "Depth drained", draindepth, "mm ");
    printf("%20s %10.2f %s\n", "Max water depth", maxdepth, "mm ");

    if (write_grid(a.output, &hdr, water) != 0) {
        perror("Couldn't write the output file");
        return 1;
    }
    printf("%20s %10.2f %s\n", "Run Time", seconds_since(&t0), "s");
    const char *totals_path = getenv("WDPM_B200_OUTLET_TOTALS");
    if (os.n > 0 && totals_path && *totals_path) {
        set_outlet_totals(&ss, &os, outlet_totals);
        FILE *f = fopen(totals_path, "w");
        if (!f) {
            perror("Couldn't write the outlet totals");
            return 1;
        }
        for (int32_t q = 0; q < os.n; q++)
            fprintf(f, "%d,%d,%.17g,%.17g\n", os.row[q], os.col[q], dem[(size_t)(os.row[q] - 1) * cols + (os.col[q] - 1)], outlet_totals[q] * cellarea);
        if (fclose(f) != 0) {
            perror("Couldn't write the outlet totals");
            return 1;
        }
    }
    free(outlet_totals);
    free(ck_totals);
    free(os.row);
    free(os.col);
    free(scratch.grid);
    if (cs) { /* keep what the next module may want: the solver (grids in HBM) and the output as its file reads back */
        cs->prev = ss;
        cs->have_prev = 1;
#pragma omp parallel for schedule(static)
        for (long long i = 0; i < (long long)n; i++) water[i] = wdpm_quantize6(water[i]);
        free(cs->water);
        cs->water = water;
        snprintf(cs->out_path, sizeof cs->out_path, "%s", a.output);
        return 0;
    }
    for (int g = 0; g < ss.n; g++) wdpm_destroy(ss.sv[g]);
    free(dem);
    free(water);
    return 0;
}
