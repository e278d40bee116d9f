/*
 * wdpm_b200 - C ABI of the B200-native WDPM water-redistribution solver.
 *
 * This is the drop-in boundary for ONE path of CentreForHydrology/WDPM: the
 * iterative 8-neighbour, 9-colour ponding stencil behind the Add, Subtract and
 * Drain modules. In the reference that path is the OpenCL branch of the solver
 * loop (src/WDPMCL.c:1126-1236) plus its kernels (src/runoff.cl:137-183), the
 * per-block prologue (src/WDPMCL.c:1055-1073) and the convergence / water-balance
 * reductions (src/WDPMCL.c:1239-1268). A host keeps WDPMCL's command line, .asc
 * I/O, printed report and stop logic (src/WDPMCL.c:1283-1376) and calls these
 * entry points instead of the cl* calls; INTEGRATION.md shows the patch.
 *
 * Conventions
 *  - plain C, no CUDA or torch types; every call returns 0 on success or a
 *    negative WDPM_E_* code and never exits the process; wdpm_last_error()
 *    returns a message for the calling thread's last failure.
 *  - grids cross the boundary as UNPADDED row-major host arrays of rows*cols
 *    elements in the solver's precision (float for WDPM_F32, double for WDPM_F64),
 *    i.e. the reference's dem[][] / water[][] (src/WDPMCL.c:560-570). Padding to
 *    bigdem / bigwater (src/WDPMCL.c:795-807) and the device layout are internal.
 *  - cell coordinates are the reference's 1-based padded ones: row 1..rows,
 *    col 1..cols (drainrow/draincol of src/WDPMCL.c:1005-1017).
 *  - one solver = one GPU (or one row stripe of a DEM on one GPU); calls on one
 *    solver must come from one host thread at a time.
 *  - there is no CPU fallback: without a CUDA device wdpm_create fails with
 *    WDPM_E_CUDA.
 */
#ifndef WDPM_B200_H
#define WDPM_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define WDPM_ABI_VERSION 1

/* modules: which relax function runs (src/runoff.cl:24-55, :57-88, :90-134) */
#define WDPM_ADD 0
#define WDPM_SUBTRACT 1
#define WDPM_DRAIN 2

/* Update schedule: which of the reference's two backends (its "cpu" flag) the arithmetic follows.
 * OPENCL (0, the default of a zeroed config): the kernels of src/runoff.cl.
 * SERIAL (1): the serial branch of src/WDPMCL.c. Add is the same as OPENCL. Subtract relaxes with
 *   runoffs, the Add step (:1934-1964), instead of runoffsubtract. Drain relaxes as runoffdrain does and
 *   then, after every whole iteration, empties the outlet's 3x3 neighbourhood (drain(), :1859-1897):
 *   the water of its cells with dem > nodata and w > 0 is summed in row-major order and added to
 *   totaldrain, and all nine cells are set to 0. wdpm_subpass stays a bare sub-pass; every other call
 *   that iterates includes the emptying. One outlet only (wdpm_set_outlets refuses a set), and a fused
 *   variant with more than one iteration per launch refuses Drain. */
#define WDPM_SCHEDULE_OPENCL 0
#define WDPM_SCHEDULE_SERIAL 1

/* precision of the device arithmetic and of the host arrays */
#define WDPM_F32 0
#define WDPM_F64 1 /* the reference's precision (src/runoff.cl:1) */

/* kernel selection */
#define WDPM_KERNEL_AUTO 0
#define WDPM_KERNEL_COLOUR 1 /* one launch per colour sub-pass, global memory (the reference's schedule) */
#define WDPM_KERNEL_FUSED 2  /* one launch per iteration: 9 sub-passes over a TMA-fed shared-memory row window */
#define WDPM_KERNEL_RESIDENT 3 /* small grids: one cooperative launch per block, tiles resident in shared memory */

/* error codes */
#define WDPM_OK 0
#define WDPM_E_ARG -1    /* bad argument */
#define WDPM_E_CUDA -2   /* CUDA runtime / driver failure, or no device */
#define WDPM_E_NOMEM -3  /* host or device allocation failed */
#define WDPM_E_STATE -4  /* call out of order (e.g. run before upload) */
#define WDPM_E_UNSUPPORTED -5
#define WDPM_E_HALO -6   /* stripes: a neighbour's halo did not arrive (WDPM_B200_HALO_TIMEOUT_MS, default 120 s); upload again */

typedef struct wdpm_solver wdpm_solver; /* opaque; owns all device memory */

typedef struct wdpm_config {
    uint32_t struct_size; /* sizeof(wdpm_config), for ABI evolution */
    int32_t rows;         /* numrows of the DEM (src/WDPMCL.c:553) */
    int32_t cols;         /* numcols (src/WDPMCL.c:552) */
    double nodata;        /* missingvalue, header line 6 (src/WDPMCL.c:554) */
    int32_t dtype;        /* WDPM_F32 | WDPM_F64 */
    int32_t module;       /* WDPM_ADD | WDPM_SUBTRACT | WDPM_DRAIN */
    double zero_threshold; /* metres; "thres" of src/WDPMCL.c:420, applied at :1055-1065 */
    int32_t device;       /* CUDA device ordinal */
    int32_t kernel;       /* WDPM_KERNEL_* */
    /* Row-stripe partition (multi-GPU). A single-GPU solver sets both to 0. Otherwise
     * this solver owns PADDED rows [stripe_row0, stripe_row0 + stripe_rows) of a DEM
     * whose padded rows are 0..rows+1; stripe_row0 must be a multiple of 3. See
     * wdpm_stripe_* below. */
    int32_t stripe_row0;
    int32_t stripe_rows;
    int32_t iters_per_launch; /* fused kernel: iterations carried per HBM round trip (0 = default) */
    int32_t fused_variant;    /* fused kernel tiling variant (0 = auto; see wdpm_fused_variant_info) */
    int32_t fused_chunk_rows; /* owned rows per CTA, rounded up to a multiple of 3 (0 = auto) */
    int32_t schedule;         /* WDPM_SCHEDULE_* */
    int32_t reserved[4];
} wdpm_config;

/* What one convergence block reports (src/WDPMCL.c:1239-1268). */
typedef struct wdpm_block_result {
    double max_diff;     /* max |w - w_at_block_start| over cells with dem > nodata (:1239-1254) */
    double masked_sum;   /* sum of w over cells with dem > nodata, in metres (x cellarea = final_vol, :1259-1267) */
    double total_drain;  /* running totaldrain after the block (Drain only; :1213) */
    int64_t wet_cells;   /* cells with w > 0 and dem > nodata after the block (diagnostic) */
    int32_t iterations;  /* iterations executed by this call */
    int32_t launches;    /* kernel launches issued by this call */
    float block_ms;      /* device time of the whole block, CUDA events on the solver's stream */
    float iterate_ms;    /* device time of the iteration kernels only */
} wdpm_block_result;

const char *wdpm_last_error(void);
int wdpm_abi_version(void);
int wdpm_device_count(void);

/* replaces create_device / clCreateContext / build_program / clCreateKernel /
 * buffer allocation (src/WDPMCL.c:598-638) */
int wdpm_create(const wdpm_config *cfg, wdpm_solver **out);
/* replaces the clRelease* calls (src/WDPMCL.c:1475-1483) */
int wdpm_destroy(wdpm_solver *s);

/* replaces flatten + clCreateBuffer + clEnqueueWriteBuffer (src/WDPMCL.c:1129-1153),
 * done once instead of once per block. `water` may be NULL (all zero). Stripe
 * solvers use wdpm_stripe_upload instead; their download returns the owned interior
 * rows only (see wdpm_stripe_band). */
int wdpm_upload(wdpm_solver *s, const void *dem, const void *water);
/* replaces only the water upload (resume from a scratch file, src/WDPMCL.c:668-673) */
int wdpm_upload_water(wdpm_solver *s, const void *water);
/* replaces clEnqueueReadBuffer of bigwater + un-flatten (src/WDPMCL.c:1217-1233) */
int wdpm_download_water(wdpm_solver *s, void *water);

/* Module initial conditions on the device, valid cells only:
 * Add (src/WDPMCL.c:778-792): w > 0 -> w += depth; then w <= 0 -> w = depth*rof.
 * Subtract (src/WDPMCL.c:919-926): w = max(w - depth, 0). Depths in metres. */
int wdpm_apply_add(wdpm_solver *s, double depth, double runoff_fraction);
int wdpm_apply_subtract(wdpm_solver *s, double depth);

/* Drain outlet (src/WDPMCL.c:1005-1017): lowest cell with dem > 0, first in
 * row-major order; 1-based padded coordinates. wdpm_find_outlet also installs it.
 * Returns WDPM_E_STATE if no cell has dem > 0. */
int wdpm_find_outlet(wdpm_solver *s, int32_t *drainrow, int32_t *draincol, double *min_elevation);
int wdpm_set_outlet(wdpm_solver *s, int32_t drainrow, int32_t draincol);
/* Extension (BASELINE configs[4], "many drain outlets"): a SET of outlet cells, in padded
 * coordinates of the whole DEM. Each outlet follows src/runoff.cl:104-111 - never a centre; a
 * neighbouring centre empties itself and the outlet into that outlet's total. One outlet is the
 * reference. Every outlet has its own accumulator; the reported total is their sum in outlet order
 * (solver precision). Replaces any earlier set. Drain solvers only. Row stripes: every stripe is given the whole
 * set; an outlet's total is kept by the stripe that owns its row - contacts from centres of a neighbouring stripe
 * are recorded there too, in sub-pass order, so each total is bit-identical to the single-GPU one - and reads as 0 on
 * the other stripes: a host adds the stripes' wdpm_get_outlet_drains element by element.
 * Up to WDPM_MAX_OUTLETS cells, each inside the DEM (row 1..rows, col 1..cols) and on a cell with dem > nodata;
 * otherwise, and for a duplicate, WDPM_E_ARG. The dem test runs once the set and an uploaded DEM meet (here, or
 * in a later upload, which then fails and leaves no set installed). The serial schedule refuses a set of more than one
 * outlet (WDPM_E_UNSUPPORTED). The solver sorts the set; the time a kernel spends on an outlet contact grows as
 * log2(n), and the device memory the set takes grows linearly in n (DESIGN.md section 3.3 gives the bound).
 * wdpm_get_outlet_drains returns the first n totals in the caller's order (n at most the set's size). */
#define WDPM_MAX_OUTLETS 1048576
int wdpm_set_outlets(wdpm_solver *s, int32_t n, const int32_t *rows, const int32_t *cols);
int wdpm_get_outlet_drains(wdpm_solver *s, double *values, int32_t n);
/* totaldrain accumulator (src/WDPMCL.c:1029, :1136); with an outlet set, set writes the first
 * outlet's total and zeroes the others, get returns the sum (computed on the device) */
int wdpm_set_total_drain(wdpm_solver *s, double value);
int wdpm_get_total_drain(wdpm_solver *s, double *value);
/* Seed every outlet's total with max(water at the outlet, 0): src/WDPMCL.c:1029 applied to each outlet. On row
 * stripes the stripe that owns the outlet's row does it and the others set 0. For one outlet it equals
 * wdpm_get_cell_water followed by wdpm_set_total_drain(max(w, 0)). */
int wdpm_seed_outlet_drains(wdpm_solver *s);
/* Restore every outlet's total, values[k] for the caller's outlet k (n = the installed set's size; 1 for the
 * reference's outlet or before any set). On row stripes it follows wdpm_seed_outlet_drains: the stripe that owns the
 * outlet's row keeps the value and the others set 0, so every stripe may be given the whole array. Converted to the
 * solver's precision. WDPM_E_STATE outside Drain, WDPM_E_ARG for another n. Resumes a Drain run with its totals
 * (wdpm_set_total_drain keeps only the first outlet's). */
int wdpm_set_outlet_drains(wdpm_solver *s, const double *values, int32_t n);
/* Exact checkpoints. wdpm_checkpoint_arm makes the next wdpm_block_begin (or wdpm_run_block) capture the state the
 * block starts from: the water after its zero-threshold pass (the snapshot of src/WDPMCL.c:1055-1073; the pass is
 * idempotent, so this water starts a block exactly as the unthresholded water before it does) and every outlet's
 * total. The block runs on while a side stream copies both into pinned host memory the solver owns (allocated by
 * the first arm, one owned grid, freed by wdpm_destroy); nothing waits for the copy on the host, and the next
 * prologue waits for it on the device. wdpm_checkpoint_wait blocks until the capture has landed and returns
 * pointers into that memory, valid until the next arm: the water as the owned interior rows (unpadded row-major, the
 * solver's precision, raw bits; a stripe's rows as wdpm_download_water returns them) and the totals as doubles in
 * the caller's outlet order (n = the set's size, 1 without a set; per stripe as wdpm_get_outlet_drains). Uploading
 * that water into a fresh solver for the same DEM and module (any kernel, any partition) and restoring the totals
 * with wdpm_set_outlet_drains continues the run bit for bit. arm: WDPM_E_STATE inside a block or before an
 * upload; wait: WDPM_E_STATE when no capture has been taken since the last arm. */
int wdpm_checkpoint_arm(wdpm_solver *s);
int wdpm_checkpoint_wait(wdpm_solver *s, const void **water, const double **totals, int32_t *n);
/* Module chaining. The reference runs Add -> Drain -> Subtract as three processes that hand the
 * water grid on through "%f" text files (validation/validate_WDPM.sh:77-99). A host that runs the
 * modules in one process can keep the grids in HBM instead:
 *   wdpm_copy_state   copies the elevations and/or the current water grid of `src` into `dst` (another
 *                     solver for the same DEM on the same device, e.g. created for the next module),
 *                     device to device;
 *   wdpm_quantize_water applies to every valid cell what the file hand-over does to it - round to 6
 *                     decimals exactly as fprintf("%f") + fscanf("%lf") do (include/wdpm_quantize.h) -
 *                     so the next module starts from bit-identical values. */
#define WDPM_COPY_DEM 1
#define WDPM_COPY_WATER 2
int wdpm_copy_state(wdpm_solver *dst, wdpm_solver *src, int32_t what);
int wdpm_quantize_water(wdpm_solver *s);
/* water depth at one cell (for totaldrain = max(bigwater[outlet],0), src/WDPMCL.c:1029) */
int wdpm_get_cell_water(wdpm_solver *s, int32_t row, int32_t col, double *value);

/* The order-free part of the final report (src/WDPMCL.c:1394-1459) computed on the device over the interior cells
 * this solver owns: cells with dem > nodata (basincount), those of them with water > 0.001 m (watercount, from
 * which "Final water coverage" and the divisor of "Mean water depth" follow) and the deepest water on a valid cell
 * ("Max water depth"). Counts add and maxima combine over stripes. The volume sums of the report are NOT here: the
 * reference accumulates them cell by cell in double and prints them with fixed decimals, which only a sequential
 * pass over the downloaded grid reproduces digit for digit. Any pointer may be NULL. */
int wdpm_final_statistics(wdpm_solver *s, int64_t *valid_cells, int64_t *wet_above_1mm, double *max_depth);

/* Order-free 64-bit checksum of the water grid this solver owns (interior cells): sum of
 * bits(w) * (2*index + 1) mod 2^64, index = row-major position in the WHOLE DEM. The sum of the stripes' checksums
 * (mod 2^64) equals the single-solver checksum iff the grids are equal bit for bit, whatever the partition.
 * New work (benchmark / consistency evidence); the reference has no counterpart. */
int wdpm_water_checksum(wdpm_solver *s, uint64_t *checksum);

/* One convergence block, all on the device, no host round trip inside:
 * zero-threshold + snapshot (src/WDPMCL.c:1055-1073), n_iters iterations of the
 * nine colour sub-passes (:1184-1206 with src/runoff.cl), then the masked
 * max-difference and sum (:1239-1268). The reference always passes 1000. */
int wdpm_run_block(wdpm_solver *s, int32_t n_iters, wdpm_block_result *out);

/* The same block in pieces, for a host thread that drives several stripe solvers (one per GPU):
 * begin = threshold + snapshot, enqueue = n more iterations, end = reductions + the only host wait.
 * begin and enqueue never block, so the host can feed all stripes round-robin; their kernels find
 * each other through the device-side halo flags. wdpm_run_block = begin + enqueue(n) + end. */
int wdpm_block_begin(wdpm_solver *s);
int wdpm_block_enqueue(wdpm_solver *s, int32_t n_iters);
int wdpm_block_end(wdpm_solver *s, wdpm_block_result *out);

/* n_iters iterations only - no threshold, snapshot or reductions (benchmarks, tests). */
int wdpm_iterate(wdpm_solver *s, int32_t n_iters);
/* a single colour sub-pass (oi, oj in 1..3), colour kernel only (tests). */
int wdpm_subpass(wdpm_solver *s, int32_t oi, int32_t oj);

/* Run on a caller-owned CUDA stream (a cudaStream_t passed as void*; NULL = the
 * solver's own stream). Lets a host time the solver with its own events. */
int wdpm_set_stream(wdpm_solver *s, void *cuda_stream);
int wdpm_synchronize(wdpm_solver *s);

/* Introspection for benchmarks: bytes of HBM the solver holds, the fused
 * kernel's tiling, and how many of this library's kernels it has launched. */
typedef struct wdpm_info {
    int64_t device_bytes;
    int64_t kernel_launches;
    int32_t kernel;          /* WDPM_KERNEL_* actually in use */
    int32_t strip_cols;      /* fused: owned columns per strip */
    int32_t window_cols;     /* fused: columns staged in shared memory per strip */
    int32_t chunk_rows;      /* fused: owned rows per CTA */
    int32_t grid_ctas;
    int32_t cta_threads;
    int32_t smem_bytes;
    int32_t iters_per_launch;
    int32_t sm_count;
    int32_t warp_autonomous; /* fused: 1 = the warp-autonomous kernel (two tiles per lane, warp shuffles), 0 = k_fused */
    int32_t reserved[6];
} wdpm_info;
int wdpm_get_info(wdpm_solver *s, wdpm_info *info);
/* Tiling of fused variant `variant` (1-based) for `dtype`; returns WDPM_E_ARG past the last one. */
int wdpm_fused_variant_info(int32_t variant, int32_t dtype, int32_t *window_cols, int32_t *strip_cols,
                            int32_t *iters_per_launch, int32_t *cta_threads, int32_t *smem_bytes);

/* ---- row-stripe partition across GPUs (one solver per GPU) -----------------
 * New work: the reference is single-device (src/WDPMCL.c:98-118). The padded DEM
 * (rows 0..rows+1, src/WDPMCL.c:795-807) is cut into contiguous bands of padded
 * rows, band starts being multiples of 3 so every cell keeps its colour. A stripe
 * solver is created with cfg.rows/cols = the WHOLE DEM's size, cfg.stripe_row0 =
 * first padded row it owns and cfg.stripe_rows = number of padded rows it owns
 * (0 = not a stripe). It also keeps WDPM_STRIPE_HALO_ABOVE rows of the band above
 * and WDPM_STRIPE_HALO_BELOW rows of the band below: what one fused iteration
 * needs to produce its owned rows exactly. After every iteration each stripe
 * writes the rows its neighbours need straight into their memory over NVLink
 * (peer stores) and raises an arrival flag there; a neighbour's next iteration
 * waits on that flag on the device. Per-block reductions stay per stripe; the
 * host combines them (max / sum in stripe order).
 * Only the fused kernel with one iteration per launch supports stripes. */
#define WDPM_STRIPE_HALO_ABOVE 3
#define WDPM_STRIPE_HALO_BELOW 6
#define WDPM_IPC_HANDLE_BYTES 64
typedef struct wdpm_stripe_endpoint {
    uint8_t water_a[WDPM_IPC_HANDLE_BYTES]; /* cudaIpcMemHandle_t of the ping water buffer */
    uint8_t water_b[WDPM_IPC_HANDLE_BYTES]; /* cudaIpcMemHandle_t of the pong water buffer */
    uint8_t flags[WDPM_IPC_HANDLE_BYTES];   /* cudaIpcMemHandle_t of the arrival flags */
    int32_t device;
    int32_t stripe_row0;
    int32_t stripe_rows;
    int32_t pitch;      /* elements per device row: must match between neighbours */
    int64_t pid;        /* exporting process, to tell in-process neighbours apart */
    uint64_t local_ptr; /* the exporting solver's address (valid only inside process `pid`) */
} wdpm_stripe_endpoint;
int wdpm_stripe_export(wdpm_solver *s, wdpm_stripe_endpoint *self);
/* `above` = the stripe holding smaller row numbers, `below` = larger; NULL at the DEM edge.
 * Endpoints from this process are wired by pointer, others through CUDA IPC. */
int wdpm_stripe_connect(wdpm_solver *s, const wdpm_stripe_endpoint *above,
                        const wdpm_stripe_endpoint *below);
/* Upload `band_rows` whole rows of the UNPADDED dem / water arrays starting at interior row
 * `band_row0` (0-based) - the band must cover the stripe's owned rows plus its halos, clipped to
 * the DEM (wdpm_stripe_band tells which rows those are). water may be NULL. */
int wdpm_stripe_band(wdpm_solver *s, int32_t *band_row0, int32_t *band_rows, int32_t *owned_row0,
                     int32_t *owned_rows);
int wdpm_stripe_upload(wdpm_solver *s, const void *dem_band, const void *water_band,
                       int32_t band_row0, int32_t band_rows);
/* One iteration without the wait for the neighbours' halos, for hosts that drive several in-process stripes in
 * lockstep (tests): phase 0 = launch the iteration kernel, which also writes this stripe's halo rows into the
 * neighbours' buffers and raises their flags; phase 1, to be called once EVERY stripe has completed phase 0, folds
 * the Drain contacts of that iteration into the outlets' totals (a neighbour records the contacts of its centres
 * with this stripe's outlets in this stripe's buffers; a no-op for Add / Subtract).
 * wdpm_iterate / wdpm_run_block do all of it per iteration on their own. */
int wdpm_stripe_phase(wdpm_solver *s, int32_t phase);

#ifdef __cplusplus
}
#endif
#endif /* WDPM_B200_H */
