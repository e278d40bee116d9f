// CUDA kernels of the WDPM redistribution solver (sm_100a).
//
// Device layout: every grid (dem, water ping, water pong, block-start snapshot)
// is a row-major array of `nrows_dev` x `pitch` elements. Padded grid cell
// (i, j) - the reference's bigdem[i][j] / bigwater[i][j], i in [0,R+1],
// j in [0,C+1] (src/WDPMCL.c:795-807) - lives at
//     (i + kPadTop) * pitch + (j + kPadLeft).
// Elevations are stored MASKED (relax.cuh): a cell with dem <= nodata holds the sentinel S.
// Everything outside the (R+2)x(C+2) padded grid is margin: dem = S,
// water = 0. A margin cell can never become a centre (dry) nor receive water
// (invalid neighbour), so kernels may compute on margins freely; this replaces
// the reference's row/col range guard (src/runoff.cl:145).
#pragma once

#include <cstdint>
#include <type_traits>
#include <cooperative_groups.h>
#include <cuda_runtime.h>

#include "../../include/wdpm_quantize.h"
#include "mw_schedule.h"
#include "relax.cuh"

namespace wdpm {

struct Geom {
    int R, C;          // interior rows / cols held by this solver
    int pitch;         // elements per device row (multiple of 32)
    int nrows_dev;     // device rows
    long long cells_dev() const { return (long long)pitch * nrows_dev; }
};

__device__ __forceinline__ size_t dev_index(const Geom& g, int i, int j) {
    return (size_t)(i + kPadTop) * (size_t)g.pitch + (size_t)(j + kPadLeft);
}

// ---------------------------------------------------------------------------
// Elementwise helpers
// ---------------------------------------------------------------------------

template <typename T>
__global__ void k_fill(T* __restrict__ a, long long n, T v) {
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
        a[i] = v;
}

// Mask the freshly uploaded DEM in place: dem <= nodata -> S (relax.cuh). Runs over the whole
// device array; margins already hold S, which the mask leaves alone.
template <typename T>
__global__ void k_mask_dem(T* __restrict__ d, long long n, T nodata) {
    for (long long k = blockIdx.x * (long long)blockDim.x + threadIdx.x; k < n; k += (long long)gridDim.x * blockDim.x)
        d[k] = mask_elevation(d[k], nodata);
}

// Add-module initial condition, valid cells only (src/WDPMCL.c:778-792). Every cell that is not a
// valid DEM cell holds the sentinel elevation, so the whole device array (halo rows of a stripe included)
// can be swept.
template <typename T>
__global__ void k_apply_add(T* __restrict__ w, const T* __restrict__ d, long long n, T depth, T depth_rof) {
    for (long long a = blockIdx.x * (long long)blockDim.x + threadIdx.x; a < n; a += (long long)gridDim.x * blockDim.x) {
        if (is_valid_elevation(d[a])) {
            T v = w[a];
            if (v > T(0)) v += depth;
            if (v <= T(0)) v = depth_rof;
            w[a] = v;
        }
    }
}

// Subtract-module initial condition (src/WDPMCL.c:919-926): max(w - depth, 0) with the
// host macro's tie rule (a > b ? a : b).
template <typename T>
__global__ void k_apply_subtract(T* __restrict__ w, const T* __restrict__ d, long long n, T depth) {
    for (long long a = blockIdx.x * (long long)blockDim.x + threadIdx.x; a < n; a += (long long)gridDim.x * blockDim.x) {
        if (is_valid_elevation(d[a])) {
            const T v = w[a] - depth;
            w[a] = (v > T(0)) ? v : T(0);
        }
    }
}

// What writing the water grid with "%f" and reading it back does to every valid cell
// (include/wdpm_quantize.h): lets chained modules keep the grid in HBM and still start from the
// values the reference's file hand-over gives them.
template <typename T>
__global__ void k_quantize_water(T* __restrict__ w, const T* __restrict__ d, long long n) {
    for (long long a = blockIdx.x * (long long)blockDim.x + threadIdx.x; a < n; a += (long long)gridDim.x * blockDim.x)
        if (is_valid_elevation(d[a])) w[a] = (T)wdpm_quantize6((double)w[a]);
}

// Does any cell that is not a valid DEM cell (NODATA, halo ring, margins) hold water != +0? (Never after the first
// block prologue for the reference's own files; the solver only needs to KNOW, see wdpm_solver::water_clean.)
template <typename T>
__global__ void k_check_invalid_water(const T* __restrict__ w, const T* __restrict__ d, long long n, int* __restrict__ dirty) {
    bool bad = false;
    for (long long a = blockIdx.x * (long long)blockDim.x + threadIdx.x; a < n; a += (long long)gridDim.x * blockDim.x) {
        const T v = w[a];
        bad = bad || (!is_valid_elevation(d[a]) && !(v == T(0) && !signbit(v)));
    }
    if (bad) *dirty = 1;
}

// Block prologue (src/WDPMCL.c:1055-1073): w < thres -> 0 over the whole padded
// grid (margins are 0 and stay 0), then snapshot. Also reports whether any invalid cell still holds
// water afterwards (k_check_invalid_water's question, asked again because the threshold pass is what
// clears the NODATA values a water file carries).
template <typename T>
__global__ void k_block_prologue(T* __restrict__ w, T* __restrict__ oldw, const T* __restrict__ d, long long n, T thres, int* __restrict__ dirty) {
    bool bad = false;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        T v = w[i];
        if (v < thres) v = T(0);
        w[i] = v;
        oldw[i] = v;
        bad = bad || (!is_valid_elevation(d[i]) && !(v == T(0) && !signbit(v)));
    }
    if (bad) *dirty = 1;
}

// ---------------------------------------------------------------------------
// Convergence + water balance (src/WDPMCL.c:1239-1268), two stages, fixed order.
// ---------------------------------------------------------------------------

struct BlockPartial {
    double max_diff;
    double sum;
    unsigned long long wet;
};

// Stage 1 walks the PADDED grid (not the device array), block b taking rows b, b+grid, ... and
// thread t columns t, t+NTHREADS, ...: the partial sums - hence the rounded total - depend only on
// (R, C, grid size), not on the kernel variant's pitch or margins.
template <typename T, int NTHREADS>
__global__ void __launch_bounds__(NTHREADS)
k_block_reduce_stage1(const T* __restrict__ w, const T* __restrict__ oldw, const T* __restrict__ d,
                      Geom g, BlockPartial* __restrict__ partials) {
    T md = T(0);
    double sum = 0.0;
    unsigned long long wet = 0;
    for (int i = blockIdx.x; i < g.R + 2; i += gridDim.x) {
        const size_t base = dev_index(g, i, 0);
        for (int j = threadIdx.x; j < g.C + 2; j += NTHREADS) {
            const size_t a = base + j;
            if (is_valid_elevation(d[a])) {
                const T v = w[a];
                T df = v - oldw[a];
                df = df < T(0) ? -df : df;
                md = df > md ? df : md;
                sum += (double)v;
                wet += (v > T(0)) ? 1ull : 0ull;
            }
        }
    }
    double mdd = (double)md;
    for (int off = 16; off > 0; off >>= 1) {
        const double om = __shfl_down_sync(0xffffffffu, mdd, off);
        mdd = om > mdd ? om : mdd;
        sum += __shfl_down_sync(0xffffffffu, sum, off);
        wet += __shfl_down_sync(0xffffffffu, wet, off);
    }
    __shared__ double s_md[NTHREADS / 32];
    __shared__ double s_sum[NTHREADS / 32];
    __shared__ unsigned long long s_wet[NTHREADS / 32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (lane == 0) { s_md[warp] = mdd; s_sum[warp] = sum; s_wet[warp] = wet; }
    __syncthreads();
    if (threadIdx.x == 0) {
        BlockPartial p{0.0, 0.0, 0ull};
        for (int k = 0; k < NTHREADS / 32; k++) {
            p.max_diff = s_md[k] > p.max_diff ? s_md[k] : p.max_diff;
            p.sum += s_sum[k];
            p.wet += s_wet[k];
        }
        partials[blockIdx.x] = p;
    }
}

__global__ void k_block_reduce_stage2(const BlockPartial* __restrict__ partials, int n, BlockPartial* __restrict__ out) {
    // single thread, fixed order: the sum is reproducible run to run
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        BlockPartial p{0.0, 0.0, 0ull};
        for (int k = 0; k < n; k++) {
            p.max_diff = partials[k].max_diff > p.max_diff ? partials[k].max_diff : p.max_diff;
            p.sum += partials[k].sum;
            p.wet += partials[k].wet;
        }
        *out = p;
    }
}

// Order-free part of the final statistics (src/WDPMCL.c:1394-1459) over the interior cells this solver owns:
// cells with dem > nodata (basincount, :1424-1431), of those the cells with more than 1 mm of water (watercount,
// :1395-1422: `water > 0.001`), and the deepest water on a valid cell (maxdepth, :1451-1459). Integer counts
// and a maximum do not depend on the order of evaluation; the volume sums of the report do (the reference adds
// the cells one by one in double) and stay with the host, which has the grid for the output file anyway.
struct FinalStats {
    unsigned long long valid_cells;
    unsigned long long wet_above_1mm;
    double max_depth;
};

template <typename T>
__global__ void k_final_stats(const T* __restrict__ w, const T* __restrict__ d, Geom g, int first_row, int n_rows, FinalStats* __restrict__ out) {
    unsigned long long nvalid = 0, nwet = 0;
    double md = -1.0e300;
    for (int i = first_row + blockIdx.x; i < first_row + n_rows; i += gridDim.x) {
        const size_t base = dev_index(g, i, 0);
        for (int j = 1 + threadIdx.x; j <= g.C; j += blockDim.x) {
            const T e = d[base + j];
            if (is_valid_elevation(e) || is_outlet(e)) {  // a Drain outlet is a valid cell wearing a mark
                const double v = (double)w[base + j];
                nvalid++;
                nwet += v > 0.001 ? 1ull : 0ull;
                md = v > md ? v : md;
            }
        }
    }
    for (int off = 16; off > 0; off >>= 1) {
        nvalid += __shfl_down_sync(0xffffffffu, nvalid, off);
        nwet += __shfl_down_sync(0xffffffffu, nwet, off);
        const double o = __shfl_down_sync(0xffffffffu, md, off);
        md = o > md ? o : md;
    }
    if ((threadIdx.x & 31) == 0) {
        if (nvalid) atomicAdd(&out->valid_cells, nvalid);
        if (nwet) atomicAdd(&out->wet_above_1mm, nwet);
        // maximum of doubles through their order-preserving integer image (water depths are >= 0 here or the max is of negatives too)
        long long bits = __double_as_longlong(md);
        bits = bits >= 0 ? bits : (long long)(0x8000000000000000ull - (unsigned long long)bits);
        atomicMax(reinterpret_cast<long long*>(&out->max_depth), bits);
    }
}

// Order-free 64-bit checksum of the interior water cells this solver owns: sum over cells of
// bits(w) * (2 * index + 1) modulo 2^64, index = the cell's position in the WHOLE DEM (row-major,
// 0-based). Integer addition commutes, so stripes can be summed in any order and the result does not depend
// on how the DEM is partitioned: equal checksums at 1, 2, 4, 8 GPUs mean equal grids (bit patterns and
// positions). Benchmarks report it; nothing in the solver reads it.
template <typename T>
__global__ void k_water_checksum(const T* __restrict__ w, Geom g, int first_row, int n_rows, int global_row0, int dem_cols,
                                 unsigned long long* __restrict__ out) {
    unsigned long long acc = 0;
    for (int i = first_row + blockIdx.x; i < first_row + n_rows; i += gridDim.x) {
        const size_t base = dev_index(g, i, 0);
        const unsigned long long row_index = (unsigned long long)(global_row0 + i - 1) * (unsigned long long)dem_cols;
        for (int j = 1 + threadIdx.x; j <= g.C; j += blockDim.x) {
            unsigned long long bits;
            if (sizeof(T) == 8) bits = (unsigned long long)__double_as_longlong((double)w[base + j]);
            else bits = (unsigned long long)(unsigned)__float_as_int((float)w[base + j]);
            acc += bits * (2ull * (row_index + (unsigned long long)(j - 1)) + 1ull);
        }
    }
    for (int off = 16; off > 0; off >>= 1) acc += __shfl_down_sync(0xffffffffu, acc, off);
    if ((threadIdx.x & 31) == 0 && acc) atomicAdd(out, acc);
}

// ---------------------------------------------------------------------------
// Drain outlet search (src/WDPMCL.c:1005-1017): min dem over dem > 0, first in
// row-major order of the padded grid on ties.
// ---------------------------------------------------------------------------

struct OutletCand {
    double elev;
    long long index;  // i*(C+2)+j in padded coordinates; -1 = none
};

__device__ __forceinline__ OutletCand better(OutletCand a, OutletCand b) {
    if (a.index < 0) return b;
    if (b.index < 0) return a;
    if (b.elev < a.elev || (b.elev == a.elev && b.index < a.index)) return b;
    return a;
}

template <typename T, int NTHREADS>
__global__ void __launch_bounds__(NTHREADS)
k_find_outlet_stage1(const T* __restrict__ d, Geom g, OutletCand* __restrict__ partials) {
    OutletCand best{1.0e8, -1};  // the reference starts from mindrain = 100000000 with strict '<'
    const long long n = (long long)(g.R + 2) * (g.C + 2);
    for (long long k = blockIdx.x * (long long)NTHREADS + threadIdx.x; k < n; k += (long long)gridDim.x * NTHREADS) {
        const int i = (int)(k / (g.C + 2)), j = (int)(k - (long long)i * (g.C + 2));
        const double v = (double)d[dev_index(g, i, j)];
        if (v > 0.0 && v < 1.0e8) best = better(best, OutletCand{v, k});
    }
    __shared__ OutletCand s[NTHREADS];
    s[threadIdx.x] = best;
    __syncthreads();
    for (int off = NTHREADS / 2; off > 0; off >>= 1) {
        if ((int)threadIdx.x < off) s[threadIdx.x] = better(s[threadIdx.x], s[threadIdx.x + off]);
        __syncthreads();
    }
    if (threadIdx.x == 0) partials[blockIdx.x] = s[0];
}

__global__ void k_find_outlet_stage2(const OutletCand* __restrict__ partials, int n, OutletCand* __restrict__ out) {
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        OutletCand best{1.0e8, -1};
        for (int k = 0; k < n; k++) best = better(best, partials[k]);
        *out = best;
    }
}

// ---------------------------------------------------------------------------
// Drain bookkeeping. Every outlet has its own accumulator in the solver's precision (one outlet:
// the reference's totaldrain, src/runoff.cl:108). An event is the pair of addends of one outlet
// contact, folded as (total + w_outlet) + w_centre, in sub-pass order. An outlet is a neighbour of
// at most one centre per colour sub-pass, so (outlet, sub-pass) identifies a contact.
// The set is sorted by (row, col) when it is installed (solver.cu); kernels find an outlet by binary search
// and keep its total at its sorted position.
// ---------------------------------------------------------------------------

template <typename T>
struct DrainPair {
    T w_outlet;
    T w_centre;
};

// Event buffers rotate over kEventSlots launches: launch L records into buffer L % 3 and folds buffer (L-1) % 3.
// Three, not two, because of row stripes: a contact is recorded in the buffer of the stripe that OWNS THE OUTLET
// (over NVLink when the centre lies in the neighbouring stripe - an outlet within one row of a stripe border is
// drained by centres of both stripes), so that one accumulator sees all contacts of an outlet in sub-pass order and
// its total does not depend on the partition. The neighbour's launch L+1 may start (and record) while this
// stripe's launch L+1 is still folding buffer L % 3; launch L+2 of the neighbour, which reuses buffer (L-1) % 3,
// cannot start before this stripe's launch L+1 has finished (halo flags), i.e. after that buffer was folded.
constexpr int kEventSlots = 3;
__host__ __device__ __forceinline__ int next_event_slot(int s) { return s == kEventSlots - 1 ? 0 : s + 1; }
__host__ __device__ __forceinline__ int prev_event_slot(int s) { return s == 0 ? kEventSlots - 1 : s - 1; }

// An event area: per buffer and entry a bit mask of the sub-pass slots that hold a contact, the addends of those
// contacts at their slots, and the list of entries touched since the buffer was last folded. Recording sets a bit
// (the first bit of an entry appends the entry to the list); folding walks the list only, so it costs time in
// proportion to the outlets that were touched, not to the size of the set. Two areas exist:
//  - the outlet area, one entry per outlet (sorted position), allocated when the set is installed;
//  - row stripes only, the border area, one entry per column of the stripe's first and of its last owned row,
//    allocated with the stripe's arrival flags (one IPC handle covers both; a neighbour records there the
//    contacts of its centres with my outlets). Every contact with an outlet in one of those two rows goes there,
//    whichever stripe's centre made it, so each outlet's events stay in one place.
struct EventCounters {
    int n_touched[kEventSlots];  // entries on each buffer's touched list
    int fold_done[kEventSlots];  // thread groups that have folded the buffer (the last one empties the lists)
};

template <typename T>
struct EventArea {
    EventCounters* ctr;
    unsigned long long* mask;  // [kEventSlots][n]
    int* touched;              // [kEventSlots][n]
    DrainPair<T>* vals;        // [kEventSlots][n][slots]
    int n;                     // entries (0 = no area)
    int slots;                 // sub-pass slots per entry and buffer: 9 per iteration of a launch, + 1 (kWipeSlot)
};

__host__ __device__ __forceinline__ size_t event_area_bytes(long long n, int slots, size_t esize) {
    const size_t mask_off = 256, touched_off = mask_off + (size_t)kEventSlots * n * 8;
    const size_t vals_off = (touched_off + (size_t)kEventSlots * n * 4 + 15) / 16 * 16;
    return vals_off + (size_t)kEventSlots * n * slots * 2 * esize;
}

template <typename T>
__host__ __device__ __forceinline__ EventArea<T> event_area(void* base, int n, int slots) {
    EventArea<T> a;
    char* b = static_cast<char*>(base);
    const size_t touched_off = 256 + (size_t)kEventSlots * n * 8;
    a.ctr = reinterpret_cast<EventCounters*>(b);
    a.mask = reinterpret_cast<unsigned long long*>(b + 256);
    a.touched = reinterpret_cast<int*>(b + touched_off);
    a.vals = reinterpret_cast<DrainPair<T>*>(b + (touched_off + (size_t)kEventSlots * n * 4 + 15) / 16 * 16);
    a.n = base ? n : 0;
    a.slots = slots;
    return a;
}

template <typename T>
struct DrainState {
    T* totaldrain;          // [n_outlets] device accumulators, in sorted order
    const int* outlet_rc;   // [n_outlets][2] padded (row, col) of each outlet in this solver's rows, sorted by (row, col)
    int n_outlets;
    EventArea<T> ev;        // outlet area
    // row stripes: this stripe's border area and its neighbours' (peer memory; n = 0: none), and its owned rows
    EventArea<T> border, border_up, border_dn;
    int P;
    int border_cols;        // entries per border row (cols + 2)
    const unsigned char* cta_outlets;  // fused kernels: [CTA] 1 = an outlet lies in the rows and columns the CTA stages
};

// sorted position of the outlet at padded (row, col); -1 if none (cannot happen for a marked cell)
template <typename T>
__device__ __forceinline__ int outlet_index(const DrainState<T>& ds, int row, int col) {
    int lo = 0, hi = ds.n_outlets;  // first position whose (row, col) is not below the key
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        const int r = ds.outlet_rc[2 * mid], c = ds.outlet_rc[2 * mid + 1];
        if (r < row || (r == row && c < col)) lo = mid + 1;
        else hi = mid;
    }
    return (lo < ds.n_outlets && ds.outlet_rc[2 * lo] == row && ds.outlet_rc[2 * lo + 1] == col) ? lo : -1;
}

// Fold entries first, first + stride, ... of the touched list of `buffer` in area `a` into their outlets' totals,
// slot by slot in sub-pass order.
template <typename T>
__device__ __forceinline__ void fold_area(const DrainState<T>& ds, const EventArea<T>& a, bool border, int buffer, int first, int stride) {
    const int n = *reinterpret_cast<volatile int*>(&a.ctr->n_touched[buffer]);
    for (int i = first; i < n; i += stride) {
        const int entry = a.touched[(size_t)buffer * a.n + i];
        const size_t e = (size_t)buffer * a.n + entry;
        unsigned long long m = a.mask[e];
        a.mask[e] = 0ull;
        const int k = border ? outlet_index(ds, entry < ds.border_cols ? 0 : ds.P - 1, entry % ds.border_cols) : entry;
        if (k < 0) continue;
        const DrainPair<T>* v = a.vals + e * a.slots;
        T td = ds.totaldrain[k];
        while (m) {
            const int s = __ffsll((long long)m) - 1;
            m &= m - 1;
            td = td + v[s].w_outlet;
            td = td + v[s].w_centre;
        }
        ds.totaldrain[k] = td;
    }
}

// Fold one event buffer: the calling threads split the touched entries (thread `first` of `stride`). Every group
// of threads that takes part must then call fold_finish once, after a barrier over the group.
template <typename T>
__device__ __forceinline__ void fold_events(const DrainState<T>& ds, int buffer, int first, int stride) {
    fold_area(ds, ds.ev, false, buffer, first, stride);
    if (ds.border.n) fold_area(ds, ds.border, true, buffer, first, stride);
}

// One thread per group that folded `buffer` (`groups` of them): the last to arrive empties the touched lists.
template <typename T>
__device__ __forceinline__ void fold_finish(const DrainState<T>& ds, int buffer, int groups) {
    if (atomicAdd(&ds.ev.ctr->fold_done[buffer], 1) == groups - 1) {
        ds.ev.ctr->n_touched[buffer] = 0;
        if (ds.border.n) ds.border.ctr->n_touched[buffer] = 0;
        ds.ev.ctr->fold_done[buffer] = 0;
    }
}

template <typename T>
__global__ void k_fold_events(DrainState<T> ds, int buffer) {
    fold_events(ds, buffer, (int)(blockIdx.x * blockDim.x + threadIdx.x), (int)(gridDim.x * blockDim.x));
    __syncthreads();
    if (threadIdx.x == 0) fold_finish(ds, buffer, (int)gridDim.x);
}

// Mark / unmark outlet cells in the elevation grid (relax.cuh, outlet_mark). `saved` keeps the
// elevations the marks replace so they can be restored (module change, new outlet set). Marking also counts in
// `bad` the outlets on cells of local rows [data_lo, data_hi) (the rows that hold DEM data) with dem <= nodata.
template <typename T>
__global__ void k_mark_outlets(T* __restrict__ d, Geom g, const int* __restrict__ rc, int n, T* __restrict__ saved, int restore,
                               int data_lo, int data_hi, int* __restrict__ bad) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n) return;
    const int i = rc[2 * k], j = rc[2 * k + 1];
    if (i < -kPadTop || i >= g.nrows_dev - kPadTop || j < 0 || j > g.C + 1) return;  // not in this solver's rows
    const size_t a = dev_index(g, i, j);
    if (restore) {
        d[a] = saved[k];
    } else {
        if (i >= data_lo && i < data_hi && !is_valid_elevation(d[a])) atomicAdd(bad, 1);
        saved[k] = d[a];
        d[a] = outlet_mark<T>();
    }
}

// Totals seeded from the water under the outlets (src/WDPMCL.c:1029 per outlet): max(w, 0) where this solver owns
// the outlet's row, 0 elsewhere.
template <typename T>
__global__ void k_seed_outlets(const T* __restrict__ w, Geom g, DrainState<T> ds) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= ds.n_outlets) return;
    const int i = ds.outlet_rc[2 * k], j = ds.outlet_rc[2 * k + 1];
    T v = T(0);
    if (i >= 0 && i < ds.P) {
        const T x = w[dev_index(g, i, j)];
        v = x > T(0) ? x : T(0);
    }
    ds.totaldrain[k] = v;
}

// The reported total: the outlets' totals added in the caller's order, in the solver's precision. One thread:
// the order is the definition (an outlet-order sum of the host-side totals gives the same bits).
template <typename T>
__global__ void k_sum_totals(const T* __restrict__ totals, const int* __restrict__ pos, int n, double* __restrict__ out) {
    if (blockIdx.x != 0 || threadIdx.x != 0) return;
    T t = totals[pos[0]];
    for (int k = 1; k < n; k++) t = t + totals[pos[k]];
    *out = (double)t;
}

// Checkpoint capture: the outlets' totals in the caller's order, widened to double (exact for both precisions).
template <typename T>
__global__ void k_gather_totals(const T* __restrict__ totals, const int* __restrict__ pos, int n, double* __restrict__ out) {
    for (int k = blockIdx.x * blockDim.x + threadIdx.x; k < n; k += gridDim.x * blockDim.x) out[k] = (double)totals[pos[k]];
}

// Record one event: its addends go into slot `slot` of `entry` in buffer `buffer` of area `a`. `sys`: a border
// area, into which the neighbour's centres record from another GPU too (system-scope atomics); only this solver's
// kernels write its outlet area.
template <typename T>
__device__ __forceinline__ void record_event(const EventArea<T>& a, int buffer, int entry, int slot, T w_outlet, T w_centre, bool sys) {
    const size_t e = (size_t)buffer * a.n + entry;
    DrainPair<T>* v = a.vals + e * a.slots + slot;
    v->w_outlet = w_outlet;
    v->w_centre = w_centre;
    const unsigned long long bit = 1ull << slot;
    const bool first = (sys ? atomicOr_system(&a.mask[e], bit) : atomicOr(&a.mask[e], bit)) == 0ull;
    if (first) a.touched[(size_t)buffer * a.n + (sys ? atomicAdd_system(&a.ctr->n_touched[buffer], 1) : atomicAdd(&a.ctr->n_touched[buffer], 1))] = entry;
}

// Where the events of the outlet at local padded (orow, ocol) go: a border area (row stripes: the outlet's row is
// the first or last owned row of this stripe or of a neighbour) or the outlet area.
template <typename T>
__device__ __forceinline__ void route_event(const DrainState<T>& ds, int buffer, int slot, int orow, int ocol, T w_outlet, T w_centre) {
    if (ds.border_up.n && orow < 0) { record_event(ds.border_up, buffer, ds.border_cols + ocol, slot, w_outlet, w_centre, true); return; }
    if (ds.border_dn.n && orow >= ds.P) { record_event(ds.border_dn, buffer, ocol, slot, w_outlet, w_centre, true); return; }
    if (ds.border.n && orow == 0) { record_event(ds.border, buffer, ocol, slot, w_outlet, w_centre, true); return; }
    if (ds.border.n && orow == ds.P - 1) { record_event(ds.border, buffer, ds.border_cols + ocol, slot, w_outlet, w_centre, true); return; }
    const int k = outlet_index(ds, orow, ocol);
    if (k >= 0) record_event(ds.ev, buffer, k, slot, w_outlet, w_centre, false);
}

// Record one contact of a centre with the outlet at padded (orow, ocol): its two addends go into slot
// (outlet, sub-pass `slot`) of event buffer `buffer` of the stripe that owns the outlet's row, to be folded in
// sub-pass order (fold_events). `direct` (colour kernel: one launch per sub-pass, a single writer per outlet) adds
// them to the total at once.
template <typename T>
__device__ __forceinline__ void record_contact(const DrainState<T>& ds, int buffer, int slot, int orow, int ocol, T w_outlet, T w_centre, bool direct) {
    if (direct) {
        const int k = outlet_index(ds, orow, ocol);
        if (k < 0) return;
        T td = ds.totaldrain[k];
        td = td + w_outlet;
        td = td + w_centre;
        ds.totaldrain[k] = td;
        return;
    }
    route_event(ds, buffer, slot, orow, ocol, w_outlet, w_centre);
}

// ---------------------------------------------------------------------------
// Serial-schedule Drain (include/wdpm_b200.h, WDPM_SCHEDULE_SERIAL): after every whole iteration the
// reference's drain() (src/WDPMCL.c:1859-1897) sums the water of the outlet's 3x3 cells that are valid
// and wet, in row-major order from 0, adds the sum to totaldrain and zeroes all nine cells. One outlet.
// The outlet cell itself is valid: on the device it wears the mark (relax.cuh, outlet_mark).
// In an event buffer the sum travels as one event in slot kWipeSlot, after the nine sub-pass slots of
// a one-iteration launch, so that fold_events adds it after that iteration's contacts:
// (total + got) + 0 == total + got, because total + got is never -0.0 (got >= +0).
// ---------------------------------------------------------------------------

constexpr int kWipeSlot = 9;  // an area's slots per entry are 9 * iterations per launch + 1 > kWipeSlot

template <typename T>
__device__ __forceinline__ T outlet_wipe_sum(const T* w, const T* d, size_t pitch) {
    T got = T(0);
    for (int a = -1; a <= 1; a++)
        for (int b = -1; b <= 1; b++) {
            const T e = d[a * (ptrdiff_t)pitch + b], v = w[a * (ptrdiff_t)pitch + b];
            if ((is_valid_elevation(e) || is_outlet(e)) && v > T(0)) got = got + v;
        }
    return got;
}

// One thread. Zeroes the nine cells of w that this solver's memory holds (a row stripe: its owned rows and the
// halo copies of its neighbours' rows, which arrived with the neighbours' export of the same iteration); the
// solver that owns the outlet's row first takes the sum. `direct` adds it to the total at once (colour kernel),
// otherwise it goes to event buffer `buffer`.
template <typename T>
__global__ void k_outlet_wipe(T* __restrict__ w, const T* __restrict__ d, Geom g, DrainState<T> ds, int buffer, int direct) {
    if (blockIdx.x != 0 || threadIdx.x != 0) return;
    const int orow = ds.outlet_rc[0], ocol = ds.outlet_rc[1];
    if (orow >= 0 && orow < ds.P) {
        const size_t c = dev_index(g, orow, ocol);
        const T got = outlet_wipe_sum(w + c, d + c, (size_t)g.pitch);
        if (direct) {
            ds.totaldrain[0] = ds.totaldrain[0] + got;
        } else {
            route_event(ds, buffer, kWipeSlot, orow, ocol, got, T(0));
        }
    }
    for (int i = orow - 1; i <= orow + 1; i++)
        if (i >= -kPadTop && i < g.nrows_dev - kPadTop)
            for (int j = ocol - 1; j <= ocol + 1; j++) w[dev_index(g, i, j)] = T(0);
}

// A Drain tile whose 3x3 holds outlets (rare): relax it in place and record the contacts. Out of line
// so that its arrays live on the stack of this call only. `owner`: this CTA owns the centre, so it
// reports the events (halo copies recompute the same contacts). `slot`: sub-pass slot in the buffer.
template <typename T>
__device__ __noinline__ void drain_tile_near_outlets(T* w0, T* w1, T* w2, const T* d0, const T* d1, const T* d2, int j,
                                                     int mask, DrainState<T> ds, int buffer, int slot, int crow, int ccol,
                                                     bool owner, bool direct) {
    T evo[8], evc[8];
    int pos[8];
    const int n = relax_tile_near_outlets<T>(w0, w1, w2, d0, d1, d2, j, mask, evo, evc, pos);
    if (!owner) return;
    for (int i = 0; i < n; i++)
        record_contact<T>(ds, buffer, slot, crow + pos[i] / 3 - 1, ccol + pos[i] % 3 - 1, evo[i], evc[i], direct);
}

// ---------------------------------------------------------------------------
// Row-stripe halo exchange over NVLink (peer stores + arrival flags), fused into k_fused:
// in iteration `epoch` a stripe writes, with the bulk stores that write its rows home,
//   its first HB owned rows  -> the stripe above, as that stripe's rows [P_above, P_above+HB)
//   its last  HA owned rows  -> the stripe below, as that stripe's rows [-HA, 0)
// (HA = 3, HB = 6: what one fused iteration reads beyond its owned rows; only the owned columns of
// each strip travel - the margins never change), and the CTA that finishes last publishes `epoch`
// in the neighbours' arrival flags. k_halo_wait holds the next launch until both halos are in.
// ---------------------------------------------------------------------------

constexpr int kHaloAbove = 3;
constexpr int kHaloBelow = 6;

struct HaloFlags {
    int from_above;   // epoch of the last halo received from the stripe above
    int from_below;
    int push_count;   // CTAs of the running iteration kernel whose rows for the stripe above have landed
    int push_count_dn;  // ... for the stripe below
    int error;        // set if a wait gave up
};

__device__ __forceinline__ int ld_acquire_sys(const int* p) {
    int v;
    asm volatile("ld.acquire.sys.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_release_sys(int* p, int v) {
    asm volatile("st.release.sys.global.s32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}

__device__ __forceinline__ unsigned long long global_timer_ns() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}

// Hold the stream until both neighbours' halos of iteration `epoch` have landed. A neighbour that does not
// show up within `timeout_ns` (dead rank, host stuck for longer than the host allows) sets the sticky
// HaloFlags::error; every later wait then returns at once, and the host reports WDPM_E_HALO at the end of
// the block (solver.cu, block_end_t) instead of a water grid computed on stale halo rows.
__global__ void k_halo_wait(HaloFlags* flags, int need_above, int need_below, int epoch, unsigned long long timeout_ns) {
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    if (ld_acquire_sys(&flags->error)) return;
    const unsigned long long t0 = global_timer_ns();
    for (unsigned spins = 0;; spins++) {
        const bool ok_a = !need_above || ld_acquire_sys(&flags->from_above) >= epoch;
        const bool ok_b = !need_below || ld_acquire_sys(&flags->from_below) >= epoch;
        if (ok_a && ok_b) return;
        if ((spins & 63u) == 63u && global_timer_ns() - t0 > timeout_ns) {
            flags->error = 1;
            __threadfence_system();
            return;
        }
        __nanosleep(200);
    }
}

// ---------------------------------------------------------------------------
// Colour kernel: one launch per colour sub-pass on global memory, in place.
// This is the reference's schedule (src/WDPMCL.c:1184-1206) - the baseline the
// fused kernel is checked against and the path for grids too small to tile.
// Thread (gx, gy) owns centre row = oi + 3*gy, col = oj + 3*gx (1-based padded).
// ---------------------------------------------------------------------------

template <typename T, int MODULE>
__global__ void __launch_bounds__(256)
k_colour(T* __restrict__ w, const T* __restrict__ d, Geom g, int oi, int oj, DrainState<T> ds) {
    const int gx = blockIdx.x * blockDim.x + threadIdx.x;
    const int gy = blockIdx.y * blockDim.y + threadIdx.y;
    const int row = oi + 3 * gy, col = oj + 3 * gx;
    if (row > g.R || col > g.C) return;
    const size_t c = dev_index(g, row, col);
    T* w1 = w + c;
    const T* d1 = d + c;
    if (MODULE == kDrain) {
        const int mask = outlet_mask_3x3<T>(d1 - g.pitch, d1, d1 + g.pitch, 0);
        if (mask) {
            drain_tile_near_outlets<T>(w1 - g.pitch, w1, w1 + g.pitch, d1 - g.pitch, d1, d1 + g.pitch, 0, mask, ds, 0, 0,
                                       row, col, true, true);
            return;
        }
    }
    relax_tile<T, MODULE>(w1 - g.pitch, w1, w1 + g.pitch, d1 - g.pitch, d1, d1 + g.pitch, 0);
}

// ---------------------------------------------------------------------------
// Fused kernel: K whole iterations (9K colour sub-passes) per launch.
// See mw_schedule.h for the schedule. Data movement is TMA bulk copies
// (cp.async.bulk, SASS UBLKCP) global -> shared completing on mbarriers, and
// shared -> global bulk stores in bulk async-groups; compute is plain SIMT on
// the shared-memory row ring (stride-3 access is bank-conflict free).
// ---------------------------------------------------------------------------

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "WAIT_%=:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra DONE_%=;\n\t"
        "bra WAIT_%=;\n\t"
        "DONE_%=:\n\t}" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
__device__ __forceinline__ void bulk_load(void* smem_dst, const void* gmem_src, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(smem_u32(smem_dst)), "l"(gmem_src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void bulk_store(void* gmem_dst, const void* smem_src, uint32_t bytes) {
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;"
                 ::"l"(gmem_dst), "r"(smem_u32(smem_src)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void bulk_wait_read() { asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory"); }
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void fence_mbar_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }

template <typename T>
struct FusedParams {
    const T* w_in;
    T* w_out;
    const T* dem;
    Geom g;
    int n_strips;
    int chunk_triples;  // owned row triples per CTA
    int total_triples;  // ceil((R+2)/3)
    int launch_slot;    // drain event buffer written by this launch (0 .. kEventSlots-1)
    DrainState<T> ds;
    // Row stripes: the halo exchange is part of this kernel. Rows the neighbouring stripes read
    // (my first kHaloBelow owned rows for the stripe above, my last kHaloAbove for the stripe below)
    // are written to the neighbour's buffer over NVLink by the same bulk stores that write them home,
    // and the last of the CTAs that own such rows publishes the iteration number in that neighbour's
    // arrival flag - for the stripe above that is after the first wave of CTAs, so its halo travels
    // while the rest of this stripe is still being computed.
    T* up_out;          // the buffer of the stripe above that takes this iteration's rows (nullptr: none)
    T* dn_out;
    int P_self, P_up;   // owned padded rows of this stripe / of the stripe above
    HaloFlags* self_flags;
    HaloFlags* up_flags;
    HaloFlags* dn_flags;
    int up_ctas, dn_ctas;  // CTAs counted in before the upward / downward flag rises (the last of them raises it)
    int epoch;
#ifdef WDPM_TEST_HOOKS
    // Test builds only (tests/test_gpu_halo_race.py; never compiled into the product library):
    int dbg_old_dn_count;    // count only the CTAs that OWN exported rows, as the kernel did before the fix
    int dbg_reader_delay_ns; // CTAs that only READ the bottom halo sleep this long before their first load
#endif
};

template <typename CFG, typename T>
constexpr size_t fused_smem_bytes() {
    return (size_t)2 * CFG::NRING * CFG::W * sizeof(T) + CFG::NSTAGE * sizeof(uint64_t) + 16;
}

// OPT bit 0 (fp64 Add only; in fp32 the predicated-add form measured faster): cap-free, sign-gated neighbour step (relax.cuh, push_add_fast) - 12 instead
// of 15 instructions per neighbour, 7 instead of 9 of them on the FP64 pipe.
constexpr int kOptAddFast = 1;
// OPT bit 1: REGISTER REALLOCATION. The register file hands registers to groups of four warps, so a
// CTA of 24 compute warps + 1 data-movement warp is budgeted as 28 warps: 72 registers per thread,
// where 24 warps alone could have 80 (measured: scripts/micro/reg_granularity.cu). With this bit the
// CTA is launched with a whole fourth warp group (4 warps, one of them the data-movement warp, the
// others exit at once); that group gives its registers back (setmaxnreg.dec to 24) and the compute
// warps take them (setmaxnreg.inc to 80): 28*72 = 4*24 + 24*80. (16 compute warps: 96 -> 112.)
constexpr int kOptRegRealloc = 2;
// OPT bit 2 (fp64 Drain only): gate and max(flow,0) folded into the scaling factor (relax.cuh,
// push_drain_fast) - 31 instead of 34 issue cycles per neighbour. Valid when water is never -0.0, which a
// zero threshold > 0 guarantees; the solver picks the variant accordingly.
constexpr int kOptDrainFast = 4;
__host__ __device__ constexpr int fused_extra_threads(int opt) { return (opt & kOptRegRealloc) ? 128 : 32; }

#ifdef WDPM_TEST_HOOKS
__device__ int g_dbg_counters[4];  // 0: reader CTAs delayed
#endif

#ifdef WDPM_TIMELINE
// Developer probe (never compiled into the product library): per-warp clock64 stamps of one CTA.
constexpr int kTlSteps = 8, kTlWarps = 32, kTlPoints = 10;
__device__ long long g_timeline[kTlSteps * kTlWarps * kTlPoints];
__device__ int g_timeline_cta = 300, g_timeline_step0 = 100;
#define WDPM_TL(point)                                                                                   \
    do {                                                                                                 \
        if ((int)blockIdx.x == g_timeline_cta && (threadIdx.x & 31) == 0 && s >= g_timeline_step0 &&       \
            s < g_timeline_step0 + kTlSteps)                                                             \
            g_timeline[((s - g_timeline_step0) * kTlWarps + (threadIdx.x >> 5)) * kTlPoints + (point)] = clock64(); \
    } while (0)
#else
#define WDPM_TL(point) do { } while (0)
#endif

// ---------------------------------------------------------------------------
// Data movement of the iteration kernels (k_fused, k_fused_wa): one elected lane of a dedicated warp
// issues every bulk copy. Per step: write home the rows the last phase finished in the step before
// (plus, for row stripes, the copies into the neighbours' halo rows), release ring slots once their
// write-back has read them, prefetch the rows of step s + PF. At the end: the halo handshake.
// ---------------------------------------------------------------------------

template <typename CFG>
__device__ __forceinline__ bool step_has_loads(const MwTile<CFG>& tile, int s) {
    for (int t = 0; t < CFG::NT; t++)
        if (tile.staged(tile.triple(s, 0, t))) return true;
    return false;
}

template <typename CFG, typename T>
__device__ __forceinline__ void issue_row_loads(const FusedParams<T>& p, const MwTile<CFG>& tile, T* ring_w, T* ring_d, uint64_t* bars, int s) {
    constexpr uint32_t kRowBytes = CFG::W * sizeof(T);
    const size_t col0 = (size_t)(tile.x0 + kPadLeft);  // device column of window column 0; multiple of 4 elements by construction
    uint64_t* bar = &bars[s % CFG::NSTAGE];
    int nrows = 0;
    for (int t = 0; t < CFG::NT; t++)
        if (tile.staged(tile.triple(s, 0, t))) nrows += 3;
    if (nrows == 0) return;
    mbar_expect_tx(bar, (uint32_t)(2 * nrows) * kRowBytes);
    for (int t = 0; t < CFG::NT; t++) {
        const int m = tile.triple(s, 0, t);
        if (!tile.staged(m)) continue;
        for (int k = 0; k < 3; k++) {
            const int row = 3 * m + k;
            const size_t src = (size_t)(row + kPadTop) * (size_t)p.g.pitch + col0;
            const int slot = tile.ring_slot(row);
            bulk_load(ring_w + (size_t)slot * CFG::W, p.w_in + src, kRowBytes, bar);
            bulk_load(ring_d + (size_t)slot * CFG::W, p.dem + src, kRowBytes, bar);
        }
    }
}

// rows finished by the last phase in step s: C-type rows 3m+2 .. 3m+4 (only_t >= 0: of that triple slot only)
template <typename CFG, typename T>
__device__ __forceinline__ void issue_row_stores(const FusedParams<T>& p, const MwTile<CFG>& tile, T* ring_w, int s, int only_t = -1) {
    const size_t col0 = (size_t)(tile.x0 + kPadLeft);
    bool any = false;
    for (int t = 0; t < CFG::NT; t++) {
        if (only_t >= 0 && t != only_t) continue;
        const int m = tile.triple(s, CFG::NPH - 1, t);
        for (int k = 0; k < 3; k++) {
            const int row = 3 * m + 2 + k;
            if (!tile.owns_row(row)) continue;
            const size_t dst = (size_t)(row + kPadTop) * (size_t)p.g.pitch + col0 + CFG::HL;
            const T* src = ring_w + (size_t)tile.ring_slot(row) * CFG::W + CFG::HL;
            bulk_store(p.w_out + dst, src, CFG::TWV * sizeof(T));
            if (p.up_out && row < kHaloBelow)  // ... and into the bottom halo of the stripe above
                bulk_store(p.up_out + (size_t)(row + p.P_up + kPadTop) * (size_t)p.g.pitch + col0 + CFG::HL, src, CFG::TWV * sizeof(T));
            if (p.dn_out && row >= p.P_self - kHaloAbove && row < p.P_self)  // ... the top halo of the stripe below
                bulk_store(p.dn_out + (size_t)(row - p.P_self + kPadTop) * (size_t)p.g.pitch + col0 + CFG::HL, src, CFG::TWV * sizeof(T));
            any = true;
        }
    }
    if (any) bulk_commit();
}

// End of a stripe's iteration kernel: say that my rows have landed in the neighbours' memory and that I have read
// my halo rows (see FusedParams); the last CTA to say so raises the neighbour's arrival flag.
template <typename CFG, typename T>
__device__ __forceinline__ void halo_handshake(const FusedParams<T>& p, const MwTile<CFG>& tile) {
    const bool exp_up = p.up_flags && 3 * tile.m0 < kHaloBelow;
    // downwards the flag also licenses the stripe below to overwrite MY bottom-halo rows [P, P+kHaloBelow) in the
    // buffer this iteration reads, so every CTA that STAGES one of those rows counts (3*(m1+BOT_TRIPLES) > P), not
    // only those that own the exported rows; such a CTA may export nothing and only bumps the counter.
#ifdef WDPM_TEST_HOOKS
    const int dn_reach = p.dbg_old_dn_count ? kHaloAbove : kHaloBelow;
#else
    constexpr int dn_reach = kHaloBelow;
#endif
    const bool exp_dn = p.dn_flags && 3 * tile.m1 > p.P_self - dn_reach && 3 * tile.m0 < p.P_self;
    if (exp_up || exp_dn) {
        // my rows have landed, also in the neighbour's memory; the CTA that is last to say so raises the flag
        asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
        __threadfence_system();
        if (exp_up && atomicAdd(&p.self_flags->push_count, 1) == p.up_ctas - 1) {
            p.self_flags->push_count = 0;
            __threadfence_system();
            st_release_sys(&p.up_flags->from_below, p.epoch);
        }
        if (exp_dn && atomicAdd(&p.self_flags->push_count_dn, 1) == p.dn_ctas - 1) {
            p.self_flags->push_count_dn = 0;
            __threadfence_system();
            st_release_sys(&p.dn_flags->from_above, p.epoch);
        }
    }
}

// NBAR = CTA-wide barriers per step the compute threads execute (this warp takes part in each)
template <typename CFG, typename T, int NBAR>
__device__ __forceinline__ void data_movement_warp(const FusedParams<T>& p, const MwTile<CFG>& tile, T* ring_w, T* ring_d, uint64_t* bars, bool lead) {
    constexpr int PF = CFG::PF;
#ifdef WDPM_TEST_HOOKS
    if (lead && p.dn_flags && p.dbg_reader_delay_ns > 0 && 3 * tile.m1 > p.P_self - kHaloBelow &&
        3 * tile.m1 <= p.P_self - kHaloAbove) {  // reads rows [P, P+3) of w_in but exports nothing: make it late
        const unsigned long long t0 = global_timer_ns();
        while (global_timer_ns() - t0 < (unsigned long long)p.dbg_reader_delay_ns) __nanosleep(1000);
        atomicAdd(&g_dbg_counters[0], 1);
        // has the stripe below already finished the NEXT iteration (whose export overwrites the halo rows I am about to read)?
        if (ld_acquire_sys(&p.self_flags->from_below) > p.epoch) atomicAdd(&g_dbg_counters[1], 1);
    }
#endif
    if (lead)
        for (int s = 0; s < PF && s < tile.n_steps; s++) issue_row_loads<CFG, T>(p, tile, ring_w, ring_d, bars, s);
    for (int s = 0; s < tile.n_steps; s++) {
        WDPM_TL(0);
        if (lead) {
            // The prefetch goes out first: phase 0 of step s + PF waits for it, and at PF = 1 a step is barely longer
            // than the trip to HBM. The ring slots it overwrites belonged to rows written home by the store group
            // of step s - 2 (committed a whole step ago), which must have been read out: every group committed so
            // far. The rows of step s - 1, stored just below, lie elsewhere in the ring (mw_schedule.h, NRING_MIN).
            if (CFG::STRICT_ORDER) {
                // deep prefetch (mw_schedule.h, WaCfg::RING_PF): the rows loaded now take the place of the rows
                // written home now, so the write-backs go first and must have read their rows out
                if (s > 0) issue_row_stores<CFG, T>(p, tile, ring_w, s - 1);
                bulk_wait_read<0>();
                if (s + PF < tile.n_steps) issue_row_loads<CFG, T>(p, tile, ring_w, ring_d, bars, s + PF);
            } else {
                if (s > 1) bulk_wait_read<0>();
                if (s + PF < tile.n_steps) issue_row_loads<CFG, T>(p, tile, ring_w, ring_d, bars, s + PF);
                if (s > 0) issue_row_stores<CFG, T>(p, tile, ring_w, s - 1);
            }
        }
        __syncwarp();
        WDPM_TL(1);
#pragma unroll
        for (int b = 0; b < NBAR; b++) __syncthreads();
        WDPM_TL(8);
    }
    if (lead) {
        issue_row_stores<CFG, T>(p, tile, ring_w, tile.n_steps - 1);
        bulk_wait_read<0>();
        halo_handshake<CFG, T>(p, tile);
    }
}

// The STAGGERED schedule (k_fused_wa with kOptStagger, NT = 2): the row groups of triple slot 1 run half a step
// behind those of slot 0, the CTA meets every half step. Half step h: slot-0 groups do the first half of step h/2
// (h even) or its second half (h odd); slot-1 groups the second half of step (h-2)/2 (h even) or the first half of
// step (h-1)/2 (h odd). Rows finished by the last phase are written home half a step after they are done, slot 0
// and slot 1 in bulk groups of their own; loads stay once per step. The ring needs no extra rows: a load for step
// s+PF lands at most 31 rows ahead of the oldest row still being computed and 34 ahead of the oldest row whose
// write-back may be in flight (PF = 1; the ring has 36), and the group before that has been waited for.
template <typename CFG, typename T>
__device__ __forceinline__ void data_movement_warp_staggered(const FusedParams<T>& p, const MwTile<CFG>& tile, T* ring_w, T* ring_d, uint64_t* bars, bool lead) {
    static_assert(CFG::NT == 2, "the staggered schedule splits a step by triple slot");
    constexpr int PF = CFG::PF;
    const int n = tile.n_steps;
    if (lead)
        for (int s = 0; s < PF && s < n; s++) issue_row_loads<CFG, T>(p, tile, ring_w, ring_d, bars, s);
    for (int h = 0; h <= 2 * n; h++) {
        if (lead) {
            const int s = h >> 1;
            if ((h & 1) == 0) {
                if (s > 0) {
                    issue_row_stores<CFG, T>(p, tile, ring_w, s - 1, 0);
                    bulk_wait_read<1>();
                }
                if (s + PF < n) issue_row_loads<CFG, T>(p, tile, ring_w, ring_d, bars, s + PF);
            } else if (s > 0) {
                issue_row_stores<CFG, T>(p, tile, ring_w, s - 1, 1);
            }
        }
        __syncwarp();
        __syncthreads();
    }
    if (lead) {
        issue_row_stores<CFG, T>(p, tile, ring_w, n - 1, 1);
        bulk_wait_read<0>();
        halo_handshake<CFG, T>(p, tile);
    }
}

template <typename T, int MODULE, typename CFG, int NTHREADS, int MINB, int OPT = 0>
__global__ void __launch_bounds__(NTHREADS + fused_extra_threads(OPT), MINB)
k_fused(const FusedParams<T> p) {
    constexpr int NALL = NTHREADS + fused_extra_threads(OPT);  // threads of the CTA
    constexpr bool REALLOC = (OPT & kOptRegRealloc) != 0;
    // launch budget (what ptxas derives from the launch bounds) and what the compute warps can have once the
    // fourth warp group has shrunk to 24: 768 compute threads -> 72 and 80; 512 -> 96 and 112
    constexpr int kLaunchRegs = (65536 / NALL) & ~7;
    constexpr int kComputeRegs = ((kLaunchRegs * NALL - 128 * 24) / NTHREADS) & ~7;
    static_assert(!REALLOC || (MINB == 1 && NTHREADS % 128 == 0 && kComputeRegs > kLaunchRegs && kComputeRegs <= 232),
                  "register reallocation needs whole warp groups, one CTA per SM");
    constexpr int W = CFG::W, NT = CFG::NT, NPH = CFG::NPH, NRING = CFG::NRING, NSTAGE = CFG::NSTAGE, PF = CFG::PF;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    T* ring_w = reinterpret_cast<T*>(smem_raw);
    T* ring_d = ring_w + (size_t)NRING * W;
    uint64_t* bars = reinterpret_cast<uint64_t*>(ring_d + (size_t)NRING * W);

    const int tid = threadIdx.x;
    const int strip = blockIdx.x % p.n_strips;
    const int chunk = blockIdx.x / p.n_strips;
    MwTile<CFG> tile;
    tile.init(strip, chunk, p.chunk_triples, p.total_triples);

    // Drain: every CTA folds its share of the previous launch's contacts (the touched entries of its event buffer)
    if (MODULE == kDrain) fold_events(p.ds, prev_event_slot(p.launch_slot), (int)blockIdx.x * NALL + tid, (int)gridDim.x * NALL);

    // Drain: does any outlet lie in the rows and columns this CTA stages? (If not, no tile of this CTA
    // can see an outlet mark and the per-tile test is skipped.) Worked out per CTA when the set is installed.
    __shared__ int s_cta_has_outlets;
    if (tid == 0) {
        for (int i = 0; i < NSTAGE; i++) mbar_init(&bars[i], 1);
        fence_mbar_init();
        s_cta_has_outlets = MODULE == kDrain ? p.ds.cta_outlets[blockIdx.x] : 0;
    }
    __syncthreads();
    if (MODULE == kDrain && tid == 0) fold_finish(p.ds, prev_event_slot(p.launch_slot), (int)gridDim.x);
    const bool cta_has_outlets = MODULE == kDrain && s_cta_has_outlets != 0;

    // Barriers. The colour sub-steps of a step only order tiles of the SAME row triple (they exchange
    // window columns); different row groups touch disjoint rows within a step. When every row group
    // is a whole number of warps and each thread owns one tile (GROUPED), the two inner barriers are
    // named barriers over one row group only, so the groups drift apart inside a step and their
    // load / compute / store bursts interleave; the whole CTA (and the data-movement warp) meets
    // once per step. Otherwise all three are block barriers.
    constexpr bool GROUPED = (CFG::NCP % 32 == 0) && (NPH * NT * CFG::NCP == NTHREADS) && (NPH * NT <= 15);

    // Warp specialisation: the last warp only moves data (one elected lane issues the bulk copies),
    // the first NTHREADS threads only compute.
    if (tid >= NTHREADS) {
        if (REALLOC) {
            asm volatile("setmaxnreg.dec.sync.aligned.u32 24;");
            if (tid >= NTHREADS + 32) return;  // the rest of the fourth warp group only lent its registers
        }
        data_movement_warp<CFG, T, GROUPED ? 1 : 3>(p, tile, ring_w, ring_d, bars, tid == NTHREADS);
        return;
    }

    if (REALLOC) asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(kComputeRegs));

    // Static work assignment: in every sub-step thread `tid` relaxes tiles number tid,
    // tid+NTHREADS, ... of the NPH*NT*NC tiles (phase-major, then triple slot, then column), so its
    // phase / triple slot / column never change and are decoded once.
    constexpr int NC = CFG::NC, NCP = CFG::NCP;
    constexpr int NITEMS = NPH * NT * NCP;
    constexpr int IPT = (NITEMS + NTHREADS - 1) / NTHREADS;
    int it_col[IPT], it_q[IPT], it_ph[IPT], it_mrel[IPT];
    bool it_ok[IPT];
#pragma unroll
    for (int k = 0; k < IPT; k++) {
        const int item = tid + k * NTHREADS;
        const int c = item % NCP, pt = item / NCP, t = pt % NT, ph = pt / NT;
        it_ok[k] = item < NITEMS && c < NC;
        it_col[k] = 3 * c + 1;
        it_ph[k] = ph;
        it_q[k] = ph % 3;
        it_mrel[k] = t - ph * CFG::LAG;
    }

    constexpr bool ADD_FAST = sizeof(T) == 8 && (((OPT & kOptAddFast) && MODULE == kAdd) || ((OPT & kOptDrainFast) && MODULE == kDrain));  // relax_window5's FAST

    // Per tile: the three ring rows it spans this step, and a register window that slides one
    // column per colour sub-pass. wt = 3x3 water (rows x cols jb-1+cofs .. jb+1+cofs), dd = the
    // 3x5 elevations under all three positions. Between sub-passes only the column that leaves
    // the window is written to shared memory (the left-hand tile needs it next) and only the
    // column that enters is read (the right-hand tile has just published it); after the third
    // sub-pass the whole window is written back.
    bool run[IPT], slow[IPT];
    int row0[IPT];
    T* wrow[IPT][3];
    T wt[IPT][3][5], dd[IPT][3][5];  // wt: columns COFS..COFS+2 are live in sub-pass COFS
    constexpr int DOFF = NRING * W;  // ring_d = ring_w + DOFF

    auto prepare = [&](int s) {  // where step s's tiles live, and their elevation windows
#pragma unroll
        for (int k = 0; k < IPT; k++) {
            const int m = tile.m_lo + NT * s + it_mrel[k];
            run[k] = it_ok[k] && tile.runnable(m, it_q[k]);
            row0[k] = 3 * m + it_q[k];
            int s0 = run[k] ? tile.ring_slot(row0[k]) : 0;
            int s1 = s0 + 1; if (s1 == NRING) s1 = 0;
            int s2 = s1 + 1; if (s2 == NRING) s2 = 0;
            wrow[k][0] = ring_w + s0 * W; wrow[k][1] = ring_w + s1 * W; wrow[k][2] = ring_w + s2 * W;
            slow[k] = false;
            if (run[k]) {
                const int jl = it_col[k] - 1;
#pragma unroll
                for (int r = 0; r < 3; r++) {
#pragma unroll
                    for (int cc = 0; cc < 5; cc++) dd[k][r][cc] = wrow[k][r][DOFF + jl + cc];
                }
                if (cta_has_outlets) {  // tiles whose 3x5 elevation window holds an outlet mark take the shared-memory path
#pragma unroll
                    for (int r = 0; r < 3; r++) {
#pragma unroll
                        for (int cc = 0; cc < 5; cc++) slow[k] = slow[k] || is_outlet(dd[k][r][cc]);
                    }
                }
            }
        }
    };
    for (int s = 0; s < tile.n_steps; s++) {
        WDPM_TL(0);
        if (step_has_loads<CFG>(tile, s)) mbar_wait(&bars[s % NSTAGE], (uint32_t)((s / NSTAGE) & 1));
        WDPM_TL(1);
        prepare(s);
#pragma unroll
        for (int k = 0; k < IPT; k++) {
            if (run[k] && !slow[k]) {
                const int jl = it_col[k] - 1;
#pragma unroll
                for (int r = 0; r < 3; r++) {
#pragma unroll
                    for (int cc = 0; cc < 3; cc++) wt[k][r][cc] = wrow[k][r][jl + cc];
                }
            }
        }

        auto substep = [&](auto cofs_tag) {
            constexpr int COFS = decltype(cofs_tag)::value;
#pragma unroll
            for (int k = 0; k < IPT; k++) {
                const int j = it_col[k] + COFS;  // centre column inside the window
                if (MODULE == kDrain && run[k] && slow[k]) {
                    const int crow = row0[k] + 1, ccol = tile.x0 + j;
                    T* w0 = wrow[k][0]; T* w1 = wrow[k][1]; T* w2 = wrow[k][2];
                    const int mask = outlet_mask_3x3<T>(w0 + DOFF, w1 + DOFF, w2 + DOFF, j);
                    if (mask) {
                        drain_tile_near_outlets<T>(w0, w1, w2, w0 + DOFF, w1 + DOFF, w2 + DOFF, j, mask, p.ds, p.launch_slot,
                                                   (it_ph[k] / 3) * 9 + it_q[k] * 3 + COFS, crow, ccol,
                                                   tile.owns_row(crow) && tile.owns_col(ccol), false);
                    } else {
                        relax_tile<T, MODULE>(w0, w1, w2, w0 + DOFF, w1 + DOFF, w2 + DOFF, j);
                    }
                    continue;
                }
                if (COFS > 0 && run[k]) {  // slide: the published left column is dead, read the entering right column
#pragma unroll
                    for (int r = 0; r < 3; r++) wt[k][r][COFS + 2] = wrow[k][r][j + 1];
                }
                const bool active = run[k] && (wt[k][1][COFS + 1] > T(0)) && is_valid_elevation(dd[k][1][COFS + 1]);
                if (active) relax_window5<T, MODULE, COFS, ADD_FAST>(wt[k], dd[k]);
                if (run[k]) {  // an untouched tile writes back what it read: harmless, and cheaper than keeping track
                    if (COFS < 2) {
#pragma unroll
                        for (int r = 0; r < 3; r++) wrow[k][r][j - 1] = wt[k][r][COFS];
                    } else {
#pragma unroll
                        for (int r = 0; r < 3; r++) {
                            wrow[k][r][j - 1] = wt[k][r][COFS];
                            wrow[k][r][j] = wt[k][r][COFS + 1];
                            wrow[k][r][j + 1] = wt[k][r][COFS + 2];
                        }
                    }
                }
            }
        };
        auto group_barrier = [&]() {
            if (GROUPED) asm volatile("bar.sync %0, %1;" ::"r"(1 + tid / CFG::NCP), "n"(CFG::NCP) : "memory");
            else __syncthreads();
        };
        WDPM_TL(2);
        substep(std::integral_constant<int, 0>{});
        WDPM_TL(3);
        group_barrier();
        WDPM_TL(4);
        substep(std::integral_constant<int, 1>{});
        WDPM_TL(5);
        group_barrier();
        WDPM_TL(6);
        substep(std::integral_constant<int, 2>{});
        fence_proxy_async();  // make this step's smem writes visible to the bulk-store engine
        WDPM_TL(7);
        __syncthreads();
        WDPM_TL(8);

    }
}

// ---------------------------------------------------------------------------
// Warp-autonomous iteration kernel (mw_schedule.h, WaCfg). Same row march, ring, bulk copies and halo
// export as k_fused; the tiles of a row triple are relaxed by KW self-contained warps:
//   * a lane holds two adjacent tiles in a 3 x 8 register window (16-byte shared-memory loads: the window
//     starts at a multiple of 6 columns), relaxes both in every colour sub-pass (two independent chains,
//     interleaved) and slides the window by taking the entering column from the lane to its right with
//     warp shuffles - no shared-memory round trip and no barrier between the sub-passes;
//   * per step a warp reads its window once (water 3 x 6, elevations 3 x 8) and writes back 3 x 6;
//   * the warps of a row triple read columns their neighbours write back (the 6-column overlap), so a
//     warp announces "my window is in registers" on the row group's mbarrier and waits for the others'
//     announcements only just before its write-back - by then long satisfied;
//   * one CTA barrier per step, with the data-movement warp.
// OPT: kOptAddFast / kOptRegRealloc as in k_fused; kOptNoGuard (fp64 Add): no activity test at all
// (relax.cuh, wa_relax_pair) - the solver selects it only while the water grid is known to be +0 wherever
// the reference would skip the centre.
// ---------------------------------------------------------------------------

constexpr int kOptNoGuard = 8;
// OPT bit 4: STAGGERED schedule - the row groups of triple slot 1 run half a step behind those of slot 0 (see
// data_movement_warp_staggered), so that one half of the warps loads / stores its windows while the other half is in
// the middle of its chains: the shared-memory bursts that open and close a step no longer meet an idle issue port.
constexpr int kOptStagger = 16;

template <typename CFG, typename T>
constexpr size_t wa_smem_bytes() {
    return (size_t)2 * CFG::NRING * CFG::W * sizeof(T) + (CFG::NSTAGE + CFG::NPH * CFG::NT) * sizeof(uint64_t) + 16;
}

template <typename T> struct Vec2;
template <> struct Vec2<double> { using type = double2; };
template <> struct Vec2<float> { using type = float2; };

__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}

template <typename T>
__device__ __forceinline__ T shfl_from_right(T v) {
    return __shfl_down_sync(0xffffffffu, v, 1);
}

template <typename T, int MODULE, typename CFG, int OPT, int MINB = 1>
__global__ void __launch_bounds__(CFG::NWARPS * 32 + fused_extra_threads(OPT), MINB)
k_fused_wa(const FusedParams<T> p) {
    constexpr int NTHREADS = CFG::NWARPS * 32;
    constexpr int NALL = NTHREADS + fused_extra_threads(OPT);
    constexpr bool REALLOC = (OPT & kOptRegRealloc) != 0;
    constexpr int kLaunchRegs = (65536 / NALL) & ~7;
    constexpr int kComputeRegsRaw = ((kLaunchRegs * NALL - 128 * 24) / NTHREADS) & ~7;
    constexpr int kComputeRegs = kComputeRegsRaw > 232 ? 232 : kComputeRegsRaw;
    static_assert(!REALLOC || (MINB == 1 && NTHREADS % 128 == 0 && kComputeRegs > kLaunchRegs), "register reallocation needs whole warp groups, one CTA per SM");
    constexpr int W = CFG::W, NT = CFG::NT, NPH = CFG::NPH, NRING = CFG::NRING, NSTAGE = CFG::NSTAGE, KW = CFG::KW;
    // the cheaper forms of the step: Add - fp64 push_add_fast, fp32 push_add_nocap; Drain (fp64) - push_drain_fast
    constexpr bool FAST = ((OPT & kOptAddFast) && MODULE == kAdd) || ((OPT & kOptDrainFast) && MODULE == kDrain && sizeof(T) == 8);
    constexpr bool GUARD = !(FAST && MODULE == kAdd && (OPT & kOptNoGuard));
    constexpr bool STAGGER = (OPT & kOptStagger) != 0;
    static_assert(!STAGGER || CFG::NT == 2, "the staggered schedule splits a step by triple slot");
    static_assert(!(STAGGER && MODULE == kDrain), "Drain runs the plain schedule (its outlet path is not split in halves)");
    using V2 = typename Vec2<T>::type;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    T* ring_w = reinterpret_cast<T*>(smem_raw);
    T* ring_d = ring_w + (size_t)NRING * W;
    uint64_t* bars = reinterpret_cast<uint64_t*>(ring_d + (size_t)NRING * W);
    uint64_t* group_bars = bars + NSTAGE;  // one per row group: "every warp of the group holds its window in registers"

    const int tid = threadIdx.x;
    const int strip = blockIdx.x % p.n_strips;
    const int chunk = blockIdx.x / p.n_strips;
    MwTile<CFG> tile;
    tile.init(strip, chunk, p.chunk_triples, p.total_triples);

    // Drain: every CTA folds its share of the previous launch's contacts (the touched entries of its event buffer)
    if (MODULE == kDrain) fold_events(p.ds, prev_event_slot(p.launch_slot), (int)blockIdx.x * NALL + tid, (int)gridDim.x * NALL);

    // Drain: does any outlet lie in the rows and columns this CTA stages? (If not, no window of this CTA can hold an
    // outlet mark and the per-step test is skipped.) Worked out per CTA when the set is installed.
    __shared__ int s_cta_has_outlets;
    if (tid == 0) {
        for (int i = 0; i < NSTAGE; i++) mbar_init(&bars[i], 1);
        for (int i = 0; i < NPH * NT; i++) mbar_init(&group_bars[i], KW);
        fence_mbar_init();
        s_cta_has_outlets = MODULE == kDrain ? p.ds.cta_outlets[blockIdx.x] : 0;
    }
    __syncthreads();
    if (MODULE == kDrain && tid == 0) fold_finish(p.ds, prev_event_slot(p.launch_slot), (int)gridDim.x);
    const bool cta_has_outlets = MODULE == kDrain && s_cta_has_outlets != 0;

    if (tid >= NTHREADS) {
        if (REALLOC) {
            asm volatile("setmaxnreg.dec.sync.aligned.u32 24;");
            if (tid >= NTHREADS + 32) return;
        }
        if constexpr (STAGGER) data_movement_warp_staggered<CFG, T>(p, tile, ring_w, ring_d, bars, tid == NTHREADS);
        else data_movement_warp<CFG, T, 1>(p, tile, ring_w, ring_d, bars, tid == NTHREADS);
        return;
    }
    if (REALLOC) asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(kComputeRegs));

    // this warp: phase ph (= colour row offset, K = 1), triple slot t, column block kw of the row triple. With the
    // staggered schedule the slots alternate over the warps of a phase (and the other way round in the next phase),
    // so every scheduler hosts warps of both halves of the step.
    const int warp = tid >> 5, lane = tid & 31;
    const int wph = warp % (NT * KW), ph = warp / (NT * KW);
    const int t = STAGGER ? ((wph & 1) ^ (ph & 1)) : wph / KW;
    const int kw = STAGGER ? wph / NT : wph % KW;
    const int grp = ph * NT + t;
    const int cb = CFG::WSTRIDE * kw + CFG::CPL * lane;  // window column of the lane's column 0
    const bool stores = lane < 31;
    constexpr int DOFF = NRING * W;
    uint64_t* gbar = &group_bars[grp];

    T wt[3][8], dd[3][8];
    T* wrow[3] = {ring_w, ring_w, ring_w};
    bool run = false;
    bool near_outlets = false;  // Drain: some lane of this warp holds an outlet mark in its window this step
    int crow = 0;               // padded row of this step's centres

    // One colour sub-pass of this lane's two tiles. Drain warps with an outlet in reach take the outlet path: the
    // walk with the outlet rule, contacts recorded by the lane that will store the centre (lanes 0..30 of the CTA
    // that owns it - lane 31 and the halo columns only hold copies).
    auto subpass = [&](auto c_tag, auto part_tag) {
        constexpr int C = decltype(c_tag)::value;
        constexpr int PART = decltype(part_tag)::value;
        if (MODULE == kDrain && near_outlets) {
            if constexpr (MODULE == kDrain) {
                wa_relax_pair_outlets<T, C, FAST>(wt, dd, [&](int tl, int a, int b, T w_outlet, T w_centre) {
                    const int ccol = tile.x0 + cb + C + 3 * tl + 1;
                    if (stores && tile.owns_row(crow) && tile.owns_col(ccol))
                        record_contact<T>(p.ds, p.launch_slot, ph * 3 + C, crow + a, ccol + b, w_outlet, w_centre, false);
                });
            }
        } else {
            wa_relax_pair<T, MODULE, C, FAST, GUARD, PART>(wt, dd);
        }
    };
    using I0 = std::integral_constant<int, 0>;
    using I1 = std::integral_constant<int, 1>;
    using I2 = std::integral_constant<int, 2>;

    // first part of step s: window into registers, first colour sub-pass (and, staggered, half of the second)
    // Loop-carried addressing: this warp's triple advances by NT per step, its first ring slot by 3*NT (mod NRING);
    // `run` is one unsigned compare against the runnable range [m_lo, m_hi - (ph > 0)] (MwTile::runnable).
    const int m_first = tile.m_lo - ph * CFG::LAG + t;               // triple of step 0 (may lie before the staged range)
    const unsigned run_span = (unsigned)(tile.m_hi - (ph > 0 ? 1 : 0) - tile.m_lo);
    int slot0 = (((3 * (m_first - tile.m_lo) + ph) % NRING) + NRING) % NRING;  // ring slot of row 3*m + ph at step 0
    auto begin_step = [&](int s) {
        const int m = m_first + NT * s;
        run = (unsigned)(m - tile.m_lo) <= run_span;
        WDPM_TL(0);
        if (ph == 0 && run) mbar_wait(&bars[s % NSTAGE], (uint32_t)((s / NSTAGE) & 1));  // phase 0 runs exactly on the staged triples
        WDPM_TL(1);
        const int s0 = slot0;
        slot0 += 3 * NT; if (slot0 >= NRING) slot0 -= NRING;
        if (run) {
            int s1 = s0 + 1; if (s1 == NRING) s1 = 0;
            int s2 = s1 + 1; if (s2 == NRING) s2 = 0;
            wrow[0] = ring_w + s0 * W + cb; wrow[1] = ring_w + s1 * W + cb; wrow[2] = ring_w + s2 * W + cb;
#pragma unroll
            for (int r = 0; r < 3; r++) {
#pragma unroll
                for (int v = 0; v < 3; v++) {
                    const V2 x = *reinterpret_cast<const V2*>(wrow[r] + 2 * v);
                    wt[r][2 * v] = x.x; wt[r][2 * v + 1] = x.y;
                }
#pragma unroll
                for (int v = 0; v < 4; v++) {
                    const V2 x = *reinterpret_cast<const V2*>(wrow[r] + DOFF + 2 * v);
                    dd[r][2 * v] = x.x; dd[r][2 * v + 1] = x.y;
                }
            }
            if (MODULE == kDrain) {
                crow = 3 * m + ph + 1;
                bool mine = false;
                if (cta_has_outlets) {
#pragma unroll
                    for (int r = 0; r < 3; r++) {
#pragma unroll
                        for (int c = 0; c < 8; c++) mine = mine || is_outlet(dd[r][c]);
                    }
                }
                near_outlets = cta_has_outlets && __any_sync(0xffffffffu, mine);
            }
            subpass(I0{}, I0{});
            WDPM_TL(2);
        }
        // every lane's window is in registers (the relax above consumed it): tell the row group. A group that
        // does not run this step arrives too, which keeps the barrier's phase in step with s.
        __syncwarp();
        if (lane == 0) mbar_arrive(gbar);
        if (run) {
#pragma unroll
            for (int r = 0; r < 3; r++) wt[r][6] = shfl_from_right(wt[r][0]);
            if (STAGGER) subpass(I1{}, I1{});
        }
    };
    // the rest of step s, and the write-back
    auto end_step = [&](int s) {
        if (run) {
            if (STAGGER) subpass(I1{}, I2{});
            else subpass(I1{}, I0{});
            WDPM_TL(3);
#pragma unroll
            for (int r = 0; r < 3; r++) wt[r][7] = shfl_from_right(wt[r][1]);
            subpass(I2{}, I0{});
            WDPM_TL(4);
            // the neighbouring warps of this row triple read columns I am about to overwrite: they must hold them by now
            if (KW > 1) mbar_wait(gbar, (uint32_t)(s & 1));
            WDPM_TL(5);
            if (stores) {
#pragma unroll
                for (int r = 0; r < 3; r++) {
#pragma unroll
                    for (int v = 1; v < 4; v++) {
                        V2 x; x.x = wt[r][2 * v]; x.y = wt[r][2 * v + 1];
                        *reinterpret_cast<V2*>(wrow[r] + 2 * v) = x;
                    }
                }
            }
        }
    };

    if (!STAGGER) {
        for (int s = 0; s < tile.n_steps; s++) {
            begin_step(s);
            end_step(s);
            if (ph == NPH - 1) fence_proxy_async();  // the last phase's rows go home by bulk store: make them visible to the async proxy
            WDPM_TL(7);
            __syncthreads();
            WDPM_TL(8);
        }
    } else {
        // half step h: slot-0 groups begin step h/2 (h even) or end it (h odd); slot-1 groups half a step later
        for (int h = 0; h <= 2 * tile.n_steps; h++) {
            const int s = (h - t) >> 1;  // the step this warp is in (h - t >= 0 wherever it is used)
            if (((h - t) & 1) == 0) {
                if (h >= t && s < tile.n_steps) begin_step(s);
            } else {
                if (h > t && s < tile.n_steps) end_step(s);
            }
            if (ph == NPH - 1) fence_proxy_async();
            __syncthreads();
        }
    }
}

// ---------------------------------------------------------------------------
// Resident kernel: grids of up to about a million cells (the reference's own DEMs: basin5 is
// 482 x 471). Such a grid cannot amortise a launch per iteration, nor fill 148 SMs with marching
// windows; what bounds an iteration is the LATENCY of nine dependent colour sub-passes. So the whole
// block of n iterations is ONE cooperative launch: every CTA owns a TR x TC tile of the padded grid,
// keeps its elevations in shared memory for the whole launch, and per iteration reads its tile plus
// halo (3 rows above, 6 below, 9 columns left, 18 right: what a whole iteration consumes, see
// mw_schedule.h) from the current water buffer - L2 resident at these sizes -, runs the nine
// sub-passes on it with block barriers, writes its owned cells to the other buffer and meets the
// other CTAs at a grid barrier. Tiles partly outside the shared-memory tile are skipped; the cells
// they would have produced lie in the halo and are never written back.
// ---------------------------------------------------------------------------

constexpr int kResHaloTop = 3, kResHaloBottom = 6, kResHaloLeft = 9, kResHaloRight = 18;

template <typename T>
struct ResidentParams {
    T* w[2];        // ping / pong; w[cur] holds the state on entry
    const T* dem;
    Geom g;
    int cur;
    int TR, TC;     // owned rows / cols per CTA (multiples of 3)
    int n_tx;       // CTAs per grid row
    int n_iters;
    int launch_slot;    // drain event buffer of the first iteration
    int serial_wipe;    // Drain, serial schedule: empty the outlet's 3x3 after every iteration (k_outlet_wipe)
    DrainState<T> ds;
};

template <typename T, int MODULE, int NTHREADS>
__global__ void __launch_bounds__(NTHREADS, 1)
k_resident(const ResidentParams<T> p) {
    namespace cg = cooperative_groups;
    cg::grid_group grid = cg::this_grid();
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const int SR = p.TR + kResHaloTop + kResHaloBottom, SC = p.TC + kResHaloLeft + kResHaloRight;
    T* sw = reinterpret_cast<T*>(smem_raw);  // [SR][SC] water
    T* sd = sw + SR * SC;                    // [SR][SC] masked elevations
    const int tid = threadIdx.x;
    const int ty = blockIdx.x / p.n_tx, tx = blockIdx.x % p.n_tx;
    const int r_own = ty * p.TR, c_own = tx * p.TC;                  // padded coordinates of the owned tile
    const int r0 = r_own - kResHaloTop, c0 = c_own - kResHaloLeft;   // ... and of the shared-memory tile
    const size_t pitch = (size_t)p.g.pitch;
    const size_t base = (size_t)(r0 + kPadTop) * pitch + (size_t)(c0 + kPadLeft);

    for (int k = tid; k < SR * SC; k += NTHREADS) {
        const int i = k / SC, j = k - i * SC;
        sd[k] = p.dem[base + (size_t)i * pitch + j];
    }
    // Serial-schedule Drain: the outlet's 3x3 is emptied after every iteration (k_outlet_wipe). Iteration k's
    // emptying happens while iteration k+1 stages its window: every CTA zeroes the cells its copy holds, and the
    // CTA that owns the outlet - its window holds the whole 3x3 (halo >= 3 on every side) - first takes the sum.
    // That CTA, not block 0, also folds the contact events: in iteration k+1 it folds iteration k's contacts
    // (recorded by any CTA before the grid barrier) and then adds the sum, so the total grows as contacts of k,
    // emptying of k, contacts of k+1, and nobody else touches it. The last iteration's emptying works on global
    // memory after the last grid barrier, where no CTA reads the water any more.
    const bool wipe = MODULE == kDrain && p.serial_wipe;
    const int orow = wipe ? p.ds.outlet_rc[0] : 0, ocol = wipe ? p.ds.outlet_rc[1] : 0;
    const bool wipe_owner = wipe && orow >= r_own && orow < r_own + p.TR && ocol >= c_own && ocol < c_own + p.TC;
    // Otherwise every CTA folds its share of the previous iteration's contacts.
    const bool fold_all = MODULE == kDrain && !wipe;
    const int fold_first = (int)blockIdx.x * NTHREADS + tid, fold_stride = (int)gridDim.x * NTHREADS;
    int cur = p.cur, evbuf = p.launch_slot;
    for (int it = 0; it < p.n_iters; it++) {
        const T* __restrict__ win = p.w[cur];
        T* __restrict__ wout = p.w[cur ^ 1];
        if (fold_all) fold_events(p.ds, prev_event_slot(evbuf), fold_first, fold_stride);
        for (int k = tid; k < SR * SC; k += NTHREADS) {
            const int i = k / SC, j = k - i * SC;
            sw[k] = win[base + (size_t)i * pitch + j];
        }
        __syncthreads();
        if (fold_all && tid == 0) fold_finish(p.ds, prev_event_slot(evbuf), (int)gridDim.x);
        if (wipe) {
            if (wipe_owner && tid == 0) {
                fold_events(p.ds, prev_event_slot(evbuf), 0, 1);
                fold_finish(p.ds, prev_event_slot(evbuf), 1);
                if (it > 0) {  // the launch before ended with its own emptying
                    const int a = (orow - r0) * SC + (ocol - c0);
                    p.ds.totaldrain[0] = p.ds.totaldrain[0] + outlet_wipe_sum(sw + a, sd + a, (size_t)SC);
                }
            }
            __syncthreads();
            if (it > 0 && tid < 9) {
                const int i = orow - 1 + tid / 3 - r0, j = ocol - 1 + tid % 3 - c0;
                if (i >= 0 && i < SR && j >= 0 && j < SC) sw[i * SC + j] = T(0);
            }
            __syncthreads();
        }
#pragma unroll 1
        for (int sub = 0; sub < 9; sub++) {
            const int oi = sub / 3, oj = sub - 3 * oi;       // tile-start offsets = (reference oi, oj) - 1
            const int na = (SR - 3 - oi) / 3 + 1, nb = (SC - 3 - oj) / 3 + 1;
            for (int k = tid; k < na * nb; k += NTHREADS) {
                const int a = k / nb, b = k - a * nb;
                const int i = oi + 3 * a, j = oj + 3 * b + 1;  // tile's first row, centre column
                T* w0 = sw + i * SC; T* w1 = w0 + SC; T* w2 = w1 + SC;
                const T* d0 = sd + i * SC; const T* d1 = d0 + SC; const T* d2 = d1 + SC;
                if (MODULE == kDrain) {
                    const int mask = outlet_mask_3x3<T>(d0, d1, d2, j);
                    if (mask) {
                        const int crow = r0 + i + 1, ccol = c0 + j;
                        // only the CTA that owns the centre reports the contact (halo copies recompute it)
                        drain_tile_near_outlets<T>(w0, w1, w2, d0, d1, d2, j, mask, p.ds, evbuf, sub, crow, ccol,
                                                   crow >= r_own && crow < r_own + p.TR && ccol >= c_own && ccol < c_own + p.TC, false);
                        continue;
                    }
                }
                relax_tile<T, MODULE, true>(w0, w1, w2, d0, d1, d2, j);
            }
            __syncthreads();
        }
        for (int k = tid; k < p.TR * p.TC; k += NTHREADS) {
            const int i = k / p.TC, j = k - i * p.TC;
            wout[(size_t)(r_own + i + kPadTop) * pitch + (size_t)(c_own + j + kPadLeft)] =
                sw[(i + kResHaloTop) * SC + j + kResHaloLeft];
        }
        grid.sync();
        cur ^= 1;
        evbuf = next_event_slot(evbuf);
    }
    if (fold_all) {
        fold_events(p.ds, prev_event_slot(evbuf), fold_first, fold_stride);
        __syncthreads();
        if (tid == 0) fold_finish(p.ds, prev_event_slot(evbuf), (int)gridDim.x);
    }
    if (wipe_owner && tid == 0 && p.n_iters > 0) {
        fold_events(p.ds, prev_event_slot(evbuf), 0, 1);
        fold_finish(p.ds, prev_event_slot(evbuf), 1);
        T* w = p.w[cur];
        const size_t c = dev_index(p.g, orow, ocol);
        p.ds.totaldrain[0] = p.ds.totaldrain[0] + outlet_wipe_sum(w + c, p.dem + c, pitch);
        for (int a = -1; a <= 1; a++)
            for (int b = -1; b <= 1; b++) w[c + a * (ptrdiff_t)pitch + b] = T(0);
    }
}

}  // namespace wdpm
