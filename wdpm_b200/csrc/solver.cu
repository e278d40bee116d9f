// C ABI of the B200-native WDPM redistribution solver: device state, launch
// plumbing and the per-block driver. Declarations and the mapping to the
// reference's call sites are in include/wdpm_b200.h.
#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <unistd.h>
#include <vector>

#include "../../include/wdpm_b200.h"
#include "kernels.cuh"

using namespace wdpm;

namespace {

constexpr int kDefaultVariantF64 = 17;  // warp-autonomous: 380-column window, two row triples per phase, 12 compute warps x 2 tiles per lane at 160 registers, Add fast step
constexpr int kDefaultVariantF32 = 16;  // warp-autonomous: 752-column window, 24 compute warps x 2 tiles per lane
// round 1's production tilings of k_fused, still selectable by number (tests, comparisons): fp64 13 (Add / Subtract), 15 / 14 (Drain
// with / without the folded-gate step), fp32 12
// Grids of a few hundred thousand cells (the reference's basin5 is 482 x 471) cannot fill 148 SMs
// with long chunks: narrow windows, two CTAs per SM and chunks of a few row triples spread the
// rows over the whole chip in one wave (measured on basin5: 18 us per iteration against 37 us for
// nine colour launches).
constexpr int kSmallGridVariantF64 = 5;
constexpr int kSmallGridVariantF32 = 7;
constexpr long long kSmallGridCells = 1ll << 22;

thread_local std::string g_err;

int fail(int code, const std::string& msg) {
    g_err = msg;
    return code;
}

#define CUDA_TRY(expr)                                                                              \
    do {                                                                                            \
        cudaError_t e_ = (expr);                                                                    \
        if (e_ != cudaSuccess)                                                                      \
            return fail(e_ == cudaErrorMemoryAllocation ? WDPM_E_NOMEM : WDPM_E_CUDA,               \
                        std::string(#expr) + ": " + cudaGetErrorString(e_));                        \
    } while (0)

// ---------------------------------------------------------------------------
// Fused-kernel variants. One entry = one instantiation of k_fused per module.
// ---------------------------------------------------------------------------

template <typename T>
using FusedLaunchFn = cudaError_t (*)(const FusedParams<T>&, int grid, cudaStream_t);

template <typename T>
struct FusedVariant {
    int W, TWV, HL, K, NT, PF, nthreads, minb;
    bool wa = false;  // k_fused_wa
    size_t smem;
    FusedLaunchFn<T> launch[3];        // per module; nullptr = this variant does not implement the module
    FusedLaunchFn<T> launch_clean[3];  // used instead while wdpm_solver::water_clean holds (nullptr = none)
    FusedLaunchFn<T> launch_ref_add;   // fp64 variants with the sign-gated Add step: Add in the reference form (nullptr = launch[kAdd] is)
    cudaError_t (*prepare)();
};

template <typename T, int MODULE, typename CFG, int NTHREADS, int MINB, int OPT>
cudaError_t launch_fused(const FusedParams<T>& p, int grid, cudaStream_t st) {
    k_fused<T, MODULE, CFG, NTHREADS, MINB, OPT><<<grid, NTHREADS + fused_extra_threads(OPT), fused_smem_bytes<CFG, T>(), st>>>(p);  // + the data-movement warp
    return cudaGetLastError();
}

template <typename T, typename CFG, int NTHREADS, int MINB, int OPT>
cudaError_t prepare_fused() {
    const int smem = (int)fused_smem_bytes<CFG, T>();
    cudaError_t e;
    e = cudaFuncSetAttribute(k_fused<T, kAdd, CFG, NTHREADS, MINB, OPT>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    if (e != cudaSuccess) return e;
    e = cudaFuncSetAttribute(k_fused<T, kSubtract, CFG, NTHREADS, MINB, OPT>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    if (e != cudaSuccess) return e;
    if constexpr (sizeof(T) == 8 && (OPT & kOptAddFast)) {
        e = cudaFuncSetAttribute(k_fused<T, kAdd, CFG, NTHREADS, MINB, OPT & ~kOptAddFast>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
        if (e != cudaSuccess) return e;
    }
    return cudaFuncSetAttribute(k_fused<T, kDrain, CFG, NTHREADS, MINB, OPT>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
}

// OPT: kernels.cuh (kOptAddFast only affects the Add instantiation)
template <typename T, typename CFG, int NTHREADS, int MINB, int OPT = 0>
FusedVariant<T> make_variant() {
    FusedVariant<T> v;
    v.W = CFG::W; v.TWV = CFG::TWV; v.HL = CFG::HL; v.K = CFG::K; v.NT = CFG::NT; v.PF = CFG::PF;
    v.nthreads = NTHREADS; v.minb = MINB;
    v.smem = fused_smem_bytes<CFG, T>();
    v.launch[kAdd] = launch_fused<T, kAdd, CFG, NTHREADS, MINB, OPT>;
    v.launch[kSubtract] = launch_fused<T, kSubtract, CFG, NTHREADS, MINB, OPT>;
    v.launch[kDrain] = launch_fused<T, kDrain, CFG, NTHREADS, MINB, OPT>;
    v.launch_clean[kAdd] = v.launch_clean[kSubtract] = v.launch_clean[kDrain] = nullptr;
    v.launch_ref_add = nullptr;
    if constexpr (sizeof(T) == 8 && (OPT & kOptAddFast)) v.launch_ref_add = launch_fused<T, kAdd, CFG, NTHREADS, MINB, OPT & ~kOptAddFast>;
    v.prepare = prepare_fused<T, CFG, NTHREADS, MINB, OPT>;
    return v;
}

// Warp-autonomous variants (kernels.cuh, k_fused_wa): Add and Subtract only.
template <typename T, int MODULE, typename CFG, int OPT, int MINB>
cudaError_t launch_wa(const FusedParams<T>& p, int grid, cudaStream_t st) {
    k_fused_wa<T, MODULE, CFG, OPT, MINB><<<grid, CFG::NWARPS * 32 + fused_extra_threads(OPT), wa_smem_bytes<CFG, T>(), st>>>(p);
    return cudaGetLastError();
}

template <typename T, typename CFG, int OPT, int MINB>
cudaError_t prepare_wa() {
    const int smem = (int)wa_smem_bytes<CFG, T>();
    cudaError_t e;
    e = cudaFuncSetAttribute(k_fused_wa<T, kAdd, CFG, OPT, MINB>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    if (e != cudaSuccess) return e;
    e = cudaFuncSetAttribute(k_fused_wa<T, kAdd, CFG, OPT | kOptNoGuard, MINB>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    if (e != cudaSuccess) return e;
    if constexpr (sizeof(T) == 8 && (OPT & kOptAddFast)) {
        e = cudaFuncSetAttribute(k_fused_wa<T, kAdd, CFG, OPT & ~kOptAddFast, MINB>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
        if (e != cudaSuccess) return e;
    }
    if constexpr (!(OPT & kOptStagger)) {
        e = cudaFuncSetAttribute(k_fused_wa<T, kDrain, CFG, OPT & ~kOptDrainFast, MINB>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
        if (e != cudaSuccess) return e;
        e = cudaFuncSetAttribute(k_fused_wa<T, kDrain, CFG, OPT | kOptDrainFast, MINB>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
        if (e != cudaSuccess) return e;
    }
    return cudaFuncSetAttribute(k_fused_wa<T, kSubtract, CFG, OPT, MINB>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
}

template <typename T, typename CFG, int OPT = 0, int MINB = 1>
FusedVariant<T> make_wa_variant() {
    FusedVariant<T> v;
    v.W = CFG::W; v.TWV = CFG::TWV; v.HL = CFG::HL; v.K = CFG::K; v.NT = CFG::NT; v.PF = CFG::PF;
    v.nthreads = CFG::NWARPS * 32; v.minb = MINB; v.wa = true;
    v.smem = wa_smem_bytes<CFG, T>();
    v.launch[kAdd] = launch_wa<T, kAdd, CFG, OPT, MINB>;
    v.launch[kSubtract] = launch_wa<T, kSubtract, CFG, OPT, MINB>;
    v.launch_clean[kAdd] = (OPT & kOptAddFast) ? launch_wa<T, kAdd, CFG, OPT | kOptNoGuard, MINB> : nullptr;
    v.launch_clean[kSubtract] = nullptr;
    v.launch_ref_add = nullptr;
    if constexpr (sizeof(T) == 8 && (OPT & kOptAddFast)) v.launch_ref_add = launch_wa<T, kAdd, CFG, OPT & ~kOptAddFast, MINB>;
    // Drain: the reference form of the step, and - fp64, while the water is known to hold no -0.0 (water_clean) - the
    // folded-gate form (relax.cuh, push_drain_fast). Not with the staggered schedule.
    if constexpr (OPT & kOptStagger) {
        v.launch[kDrain] = v.launch_clean[kDrain] = nullptr;
    } else {
        v.launch[kDrain] = launch_wa<T, kDrain, CFG, OPT & ~kOptDrainFast, MINB>;
        v.launch_clean[kDrain] = sizeof(T) == 8 ? launch_wa<T, kDrain, CFG, OPT | kOptDrainFast, MINB> : nullptr;
    }
    v.prepare = prepare_wa<T, CFG, OPT, MINB>;
    return v;
}

// Variant ids are 1-based in the ABI. 1 is the production tiling for each
// precision; the small windows exist so tests can force many strips / chunks /
// iterations-per-launch on small grids.
template <typename T>
const std::vector<FusedVariant<T>>& fused_variants();

template <>
const std::vector<FusedVariant<double>>& fused_variants<double>() {
    static const std::vector<FusedVariant<double>> v = {
        make_variant<double, MwCfg<512, 1, 1, 2>, 512, 1>(),   // 1: 192 KB ring, one CTA per SM, one tile per thread
        make_variant<double, MwCfg<64, 1, 1, 1>, 128, 1>(),    // 2: test
        make_variant<double, MwCfg<128, 1, 2, 2>, 128, 1>(),   // 3: test, two iterations per launch, two tiles per thread
        make_variant<double, MwCfg<384, 2, 1, 1>, 512, 1>(),   // 4: two triples per phase, two tiles per thread
        make_variant<double, MwCfg<256, 1, 1, 2>, 256, 2>(),   // 5: two CTAs per SM
        make_variant<double, MwCfg<256, 1, 2, 2>, 512, 1>(),   // 6: two iterations per launch
        make_variant<double, MwCfg<512, 1, 1, 2>, 256, 1>(),   // 7: as 1, two tiles per thread
        make_variant<double, MwCfg<384, 2, 1, 1>, 384, 1>(),   // 8: two triples per phase, two tiles per thread (exact fit)
        make_variant<double, MwCfg<384, 2, 1, 1>, 256, 1>(),   // 9: two triples per phase, three tiles per thread
        make_variant<double, MwCfg<384, 2, 1, 1>, 768, 1>(),   // 10: two triples per phase, 24 warps, one tile per thread
        make_variant<double, MwCfg<384, 2, 1, 1>, 768, 1, kOptAddFast>(),  // 11: as 10, Add with the sign gate and cap-free chains
        make_variant<double, MwCfg<64, 1, 1, 1>, 128, 1, kOptAddFast>(),   // 12: test window with the Add fast path
        make_variant<double, MwCfg<384, 2, 1, 1>, 768, 1, kOptAddFast | kOptRegRealloc>(),  // 13: as 11, compute warps at 80 registers
        make_variant<double, MwCfg<512, 1, 1, 2>, 512, 1, kOptRegRealloc>(),                // 14: as 1, compute warps at 112 registers
        make_variant<double, MwCfg<512, 1, 1, 2>, 512, 1, kOptRegRealloc | kOptDrainFast>(), // 15: as 14, Drain with the gate folded into the factor
        make_variant<double, MwCfg<64, 1, 1, 1>, 128, 1, kOptDrainFast>(),                  // 16: test window for 15
        make_wa_variant<double, WaCfg<2, 2, 1>, kOptAddFast | kOptRegRealloc>(),            // 17: warp-autonomous, 12 warps x 2 tiles per lane, 380-column window
        make_wa_variant<double, WaCfg<1, 1, 1>, kOptAddFast>(),                             // 18: test window (196 columns, 3 warps) for 17
        make_wa_variant<double, WaCfg<2, 2, 1>, kOptAddFast>(),                             // 19: as 17 without register reallocation
        make_wa_variant<double, WaCfg<2, 1, 1>, kOptAddFast>(),                             // 20: one triple per phase (6 warps; small grids)
        make_wa_variant<double, WaCfg<3, 1, 1>, kOptAddFast>(),                             // 21: 566-column window, one triple per phase (9 warps)
        make_wa_variant<double, WaCfg<2, 2, 1>, kOptAddFast | kOptRegRealloc | kOptStagger>(),  // 22: as 17, staggered: triple slot 1 half a step behind slot 0
        make_wa_variant<double, WaCfg<1, 2, 1>, kOptAddFast | kOptStagger>(),               // 23: test window for 22
        make_wa_variant<double, WaCfg<2, 2, 2, 1>, kOptAddFast | kOptRegRealloc>(),         // 24: as 17, bulk loads two steps ahead on the same ring (strict order)
        make_wa_variant<double, WaCfg<1, 1, 2, 1>, kOptAddFast>(),                          // 25: test window for 24
    };
    return v;
}
template <>
const std::vector<FusedVariant<float>>& fused_variants<float>() {
    static const std::vector<FusedVariant<float>> v = {
        make_variant<float, MwCfg<512, 1, 1, 2>, 256, 2>(),    // 1: 96 KB ring, two CTAs per SM, two tiles per thread
        make_variant<float, MwCfg<64, 1, 1, 1>, 128, 1>(),     // 2: test
        make_variant<float, MwCfg<128, 1, 2, 2>, 128, 1>(),    // 3: test, two iterations per launch
        make_variant<float, MwCfg<384, 2, 1, 2>, 512, 1>(),    // 4
        make_variant<float, MwCfg<1024, 1, 1, 2>, 512, 1>(),   // 5: wide window, two tiles per thread
        make_variant<float, MwCfg<512, 1, 2, 2>, 512, 1>(),    // 6: two iterations per launch
        make_variant<float, MwCfg<512, 1, 1, 2>, 512, 2>(),    // 7: as 1, one tile per thread
        make_variant<float, MwCfg<640, 2, 1, 1>, 640, 1>(),    // 8: two triples per phase, two tiles per thread
        make_variant<float, MwCfg<768, 2, 1, 1>, 512, 1>(),    // 9: two triples per phase, three tiles per thread
        make_variant<float, MwCfg<384, 2, 1, 1>, 768, 2>(),    // 10: two CTAs of 24 warps per SM
        make_variant<float, MwCfg<580, 1, 1, 2>, 576, 2>(),    // 11: 192 tiles per row group (whole warps), two CTAs per SM
        make_variant<float, MwCfg<484, 1, 1, 2>, 480, 2>(),    // 12: 160 tiles per row group, two CTAs per SM
        make_variant<float, MwCfg<772, 2, 1, 1>, 768, 1>(),    // 13: 256 tiles per row group... one CTA per SM
        make_wa_variant<float, WaCfg<2, 2, 1>, kOptRegRealloc>(),  // 14: warp-autonomous, 12 warps x 2 tiles per lane
        make_wa_variant<float, WaCfg<1, 1, 1>, kOptAddFast>(),     // 15: test window for 16
        make_wa_variant<float, WaCfg<4, 2, 1>, kOptAddFast | kOptRegRealloc>(),  // 16: 752-column window, 24 warps, cap-free Add step
        make_wa_variant<float, WaCfg<2, 2, 1>, kOptAddFast, 2>(),  // 17: as 14, two CTAs per SM
        make_wa_variant<float, WaCfg<3, 2, 1>, kOptAddFast>(),     // 18: 566-column window, 18 warps
        make_wa_variant<float, WaCfg<4, 2, 1>, kOptRegRealloc>(),  // 19: as 16 with the reference form of the step (comparison)
        make_wa_variant<float, WaCfg<4, 2, 1>, kOptAddFast | kOptRegRealloc | kOptStagger>(),  // 20: as 16, staggered
        make_wa_variant<float, WaCfg<1, 2, 1>, kOptAddFast | kOptStagger>(),               // 21: test window for 20
        make_wa_variant<float, WaCfg<4, 2, 2, 1>, kOptAddFast | kOptRegRealloc>(),         // 22: as 16, bulk loads two steps ahead on the same ring
        make_wa_variant<float, WaCfg<1, 1, 2, 1>, kOptAddFast>(),                          // 23: test window for 22
    };
    return v;
}

}  // namespace

// ---------------------------------------------------------------------------

struct wdpm_solver {
    wdpm_config cfg{};
    int dtype = WDPM_F64, module = WDPM_ADD;
    int schedule = WDPM_SCHEDULE_OPENCL;
    // the module whose relax arithmetic the kernels run: the serial schedule's Subtract relaxes with the Add step
    // (runoffs, src/WDPMCL.c:1934-1964, is runoffadd bit for bit on every input the solver takes: relax.cuh,
    // rewrite (1), and the host macro's tie rule differs from mini's only on signed zeros that cannot occur there)
    int relax = WDPM_ADD;
    size_t esize = 8;
    Geom g{};
    int kernel = WDPM_KERNEL_COLOUR;
    int variant = 0;  // 0-based index into fused_variants
    int n_strips = 0, total_triples = 0, chunk_triples = 0, n_chunks = 0;
    int sm_count = 0;
    int device = 0;
    // resident kernel tiling (kernels.cuh, k_resident); res_ok = the grid fits one co-resident wave
    bool res_ok = false;
    bool resident_by_auto = false;  // AUTO picked the resident kernel: a refused cooperative launch falls back to the fused one
    int res_TR = 0, res_TC = 0, res_ntx = 0, res_nty = 0;
    size_t res_smem = 0;

    void* dem = nullptr;
    void* w[2] = {nullptr, nullptr};
    void* oldw = nullptr;
    int cur = 0;
    bool have_dem = false;
    // water_clean: the current water grid is +0 (not negative, not -0.0, not water on an invalid cell) wherever
    // the reference would skip the centre, so the unguarded Add step may run (relax.cuh, wa_relax_pair).
    // True after a block prologue with a zero threshold > 0 (WDPMCL.c:1055-1065 wipes negatives and -0.0)
    // provided the last upload put no water on invalid cells (invalid_dry); the kernels preserve both.
    bool water_clean = false, invalid_dry = false;
    // negzero_free: no valid cell holds -0.0. The fp64 sign-gated Add step (relax.cuh, push_add_fast) would turn a
    // -0.0 neighbour at h == +0 into +0.0; the Add module never sees one (apply_add rewrites every valid cell), but
    // the serial schedule's Subtract can (water uploaded without apply_subtract, zero threshold 0). While this is
    // false such a solver runs a reference form of the Add step. True after apply_subtract and after a block
    // prologue with a zero threshold > 0; no relax step creates a -0.0 (x - x = +0, +0 + -0 = +0).
    bool negzero_free = false;
    int* d_dirty = nullptr;   // device flag of k_check_invalid_water

    // Drain outlets (kernels.cuh "Drain bookkeeping"). The per-outlet arrays hold outlet_cap entries: the installed
    // set's size (1 before any set, so that the single total exists).
    int outlet_cap = 0;
    void* totaldrain = nullptr;    // T[outlet_cap] per-outlet accumulators, sorted order
    void* ev_area = nullptr;       // the outlet event area (kernels.cuh, EventArea) for outlet_cap entries
    int ev_slots = 10;             // its sub-pass slots per entry: 9 * iterations per launch + 1
    void* events = nullptr;        // row stripes (Drain): the border event area, after the arrival flags; nullptr otherwise
    void* saved_elev = nullptr;    // T[outlet_cap] elevations under the outlet marks
    int* d_outlet_rc = nullptr;    // int[outlet_cap][2] padded (row, col), rows local to this solver, sorted by (row, col)
    int* d_outlet_pos = nullptr;   // int[outlet_cap]: sorted position of the caller's outlet k
    unsigned char* d_cta_outlets = nullptr;  // fused kernels: per CTA, does an outlet lie in what it stages
    double* d_total = nullptr;     // the outlet-order sum of the totals (k_sum_totals)
    int* d_bad = nullptr;          // outlets found on cells with dem <= nodata (k_mark_outlets)
    std::vector<int> outlet_rc;    // host copy of d_outlet_rc
    std::vector<int> outlet_pos;   // host copy of d_outlet_pos
    int n_outlets = 0;
    bool marks_applied = false;
    bool have_outlet = false;
    int launch_slot = 0;       // drain event buffer of the next launch (kernels.cuh, kEventSlots)
    bool wipe_due = false;     // serial-schedule Drain: the last launched iteration's outlet emptying is still to come

    BlockPartial* partials = nullptr;
    BlockPartial* d_result = nullptr;
    BlockPartial* h_result = nullptr;  // pinned
    OutletCand* outlet_partials = nullptr;
    OutletCand* d_outlet = nullptr;
    int reduce_blocks = 0;

    // row-stripe state (include/wdpm_b200.h "row-stripe partition")
    bool stripe = false;
    int G = 0, P = 0;          // first owned padded row of the whole DEM, owned padded rows
    HaloFlags* flags = nullptr;
    struct Peer {
        bool present = false;
        void* w[2] = {nullptr, nullptr};
        HaloFlags* flags = nullptr;
        void* events = nullptr;  // the neighbour's drain event buffers (same allocation as its flags)
        int P = 0;
        bool ipc = false;
    } above, below;
    int epoch = 0;             // halo pushes done since the last upload
    unsigned long long halo_timeout_ns = 120ull * 1000000000ull;  // WDPM_B200_HALO_TIMEOUT_MS; k_halo_wait gives up after this
    bool halo_failed = false;  // a wait gave up: results since then are void until the next upload
    int* h_halo_error = nullptr;  // pinned copy of HaloFlags::error

    cudaStream_t own_stream = nullptr;
    cudaStream_t stream = nullptr;
    cudaEvent_t ev[4] = {nullptr, nullptr, nullptr, nullptr};
    long long launches = 0;
    long long device_bytes = 0;
    // state of an open block (wdpm_block_begin .. wdpm_block_end)
    bool in_block = false;
    long long blk_launches0 = 0;
    int blk_iters = 0;

    // Checkpoint capture (wdpm_checkpoint_arm / wdpm_checkpoint_wait): an armed block prologue gathers the totals,
    // and a side stream copies the snapshot it wrote (oldw) and those totals into pinned staging while the block
    // runs. ck_done marks the copies' completion; every later writer of oldw or d_ck_totals waits on it on the
    // device (ck_fence).
    cudaStream_t ck_stream = nullptr;
    cudaEvent_t ck_ready = nullptr, ck_done = nullptr;
    bool ck_armed = false, ck_captured = false;
    void* ck_water = nullptr;       // pinned: the owned interior rows, unpadded, solver precision
    double* ck_totals = nullptr;    // pinned: ck_cap totals
    double* d_ck_totals = nullptr;  // device: ck_cap totals, the gather's output
    int ck_cap = 0, ck_n = 0;
};

namespace {

int border_entries(const wdpm_solver* s) { return 2 * (s->g.C + 2); }

template <typename T>
DrainState<T> drain_state(wdpm_solver* s) {
    DrainState<T> ds;
    ds.totaldrain = static_cast<T*>(s->totaldrain);
    ds.outlet_rc = s->d_outlet_rc;
    ds.n_outlets = s->n_outlets;
    ds.ev = event_area<T>(s->ev_area, s->outlet_cap, s->ev_slots);
    // row stripes: contacts with an outlet in the first or last owned row of a stripe are recorded in that stripe's
    // border area, a neighbour's over NVLink (kernels.cuh)
    ds.border = event_area<T>(s->events, border_entries(s), s->ev_slots);
    ds.border_up = event_area<T>((s->stripe && s->above.present) ? s->above.events : nullptr, border_entries(s), s->ev_slots);
    ds.border_dn = event_area<T>((s->stripe && s->below.present) ? s->below.events : nullptr, border_entries(s), s->ev_slots);
    ds.P = s->P;
    ds.border_cols = s->g.C + 2;
    ds.cta_outlets = s->d_cta_outlets;
    return ds;
}

bool serial_drain(const wdpm_solver* s) { return s->schedule == WDPM_SCHEDULE_SERIAL && s->module == WDPM_DRAIN; }

// Serial-schedule fp64 Subtract on water that may hold -0.0 (wdpm_solver::negzero_free): the Add step must keep
// the reference's gate.
bool needs_ref_add(const wdpm_solver* s) { return s->dtype == WDPM_F64 && s->relax == WDPM_ADD && s->module != WDPM_ADD && !s->negzero_free; }

// Serial-schedule Drain: empty the outlet's 3x3 after the iteration that produced w[cur] (kernels.cuh,
// k_outlet_wipe). `direct`: add the sum to the total at once (colour kernel); otherwise it goes into the event
// buffer of that iteration's launch, after its contacts, and is folded with them.
template <typename T>
int outlet_wipe(wdpm_solver* s, bool direct) {
    k_outlet_wipe<T><<<1, 32, 0, s->stream>>>(static_cast<T*>(s->w[s->cur]), static_cast<const T*>(s->dem), s->g, drain_state<T>(s),
                                              prev_event_slot(s->launch_slot), direct ? 1 : 0);
    s->launches++;
    s->wipe_due = false;
    CUDA_TRY(cudaGetLastError());
    return WDPM_OK;
}

constexpr int kMaxOutlets = WDPM_MAX_OUTLETS;
constexpr size_t kFlagsBytes = 256;  // HaloFlags, padded; a Drain stripe's border event area follows in the same allocation

// grid of the event fold: enough threads for the touched entries (at most the area's entries)
int fold_grid(const wdpm_solver* s) {
    const long long n = (long long)s->outlet_cap + (s->events ? border_entries(s) : 0);
    return (int)std::min<long long>((n + 255) / 256, (long long)s->sm_count * 4);
}

// Row stripes: load, at creation, every kernel a stripe enqueues behind a k_halo_wait. With lazy module loading
// (the CUDA default) a kernel's first launch loads it, and loading may wait for the kernels running on the device. On
// one device, a stripe's k_halo_wait spins until its neighbour's iteration kernel has run; if the host is still in the
// first launch of, say, k_fold_events for this stripe, it has not launched the neighbour's kernel yet, and the wait
// ends only at its timeout (WDPM_E_HALO). cudaFuncGetAttributes loads the kernel without running it.
template <typename T>
cudaError_t preload_stripe_kernels() {
    cudaFuncAttributes a;
    cudaError_t e;
    if ((e = cudaFuncGetAttributes(&a, (const void*)k_halo_wait)) != cudaSuccess) return e;
    if ((e = cudaFuncGetAttributes(&a, (const void*)k_block_prologue<T>)) != cudaSuccess) return e;
    if ((e = cudaFuncGetAttributes(&a, (const void*)k_gather_totals<T>)) != cudaSuccess) return e;
    if ((e = cudaFuncGetAttributes(&a, (const void*)k_outlet_wipe<T>)) != cudaSuccess) return e;
    return cudaFuncGetAttributes(&a, (const void*)k_fold_events<T>);
}

int grid_for(long long n, int threads, int sm_count) {
    long long b = (n + threads - 1) / threads;
    const long long cap = (long long)sm_count * 16;
    if (b > cap) b = cap;
    if (b < 1) b = 1;
    return (int)b;
}

template <typename T>
int colour_subpass(wdpm_solver* s, int oi, int oj) {
    const dim3 block(32, 8);
    const int ncx = (s->g.C - oj) / 3 + 1, ncy = (s->g.R - oi) / 3 + 1;
    if (ncx <= 0 || ncy <= 0) return WDPM_OK;
    const dim3 grid((ncx + block.x - 1) / block.x, (ncy + block.y - 1) / block.y);
    T* w = static_cast<T*>(s->w[s->cur]);
    const T* d = static_cast<const T*>(s->dem);
    DrainState<T> ds = drain_state<T>(s);
    switch (s->relax) {
        case WDPM_ADD: k_colour<T, kAdd><<<grid, block, 0, s->stream>>>(w, d, s->g, oi, oj, ds); break;
        case WDPM_SUBTRACT: k_colour<T, kSubtract><<<grid, block, 0, s->stream>>>(w, d, s->g, oi, oj, ds); break;
        default: k_colour<T, kDrain><<<grid, block, 0, s->stream>>>(w, d, s->g, oi, oj, ds); break;
    }
    s->launches++;
    CUDA_TRY(cudaGetLastError());
    return WDPM_OK;
}

template <typename T>
int colour_iterations(wdpm_solver* s, int n) {
    for (int it = 0; it < n; it++) {
        for (int oi = 1; oi <= 3; oi++)
            for (int oj = 1; oj <= 3; oj++) {
                const int rc = colour_subpass<T>(s, oi, oj);
                if (rc) return rc;
            }
        if (serial_drain(s)) {
            const int rc = outlet_wipe<T>(s, true);
            if (rc) return rc;
        }
    }
    return WDPM_OK;
}

// Fill in what the iteration kernel needs to export this iteration's halo rows (kernels.cuh, FusedParams).
// The neighbours run in lockstep on the buffer index, so their target buffer has my output's index.
template <typename T>
void set_halo_export(wdpm_solver* s, FusedParams<T>& p) {
    const bool up = s->stripe && s->above.present, dn = s->stripe && s->below.present;
    if (s->stripe) s->epoch++;
    p.up_out = up ? static_cast<T*>(s->above.w[s->cur ^ 1]) : nullptr;
    p.dn_out = dn ? static_cast<T*>(s->below.w[s->cur ^ 1]) : nullptr;
    p.P_self = s->P;
    p.P_up = s->above.P;
    p.self_flags = s->flags;
    p.up_flags = up ? s->above.flags : nullptr;
    p.dn_flags = dn ? s->below.flags : nullptr;
    p.up_ctas = p.dn_ctas = 0;
    int dn_reach = kHaloBelow;  // every CTA that reads my bottom-halo rows counts, see k_fused
#ifdef WDPM_TEST_HOOKS
    p.dbg_old_dn_count = getenv("WDPM_TEST_HALO_OLD_COUNT") ? atoi(getenv("WDPM_TEST_HALO_OLD_COUNT")) : 0;
    p.dbg_reader_delay_ns = getenv("WDPM_TEST_HALO_READER_DELAY_NS") ? atoi(getenv("WDPM_TEST_HALO_READER_DELAY_NS")) : 0;
    if (p.dbg_old_dn_count) dn_reach = kHaloAbove;
#endif
    for (int c = 0; c < s->n_chunks; c++) {  // the kernel's own test, per chunk of rows (all strips of a chunk agree)
        const int m0 = c * s->chunk_triples;
        const int m1 = m0 + s->chunk_triples < s->total_triples ? m0 + s->chunk_triples : s->total_triples;
        if (up && 3 * m0 < kHaloBelow) p.up_ctas += s->n_strips;
        if (dn && 3 * m1 > s->P - dn_reach && 3 * m0 < s->P) p.dn_ctas += s->n_strips;
    }
    p.epoch = s->epoch;
}

template <typename T>
int fused_launch_only(wdpm_solver* s);

template <typename T>
FusedLaunchFn<T> pick_launch(const wdpm_solver* s, const FusedVariant<T>& v) {
    if (needs_ref_add(s) && v.launch_ref_add) return v.launch_ref_add;
    return (s->water_clean && v.launch_clean[s->relax]) ? v.launch_clean[s->relax] : v.launch[s->relax];
}

template <typename T>
int fused_iterations(wdpm_solver* s, int n) {
    const FusedVariant<T>& v = fused_variants<T>()[s->variant];
    const int n_launch = n / v.K;
    for (int l = 0; l < n_launch; l++) {
        FusedParams<T> p;
        p.w_in = static_cast<const T*>(s->w[s->cur]);
        p.w_out = static_cast<T*>(s->w[s->cur ^ 1]);
        p.dem = static_cast<const T*>(s->dem);
        p.g = s->g;
        p.n_strips = s->n_strips;
        p.chunk_triples = s->chunk_triples;
        p.total_triples = s->total_triples;
        p.launch_slot = s->launch_slot;
        p.ds = drain_state<T>(s);
        if (s->stripe && s->epoch > 0 && (s->above.present || s->below.present)) {
            k_halo_wait<<<1, 32, 0, s->stream>>>(s->flags, s->above.present, s->below.present, s->epoch, s->halo_timeout_ns);
            s->launches++;
        }
        // Serial-schedule Drain: the previous iteration's emptying. A row stripe does it after the wait above: its
        // copy of a neighbour's rows of the 3x3 has then arrived (with values from before the emptying), and every
        // stripe that holds one of the nine cells zeroes its own copy.
        if (s->wipe_due) {
            const int rc = outlet_wipe<T>(s, false);
            if (rc) return rc;
        }
        set_halo_export<T>(s, p);  // the launch also pushes the halo rows and raises the neighbours' flags
        CUDA_TRY(pick_launch<T>(s, v)(p, s->n_strips * s->n_chunks, s->stream));
        s->launches++;
        s->cur ^= 1;
        s->launch_slot = next_event_slot(s->launch_slot);
        s->wipe_due = serial_drain(s);
    }
    if (s->module == WDPM_DRAIN && n_launch > 0) {
        if (s->stripe && (s->above.present || s->below.present)) {
            // the neighbours' last iteration records contacts with my outlets in my buffers: wait for it
            k_halo_wait<<<1, 32, 0, s->stream>>>(s->flags, s->above.present, s->below.present, s->epoch, s->halo_timeout_ns);
            s->launches++;
        }
        if (s->wipe_due) {
            const int rc = outlet_wipe<T>(s, false);
            if (rc) return rc;
        }
        k_fold_events<T><<<fold_grid(s), 256, 0, s->stream>>>(drain_state<T>(s), prev_event_slot(s->launch_slot));
        s->launches++;
        CUDA_TRY(cudaGetLastError());
    }
    // iterations that do not fill a launch run through the colour kernel (same results)
    return colour_iterations<T>(s, n - n_launch * v.K);
}

// The iteration kernel alone (no halo wait; it exports its halo rows itself): hosts driving in-process
// stripes in lockstep.
template <typename T>
int fused_launch_only(wdpm_solver* s) {
    const FusedVariant<T>& v = fused_variants<T>()[s->variant];
    FusedParams<T> p;
    p.w_in = static_cast<const T*>(s->w[s->cur]);
    p.w_out = static_cast<T*>(s->w[s->cur ^ 1]);
    p.dem = static_cast<const T*>(s->dem);
    p.g = s->g;
    p.n_strips = s->n_strips;
    p.chunk_triples = s->chunk_triples;
    p.total_triples = s->total_triples;
    p.launch_slot = s->launch_slot;
    p.ds = drain_state<T>(s);
    set_halo_export<T>(s, p);
    CUDA_TRY(pick_launch<T>(s, v)(p, s->n_strips * s->n_chunks, s->stream));
    s->launches++;
    s->cur ^= 1;
    s->launch_slot = next_event_slot(s->launch_slot);
    s->wipe_due = serial_drain(s);
    return WDPM_OK;  // Drain: the contacts are folded by the next launch, or by phase 1 (fold_last_launch)
}

// Lockstep hosts: fold the contacts of the last iteration once EVERY stripe has run it (a neighbour records the
// contacts of its centres with my outlets in my buffers).
template <typename T>
int fold_last_launch(wdpm_solver* s) {
    if (s->module != WDPM_DRAIN) return WDPM_OK;
    if (s->wipe_due) {  // serial schedule: every stripe's copy of the last iteration's rows is in place by now
        const int rc = outlet_wipe<T>(s, false);
        if (rc) return rc;
    }
    k_fold_events<T><<<fold_grid(s), 256, 0, s->stream>>>(drain_state<T>(s), prev_event_slot(s->launch_slot));
    s->launches++;
    CUDA_TRY(cudaGetLastError());
    return WDPM_OK;
}

constexpr int kResidentThreads = 512;

template <typename T, int MODULE>
cudaError_t launch_resident(wdpm_solver* s, int n) {
    ResidentParams<T> p;
    p.w[0] = static_cast<T*>(s->w[0]);
    p.w[1] = static_cast<T*>(s->w[1]);
    p.dem = static_cast<const T*>(s->dem);
    p.g = s->g;
    p.cur = s->cur;
    p.TR = s->res_TR;
    p.TC = s->res_TC;
    p.n_tx = s->res_ntx;
    p.n_iters = n;
    p.launch_slot = s->launch_slot;
    p.serial_wipe = serial_drain(s) ? 1 : 0;
    p.ds = drain_state<T>(s);
    void* args[] = {&p};
    auto kern = k_resident<T, MODULE, kResidentThreads>;  // shared-memory limit set in wdpm_create (resident_fits)
    return cudaLaunchCooperativeKernel((void*)kern, dim3(s->res_ntx * s->res_nty), dim3(kResidentThreads), args, s->res_smem, s->stream);
}

// Can the whole grid of the resident kernel be co-resident (a cooperative launch needs it)? Also sets the
// kernel's dynamic shared-memory limit once. Called from wdpm_create.
template <typename T, int MODULE>
bool resident_fits(const wdpm_solver* s) {
    auto kern = k_resident<T, MODULE, kResidentThreads>;
    if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)s->res_smem) != cudaSuccess) { cudaGetLastError(); return false; }
    int per_sm = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, kResidentThreads, s->res_smem) != cudaSuccess) { cudaGetLastError(); return false; }
    return (long long)per_sm * s->sm_count >= (long long)s->res_ntx * s->res_nty;
}

template <typename T>
bool resident_fits_module(const wdpm_solver* s) {
    switch (s->relax) {
        case WDPM_ADD: return resident_fits<T, kAdd>(s);
        case WDPM_SUBTRACT: return resident_fits<T, kSubtract>(s);
        default: return resident_fits<T, kDrain>(s);
    }
}

template <typename T>
int resident_iterations(wdpm_solver* s, int n) {
    if (n <= 0) return WDPM_OK;
    cudaError_t e;
    switch (s->relax) {
        case WDPM_ADD: e = launch_resident<T, kAdd>(s, n); break;
        case WDPM_SUBTRACT: e = launch_resident<T, kSubtract>(s, n); break;
        default: e = launch_resident<T, kDrain>(s, n); break;
    }
    if (e != cudaSuccess && s->resident_by_auto) {
        // AUTO chose this kernel; the cooperative launch can still be refused at run time (GPU shared with other
        // contexts, fewer SMs available): nothing has run, so fall back to the fused kernel for good
        cudaGetLastError();
        s->kernel = WDPM_KERNEL_FUSED;
        s->resident_by_auto = false;
        return fused_iterations<T>(s, n);
    }
    CUDA_TRY(e);
    s->launches++;
    if (n & 1) s->cur ^= 1;
    s->launch_slot = (s->launch_slot + n) % kEventSlots;
    return WDPM_OK;
}

template <typename T>
int iterate_t(wdpm_solver* s, int n) {
    // the resident kernel's fp64 Add step is the sign-gated one: the colour kernel runs the reference form instead
    if (s->kernel == WDPM_KERNEL_RESIDENT && needs_ref_add(s)) return colour_iterations<T>(s, n);
    if (s->kernel == WDPM_KERNEL_RESIDENT) return resident_iterations<T>(s, n);
    if (s->kernel == WDPM_KERNEL_FUSED) return fused_iterations<T>(s, n);
    return colour_iterations<T>(s, n);
}

int iterate(wdpm_solver* s, int n) {
    return s->dtype == WDPM_F64 ? iterate_t<double>(s, n) : iterate_t<float>(s, n);
}

// The interior rows this solver owns in a device grid: address of the first one's first cell, and their number
// (all rows of a single solver; a stripe's owned rows clipped to the DEM).
const char* owned_interior(const wdpm_solver* s, const void* base, int* n_rows) {
    const int lo = std::max(s->G, 1), hi = std::min(s->G + s->P, s->cfg.rows + 1);
    *n_rows = hi - lo;
    return static_cast<const char*>(base) + ((size_t)(lo - s->G + kPadTop) * s->g.pitch + (size_t)(1 + kPadLeft)) * s->esize;
}

// Device-side ordering against the last checkpoint capture: work enqueued after this on the solver stream starts
// only once the capture's copies out of oldw and d_ck_totals have completed.
int ck_fence(wdpm_solver* s) {
    if (s->ck_done) CUDA_TRY(cudaStreamWaitEvent(s->stream, s->ck_done, 0));
    return WDPM_OK;
}

// An armed capture, right after the prologue: gather the totals, then copy them and the snapshot to the staging on
// the side stream, which waits for the prologue and the gather on the device.
template <typename T>
int capture_t(wdpm_solver* s) {
    // sized here, not at the arm: a larger outlet set may have been installed since
    const int n = std::max(s->n_outlets, 1);
    if (n > s->ck_cap) {
        CUDA_TRY(cudaStreamSynchronize(s->ck_stream));  // the last capture's copy still reads the old arrays
        if (s->ck_totals) cudaFreeHost(s->ck_totals);
        if (s->d_ck_totals) cudaFree(s->d_ck_totals);
        s->ck_totals = s->d_ck_totals = nullptr;
        s->device_bytes -= (long long)sizeof(double) * s->ck_cap;
        s->ck_cap = 0;
        CUDA_TRY(cudaHostAlloc((void**)&s->ck_totals, sizeof(double) * n, cudaHostAllocDefault));
        CUDA_TRY(cudaMalloc((void**)&s->d_ck_totals, sizeof(double) * n));
        s->ck_cap = n;
        s->device_bytes += (long long)sizeof(double) * n;
    }
    k_gather_totals<T><<<(n + 255) / 256, 256, 0, s->stream>>>(static_cast<const T*>(s->totaldrain), s->d_outlet_pos, n, s->d_ck_totals);
    s->launches++;
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaEventRecord(s->ck_ready, s->stream));
    CUDA_TRY(cudaStreamWaitEvent(s->ck_stream, s->ck_ready, 0));
    int rows = 0;
    const char* src = owned_interior(s, s->oldw, &rows);
    CUDA_TRY(cudaMemcpy2DAsync(s->ck_water, (size_t)s->g.C * s->esize, src, (size_t)s->g.pitch * s->esize, (size_t)s->g.C * s->esize,
                               (size_t)rows, cudaMemcpyDeviceToHost, s->ck_stream));
    CUDA_TRY(cudaMemcpyAsync(s->ck_totals, s->d_ck_totals, sizeof(double) * n, cudaMemcpyDeviceToHost, s->ck_stream));
    CUDA_TRY(cudaEventRecord(s->ck_done, s->ck_stream));
    s->ck_armed = false;
    s->ck_captured = true;
    s->ck_n = n;
    return WDPM_OK;
}

// A block in three non-blocking-then-blocking pieces (see wdpm_block_begin/enqueue/end).
template <typename T>
int block_begin_t(wdpm_solver* s) {
    const long long n = s->g.cells_dev();
    s->blk_launches0 = s->launches;
    s->blk_iters = 0;
    CUDA_TRY(cudaEventRecord(s->ev[0], s->stream));
    {   // the prologue overwrites oldw, and an armed one the gathered totals: not before the last capture is out
        const int rc = ck_fence(s);
        if (rc) return rc;
    }
    if (s->stripe && s->epoch > 0 && (s->above.present || s->below.present)) {
        // the neighbours' last halo push must land before the threshold pass touches the halo rows
        k_halo_wait<<<1, 32, 0, s->stream>>>(s->flags, s->above.present, s->below.present, s->epoch, s->halo_timeout_ns);
        s->launches++;
    }
    if (s->cfg.zero_threshold > 0.0 && s->invalid_dry) s->water_clean = true;  // no negative water, no -0.0 left (see wdpm_solver)
    if (s->cfg.zero_threshold > 0.0) s->negzero_free = true;
    CUDA_TRY(cudaMemsetAsync(s->d_dirty, 0, sizeof(int), s->stream));
    k_block_prologue<T><<<grid_for(n, 256, s->sm_count), 256, 0, s->stream>>>(
        static_cast<T*>(s->w[s->cur]), static_cast<T*>(s->oldw), static_cast<const T*>(s->dem), n, (T)s->cfg.zero_threshold, s->d_dirty);
    s->launches++;
    CUDA_TRY(cudaGetLastError());
    if (s->ck_armed) {
        const int rc = capture_t<T>(s);
        if (rc) return rc;
    }
    CUDA_TRY(cudaEventRecord(s->ev[1], s->stream));
    s->in_block = true;
    return WDPM_OK;
}

template <typename T>
int block_end_t(wdpm_solver* s, wdpm_block_result* out) {
    CUDA_TRY(cudaEventRecord(s->ev[2], s->stream));
    k_block_reduce_stage1<T, 256><<<s->reduce_blocks, 256, 0, s->stream>>>(
        static_cast<const T*>(s->w[s->cur]), static_cast<const T*>(s->oldw), static_cast<const T*>(s->dem), s->g, s->partials);
    k_block_reduce_stage2<<<1, 32, 0, s->stream>>>(s->partials, s->reduce_blocks, s->d_result);
    s->launches += 2;
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaMemcpyAsync(s->h_result, s->d_result, sizeof(BlockPartial), cudaMemcpyDeviceToHost, s->stream));
    // one outlet: the reference's totaldrain; a set: summed in outlet order, solver precision, on the device
    k_sum_totals<T><<<1, 32, 0, s->stream>>>(static_cast<const T*>(s->totaldrain), s->d_outlet_pos, std::max(s->n_outlets, 1), s->d_total);
    s->launches++;
    CUDA_TRY(cudaGetLastError());
    double td = 0.0;
    CUDA_TRY(cudaMemcpyAsync(&td, s->d_total, sizeof(double), cudaMemcpyDeviceToHost, s->stream));
    if (s->stripe) CUDA_TRY(cudaMemcpyAsync(s->h_halo_error, &s->flags->error, sizeof(int), cudaMemcpyDeviceToHost, s->stream));
    int dirty = 1;
    CUDA_TRY(cudaMemcpyAsync(&dirty, s->d_dirty, sizeof(int), cudaMemcpyDeviceToHost, s->stream));
    CUDA_TRY(cudaEventRecord(s->ev[3], s->stream));
    CUDA_TRY(cudaStreamSynchronize(s->stream));
    if (s->stripe && *s->h_halo_error) {
        s->in_block = false;
        s->halo_failed = true;
        return fail(WDPM_E_HALO, "a neighbouring stripe's halo did not arrive in time (WDPM_B200_HALO_TIMEOUT_MS): the block's results are void; upload again");
    }
    s->invalid_dry = dirty == 0;  // as of this block's prologue; the kernels never put water on an invalid cell
    s->in_block = false;
    if (out) {
        out->max_diff = s->h_result->max_diff;
        out->masked_sum = s->h_result->sum;
        out->wet_cells = (int64_t)s->h_result->wet;
        out->total_drain = td;
        out->iterations = s->blk_iters;
        out->launches = (int32_t)(s->launches - s->blk_launches0);
        CUDA_TRY(cudaEventElapsedTime(&out->block_ms, s->ev[0], s->ev[3]));
        CUDA_TRY(cudaEventElapsedTime(&out->iterate_ms, s->ev[1], s->ev[2]));
    }
    return WDPM_OK;
}

template <typename T>
int run_block_t(wdpm_solver* s, int n_iters, wdpm_block_result* out) {
    int rc = block_begin_t<T>(s);
    if (rc) return rc;
    rc = iterate_t<T>(s, n_iters);
    if (rc) return rc;
    s->blk_iters += n_iters;
    return block_end_t<T>(s, out);
}

template <typename T>
int fill_dem(wdpm_solver* s) {
    const long long n = s->g.cells_dev();
    k_fill<T><<<grid_for(n, 256, s->sm_count), 256, 0, s->stream>>>(static_cast<T*>(s->dem), n, invalid_elevation<T>());
    s->launches++;
    CUDA_TRY(cudaGetLastError());
    return WDPM_OK;
}

void* interior_ptr(wdpm_solver* s, void* base) {
    return static_cast<char*>(base) + ((size_t)(1 + kPadTop) * s->g.pitch + (size_t)(1 + kPadLeft)) * s->esize;
}

int upload_grid(wdpm_solver* s, void* dst_base, const void* host) {
    CUDA_TRY(cudaMemcpy2DAsync(interior_ptr(s, dst_base), (size_t)s->g.pitch * s->esize, host, (size_t)s->g.C * s->esize,
                               (size_t)s->g.C * s->esize, (size_t)s->g.R, cudaMemcpyHostToDevice, s->stream));
    return WDPM_OK;
}

// Pick the number of row chunks: whole waves of CTAs, counting the per-chunk
// pipeline fill (halo triples + phase lags) as wasted steps.
void choose_chunks(wdpm_solver* s, int K, int NT, int minb, int forced_rows) {
    const int total = s->total_triples;
    if (forced_rows > 0) {
        s->chunk_triples = (forced_rows + 2) / 3;
        if (s->chunk_triples > total) s->chunk_triples = total;
        s->n_chunks = (total + s->chunk_triples - 1) / s->chunk_triples;
        return;
    }
    const int slots = s->sm_count * (minb > 0 ? minb : 1);
    const int fill = 3 * K + (3 * K - 1) * (NT + 1);
    double best_cost = 1e300;
    int best_ct = total;
    const int max_chunks = total / 3 > 0 ? total / 3 : 1;  // at least three row triples per CTA
    for (int nch = 1; nch <= max_chunks && nch <= 4096; nch++) {
        const int ct = (total + nch - 1) / nch;
        const int real_nch = (total + ct - 1) / ct;
        const long long ctas = (long long)real_nch * s->n_strips;
        const long long waves = (ctas + slots - 1) / slots;
        const double cost = (double)waves * (ct + fill);
        if (cost < best_cost - 1e-9) { best_cost = cost; best_ct = ct; }
    }
    s->chunk_triples = best_ct;
    s->n_chunks = (total + best_ct - 1) / best_ct;
}

// Put the outlet marks into the elevation grid (on = true) or take them out again, restoring the
// elevations they replaced (kernels.cuh, k_mark_outlets). Idempotent. An outlet on a cell with dem <= nodata in the
// rows this solver holds DEM data for uninstalls the set and returns WDPM_E_ARG: the mark would make that cell count
// as valid in the block reductions.
int apply_outlet_marks(wdpm_solver* s, bool on) {
    if (s->n_outlets == 0 || s->marks_applied == on) return WDPM_OK;
    const int n = s->n_outlets, blocks = (n + 127) / 128;
    // local rows with DEM data: the interior rows of the band a stripe was given (owned rows + halos)
    const int data_lo = std::max(s->G - kHaloAbove, 1) - s->G, data_hi = std::min(s->G + s->P + kHaloBelow, s->cfg.rows + 1) - s->G;
    if (on) CUDA_TRY(cudaMemsetAsync(s->d_bad, 0, sizeof(int), s->stream));
    if (s->dtype == WDPM_F64)
        k_mark_outlets<double><<<blocks, 128, 0, s->stream>>>(static_cast<double*>(s->dem), s->g, s->d_outlet_rc, n, static_cast<double*>(s->saved_elev), on ? 0 : 1,
                                                              s->stripe ? data_lo : 1, s->stripe ? data_hi : s->g.R + 1, s->d_bad);
    else
        k_mark_outlets<float><<<blocks, 128, 0, s->stream>>>(static_cast<float*>(s->dem), s->g, s->d_outlet_rc, n, static_cast<float*>(s->saved_elev), on ? 0 : 1,
                                                             s->stripe ? data_lo : 1, s->stripe ? data_hi : s->g.R + 1, s->d_bad);
    s->launches++;
    CUDA_TRY(cudaGetLastError());
    s->marks_applied = on;
    if (!on) return WDPM_OK;
    int bad = 0;
    CUDA_TRY(cudaMemcpyAsync(&bad, s->d_bad, sizeof(int), cudaMemcpyDeviceToHost, s->stream));
    CUDA_TRY(cudaStreamSynchronize(s->stream));
    if (bad == 0) return WDPM_OK;
    const int rc = apply_outlet_marks(s, false);
    if (rc) return rc;
    s->n_outlets = 0;
    s->have_outlet = false;
    return fail(WDPM_E_ARG, std::to_string(bad) + " outlet(s) on cells with dem <= nodata: the set is refused");
}

// (Re)allocate the per-outlet arrays for `cap` outlets; new arrays are zeroed.
int alloc_outlets(wdpm_solver* s, int cap) {
    if (cap == s->outlet_cap) return WDPM_OK;
    const size_t ev_bytes = event_area_bytes(cap, s->ev_slots, s->esize);
    const size_t old_bytes = s->outlet_cap ? event_area_bytes(s->outlet_cap, s->ev_slots, s->esize) + (size_t)s->outlet_cap * (2 * s->esize + 12) : 0;
    void* ptrs[] = {s->totaldrain, s->ev_area, s->saved_elev, s->d_outlet_rc, s->d_outlet_pos};
    for (void* p : ptrs)
        if (p) cudaFree(p);
    s->totaldrain = s->ev_area = s->saved_elev = nullptr;
    s->d_outlet_rc = s->d_outlet_pos = nullptr;
    s->device_bytes -= (long long)old_bytes;
    s->outlet_cap = 0;
    CUDA_TRY(cudaMalloc(&s->totaldrain, s->esize * cap));
    CUDA_TRY(cudaMalloc(&s->ev_area, ev_bytes));
    CUDA_TRY(cudaMalloc(&s->saved_elev, s->esize * cap));
    CUDA_TRY(cudaMalloc((void**)&s->d_outlet_rc, sizeof(int) * 2 * cap));
    CUDA_TRY(cudaMalloc((void**)&s->d_outlet_pos, sizeof(int) * cap));
    CUDA_TRY(cudaMemsetAsync(s->totaldrain, 0, s->esize * cap, s->stream));
    CUDA_TRY(cudaMemsetAsync(s->ev_area, 0, ev_bytes, s->stream));
    CUDA_TRY(cudaMemsetAsync(s->d_outlet_pos, 0, sizeof(int) * cap, s->stream));
    s->outlet_cap = cap;
    s->device_bytes += (long long)(ev_bytes + (size_t)cap * (2 * s->esize + 12));
    return WDPM_OK;
}

// Which CTAs of the fused kernels stage an outlet cell (kernels.cuh, k_fused / k_fused_wa: s_cta_has_outlets). A
// CTA of strip st and chunk c stages padded columns [st*TWV - HL, st*TWV - HL + W) and the rows of triples
// m_lo = c*chunk - K .. m_hi = min((c+1)*chunk, total) + 2K - 1 (mw_schedule.h, MwTile::init).
template <typename T>
int compute_cta_outlets(wdpm_solver* s) {
    const FusedVariant<T>& v = fused_variants<T>()[s->variant];
    const int top = v.wa ? 1 : v.K, bot = v.wa ? 2 : 2 * v.K;
    const int ct = s->chunk_triples;
    std::vector<unsigned char> flags((size_t)s->n_strips * s->n_chunks, 0);
    for (int k = 0; k < s->n_outlets; k++) {
        const int r = s->outlet_rc[2 * k], col = s->outlet_rc[2 * k + 1];
        const int c_first = std::max(0, (r / 3 - bot - ct) / ct - 1), c_last = std::min(s->n_chunks - 1, (r / 3 + top) / ct + 1);
        for (int c = c_first; c <= c_last; c++) {
            const int m_lo = c * ct - top, m_hi = std::min((c + 1) * ct, s->total_triples) + bot - 1;
            if (r < 3 * m_lo || r > 3 * m_hi + 2) continue;
            const int st_first = std::max(0, (col + v.HL - v.W) / v.TWV), st_last = std::min(s->n_strips - 1, (col + v.HL) / v.TWV);
            for (int st = st_first; st <= st_last; st++) {
                const int x0 = st * v.TWV - v.HL;
                if (col >= x0 && col < x0 + v.W) flags[(size_t)c * s->n_strips + st] = 1;
            }
        }
    }
    CUDA_TRY(cudaMemcpyAsync(s->d_cta_outlets, flags.data(), flags.size(), cudaMemcpyHostToDevice, s->stream));
    CUDA_TRY(cudaStreamSynchronize(s->stream));
    return WDPM_OK;
}

// After any change of the water grid from outside (upload, copy, quantise): nothing is known about signs until the
// next block prologue; whether invalid cells are dry is established here (one pass, the callers synchronise anyway).
int refresh_water_flags(wdpm_solver* s) {
    s->water_clean = false;
    s->negzero_free = false;
    s->wipe_due = false;  // new water: an emptying still pending belonged to the old one
    const long long n = s->g.cells_dev();
    const int grid = grid_for(n, 256, s->sm_count);
    CUDA_TRY(cudaMemsetAsync(s->d_dirty, 0, sizeof(int), s->stream));
    if (s->dtype == WDPM_F64) k_check_invalid_water<double><<<grid, 256, 0, s->stream>>>(static_cast<const double*>(s->w[s->cur]), static_cast<const double*>(s->dem), n, s->d_dirty);
    else k_check_invalid_water<float><<<grid, 256, 0, s->stream>>>(static_cast<const float*>(s->w[s->cur]), static_cast<const float*>(s->dem), n, s->d_dirty);
    s->launches++;
    CUDA_TRY(cudaGetLastError());
    int dirty = 1;
    CUDA_TRY(cudaMemcpyAsync(&dirty, s->d_dirty, sizeof(int), cudaMemcpyDeviceToHost, s->stream));
    CUDA_TRY(cudaStreamSynchronize(s->stream));
    s->invalid_dry = dirty == 0;
    return WDPM_OK;
}

}  // namespace

// ---------------------------------------------------------------------------
// extern "C"
// ---------------------------------------------------------------------------

extern "C" {

const char* wdpm_last_error(void) { return g_err.c_str(); }
int wdpm_abi_version(void) { return WDPM_ABI_VERSION; }

int wdpm_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}

int wdpm_fused_variant_info(int32_t variant, int32_t dtype, int32_t* window_cols, int32_t* strip_cols,
                            int32_t* iters_per_launch, int32_t* cta_threads, int32_t* smem_bytes) {
    if (variant < 1) return fail(WDPM_E_ARG, "variant ids start at 1");
    int W, TWV, K, nt; size_t smem;
    if (dtype == WDPM_F64) {
        const auto& v = fused_variants<double>();
        if (variant > (int)v.size()) return fail(WDPM_E_ARG, "no such fused variant");
        W = v[variant - 1].W; TWV = v[variant - 1].TWV; K = v[variant - 1].K; nt = v[variant - 1].nthreads; smem = v[variant - 1].smem;
    } else if (dtype == WDPM_F32) {
        const auto& v = fused_variants<float>();
        if (variant > (int)v.size()) return fail(WDPM_E_ARG, "no such fused variant");
        W = v[variant - 1].W; TWV = v[variant - 1].TWV; K = v[variant - 1].K; nt = v[variant - 1].nthreads; smem = v[variant - 1].smem;
    } else {
        return fail(WDPM_E_ARG, "dtype must be WDPM_F32 or WDPM_F64");
    }
    if (window_cols) *window_cols = W;
    if (strip_cols) *strip_cols = TWV;
    if (iters_per_launch) *iters_per_launch = K;
    if (cta_threads) *cta_threads = nt;
    if (smem_bytes) *smem_bytes = (int32_t)smem;
    return WDPM_OK;
}

int wdpm_create(const wdpm_config* cfg, wdpm_solver** out) {
    if (!cfg || !out) return fail(WDPM_E_ARG, "null argument");
    *out = nullptr;
    if (cfg->struct_size != sizeof(wdpm_config)) return fail(WDPM_E_ARG, "wdpm_config.struct_size mismatch (ABI version?)");
    if (cfg->rows < 1 || cfg->cols < 1) return fail(WDPM_E_ARG, "rows and cols must be positive");
    if (cfg->dtype != WDPM_F32 && cfg->dtype != WDPM_F64) return fail(WDPM_E_ARG, "dtype must be WDPM_F32 or WDPM_F64");
    if (cfg->module < WDPM_ADD || cfg->module > WDPM_DRAIN) return fail(WDPM_E_ARG, "unknown module");
    if (cfg->kernel < WDPM_KERNEL_AUTO || cfg->kernel > WDPM_KERNEL_RESIDENT) return fail(WDPM_E_ARG, "unknown kernel selector");
    if (cfg->schedule != WDPM_SCHEDULE_OPENCL && cfg->schedule != WDPM_SCHEDULE_SERIAL) return fail(WDPM_E_ARG, "unknown schedule");
    const bool is_stripe = cfg->stripe_rows > 0;
    if (is_stripe) {
        if (cfg->stripe_row0 < 0 || cfg->stripe_row0 % 3 != 0) return fail(WDPM_E_ARG, "stripe_row0 must be a non-negative multiple of 3");
        if (cfg->stripe_row0 + cfg->stripe_rows > cfg->rows + 2) return fail(WDPM_E_ARG, "stripe exceeds the padded DEM");
        if (cfg->stripe_rows % 3 != 0 && cfg->stripe_row0 + cfg->stripe_rows != cfg->rows + 2)
            return fail(WDPM_E_ARG, "stripe_rows must be a multiple of 3 unless the stripe ends the DEM");
        if (cfg->stripe_rows < 9) return fail(WDPM_E_ARG, "a stripe needs at least 9 rows (its neighbours' halos come from it)");
        if (cfg->kernel == WDPM_KERNEL_COLOUR) return fail(WDPM_E_UNSUPPORTED, "stripes need the fused kernel");
    } else if (cfg->stripe_row0 != 0) {
        return fail(WDPM_E_ARG, "stripe_row0 without stripe_rows");
    }
    if ((long long)(cfg->rows + 64) * (long long)(cfg->cols + 2048) > (1ll << 40)) return fail(WDPM_E_ARG, "grid too large");

    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
        cudaGetLastError();
        return fail(WDPM_E_CUDA, "no CUDA device: this library has no CPU path");
    }
    if (cfg->device < 0 || cfg->device >= ndev) return fail(WDPM_E_ARG, "device ordinal out of range");
    CUDA_TRY(cudaSetDevice(cfg->device));

    wdpm_solver* s = new (std::nothrow) wdpm_solver();
    if (!s) return fail(WDPM_E_NOMEM, "host allocation failed");
    s->cfg = *cfg;
    s->dtype = cfg->dtype;
    s->module = cfg->module;
    s->schedule = cfg->schedule;
    s->relax = (cfg->schedule == WDPM_SCHEDULE_SERIAL && cfg->module == WDPM_SUBTRACT) ? WDPM_ADD : cfg->module;
    s->esize = cfg->dtype == WDPM_F64 ? 8 : 4;
    s->device = cfg->device;
    cudaDeviceProp prop;
    cudaError_t e = cudaGetDeviceProperties(&prop, cfg->device);
    if (e != cudaSuccess) { delete s; return fail(WDPM_E_CUDA, cudaGetErrorString(e)); }
    s->sm_count = prop.multiProcessorCount;
    if (const char* t = getenv("WDPM_B200_HALO_TIMEOUT_MS")) {
        const double ms = atof(t);
        if (ms > 0) s->halo_timeout_ns = (unsigned long long)(ms * 1e6);
    }

    // kernel + variant
    const long long cells = (long long)(cfg->rows + 2) * (cfg->cols + 2);
    s->kernel = cfg->kernel == WDPM_KERNEL_AUTO ? WDPM_KERNEL_FUSED : cfg->kernel;
    if (is_stripe) s->kernel = WDPM_KERNEL_FUSED;
    s->stripe = is_stripe;
    s->G = cfg->stripe_row0;
    s->P = is_stripe ? cfg->stripe_rows : cfg->rows + 2;
    const int nvar = s->dtype == WDPM_F64 ? (int)fused_variants<double>().size() : (int)fused_variants<float>().size();
    int variant = cfg->fused_variant;
    if (variant < 0 || variant > nvar) { delete s; return fail(WDPM_E_ARG, "fused_variant out of range"); }
    if (variant == 0) {
        // one kernel for the three modules (k_fused_wa); Drain's folded-gate step is chosen per launch, while the
        // water is known to hold no -0.0 (wdpm_solver::water_clean), not here
        variant = s->dtype == WDPM_F64 ? kDefaultVariantF64 : kDefaultVariantF32;
        if (cells < kSmallGridCells && !is_stripe) variant = s->dtype == WDPM_F64 ? kSmallGridVariantF64 : kSmallGridVariantF32;
        if (cfg->iters_per_launch > 1) {
            variant = 0;
            for (int i = 0; i < nvar; i++) {
                const int K = s->dtype == WDPM_F64 ? fused_variants<double>()[i].K : fused_variants<float>()[i].K;
                const int W = s->dtype == WDPM_F64 ? fused_variants<double>()[i].W : fused_variants<float>()[i].W;
                if (K == cfg->iters_per_launch && W >= 256) { variant = i + 1; break; }
            }
            if (variant == 0) { delete s; return fail(WDPM_E_UNSUPPORTED, "no production fused variant with that iters_per_launch"); }
        }
    }
    s->variant = variant - 1;
    int W, TWV, HL, K, NT, minb;
    cudaError_t (*prepare)();
    if (s->dtype == WDPM_F64) {
        const auto& v = fused_variants<double>()[s->variant];
        W = v.W; TWV = v.TWV; HL = v.HL; K = v.K; NT = v.NT; minb = v.minb; prepare = v.prepare;
    } else {
        const auto& v = fused_variants<float>()[s->variant];
        W = v.W; TWV = v.TWV; HL = v.HL; K = v.K; NT = v.NT; minb = v.minb; prepare = v.prepare;
    }
    {
        const bool has_module = s->dtype == WDPM_F64 ? fused_variants<double>()[s->variant].launch[s->relax] != nullptr
                                                     : fused_variants<float>()[s->variant].launch[s->relax] != nullptr;
        if (!has_module) { delete s; return fail(WDPM_E_UNSUPPORTED, "this fused variant does not implement the module (warp-autonomous variants: Add and Subtract)"); }
    }
    if (s->kernel == WDPM_KERNEL_FUSED) {
        e = prepare();
        if (e != cudaSuccess) { delete s; return fail(WDPM_E_CUDA, std::string("fused kernel setup: ") + cudaGetErrorString(e)); }
    }

    if (is_stripe && K != 1) { delete s; return fail(WDPM_E_UNSUPPORTED, "stripes need a fused variant with one iteration per launch"); }
    if (is_stripe) {
        e = s->dtype == WDPM_F64 ? preload_stripe_kernels<double>() : preload_stripe_kernels<float>();
        if (e != cudaSuccess) { delete s; return fail(WDPM_E_CUDA, std::string("stripe kernel setup: ") + cudaGetErrorString(e)); }
    }
    // the outlet's emptying sits between two iterations, and its event after the nine sub-pass slots of one iteration
    if (serial_drain(s) && s->kernel == WDPM_KERNEL_FUSED && K != 1) { delete s; return fail(WDPM_E_UNSUPPORTED, "serial-schedule Drain needs a fused variant with one iteration per launch"); }

    // geometry (the tests' schedule emulator uses the same formulas). A stripe is a grid of P padded
    // rows whose halo rows live in the row margins above and below.
    s->g.R = s->P - 2;
    s->g.C = cfg->cols;
    s->n_strips = (cfg->cols + 2 + TWV - 1) / TWV;
    s->total_triples = (s->P + 2) / 3;
    s->g.pitch = ((kPadLeft + s->n_strips * TWV + (W - TWV - HL) + 31) / 32) * 32;
    s->g.nrows_dev = kPadTop + 3 * (s->total_triples + 2 * kMaxItersPerLaunch) + 3;
    {   // room for the resident kernel's tiles (whole tiles + halo, whatever tiling is chosen below)
        const int extra_cols = kPadLeft + (cfg->cols + 2) + (cfg->cols + 2) / 2 + 64;
        const int extra_rows = kPadTop + (s->P) + (s->P) / 2 + 32;
        if ((long long)(cfg->rows + 2) * (cfg->cols + 2) <= (1ll << 21)) {
            s->g.pitch = std::max(s->g.pitch, ((extra_cols + 31) / 32) * 32);
            s->g.nrows_dev = std::max(s->g.nrows_dev, extra_rows);
        }
    }
    choose_chunks(s, K, NT, minb, cfg->fused_chunk_rows);

    // resident tiling: at most one CTA per SM (cooperative launch), tiles aligned to multiples of 3
    if (!is_stripe) {
        int coop = 0;
        cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, cfg->device);
        const int PR = cfg->rows + 2, PC = cfg->cols + 2;
        long long best = -1;
        for (int ntx = 1; ntx <= s->sm_count && coop; ntx++) {
            const int nty_max = s->sm_count / ntx;
            if (nty_max < 1) break;
            const int TC = 3 * ((((PC + ntx - 1) / ntx) + 2) / 3);
            const int nty = std::min(nty_max, std::max(1, (PR + 2) / 3));
            const int TR = 3 * ((((PR + nty - 1) / nty) + 2) / 3);
            const int real_ntx = (PC + TC - 1) / TC, real_nty = (PR + TR - 1) / TR;
            const long long cost = (long long)(TR + kResHaloTop + kResHaloBottom) * (TC + kResHaloLeft + kResHaloRight);
            if (best < 0 || cost < best) {
                best = cost;
                s->res_TR = TR; s->res_TC = TC; s->res_ntx = real_ntx; s->res_nty = real_nty;
            }
        }
        if (best > 0) {
            s->res_smem = (size_t)2 * best * s->esize;
            // a thread should own at most a few tiles per sub-pass, and the tile must fit shared memory
            s->res_ok = s->res_smem <= 200 * 1024 && best <= 9ll * 4 * kResidentThreads && cells <= (1ll << 21);
        }
    }
    if (s->res_ok) s->res_ok = s->dtype == WDPM_F64 ? resident_fits_module<double>(s) : resident_fits_module<float>(s);
    if (cfg->kernel == WDPM_KERNEL_RESIDENT && !s->res_ok) { delete s; return fail(WDPM_E_UNSUPPORTED, "grid too large (or device unsuitable) for the resident kernel"); }
    if (cfg->kernel == WDPM_KERNEL_AUTO && s->res_ok && cells <= (1ll << 20)) { s->kernel = WDPM_KERNEL_RESIDENT; s->resident_by_auto = true; }

    auto cleanup = [&](int code, const std::string& msg) {
        wdpm_destroy(s);
        return fail(code, msg);
    };
    const size_t grid_bytes = (size_t)s->g.cells_dev() * s->esize;
    void** grids[4] = {&s->dem, &s->w[0], &s->w[1], &s->oldw};
    for (auto gp : grids) {
        e = cudaMalloc(gp, grid_bytes);
        if (e != cudaSuccess) return cleanup(WDPM_E_NOMEM, std::string("cudaMalloc grid: ") + cudaGetErrorString(e));
        s->device_bytes += (long long)grid_bytes;
    }
    s->reduce_blocks = s->sm_count * 8;
    // the arrival flags and a Drain stripe's border event area share one allocation: both are written by the
    // neighbouring stripes, and one IPC handle then covers both
    s->ev_slots = 9 * K + 1;
    const size_t ev_bytes = (is_stripe && cfg->module == WDPM_DRAIN) ? event_area_bytes(2 * (cfg->cols + 2), s->ev_slots, s->esize) : 0;
    if ((e = cudaMalloc((void**)&s->flags, kFlagsBytes + ev_bytes)) != cudaSuccess) return cleanup(WDPM_E_NOMEM, cudaGetErrorString(e));
    s->device_bytes += (long long)(kFlagsBytes + ev_bytes);
    if (ev_bytes) s->events = reinterpret_cast<char*>(s->flags) + kFlagsBytes;
    if ((e = cudaMalloc((void**)&s->partials, sizeof(BlockPartial) * s->reduce_blocks)) != cudaSuccess ||
        (e = cudaMalloc((void**)&s->d_cta_outlets, (size_t)s->n_strips * s->n_chunks)) != cudaSuccess ||
        (e = cudaMalloc((void**)&s->d_total, sizeof(double))) != cudaSuccess ||
        (e = cudaMalloc((void**)&s->d_bad, sizeof(int))) != cudaSuccess ||
        (e = cudaMalloc((void**)&s->d_result, sizeof(BlockPartial))) != cudaSuccess ||
        (e = cudaMalloc((void**)&s->outlet_partials, sizeof(OutletCand) * s->reduce_blocks)) != cudaSuccess ||
        (e = cudaMalloc((void**)&s->d_outlet, sizeof(OutletCand))) != cudaSuccess ||
        (e = cudaMalloc((void**)&s->d_dirty, sizeof(int))) != cudaSuccess ||
        (e = cudaHostAlloc((void**)&s->h_result, sizeof(BlockPartial), cudaHostAllocDefault)) != cudaSuccess ||
        (e = cudaHostAlloc((void**)&s->h_halo_error, sizeof(int), cudaHostAllocDefault)) != cudaSuccess)
        return cleanup(WDPM_E_NOMEM, std::string("cudaMalloc scratch: ") + cudaGetErrorString(e));
    if ((e = cudaStreamCreateWithFlags(&s->own_stream, cudaStreamNonBlocking)) != cudaSuccess)
        return cleanup(WDPM_E_CUDA, cudaGetErrorString(e));
    s->stream = s->own_stream;
    for (auto& evn : s->ev)
        if ((e = cudaEventCreate(&evn)) != cudaSuccess) return cleanup(WDPM_E_CUDA, cudaGetErrorString(e));

    if ((e = cudaMemsetAsync(s->w[0], 0, grid_bytes, s->stream)) != cudaSuccess ||
        (e = cudaMemsetAsync(s->w[1], 0, grid_bytes, s->stream)) != cudaSuccess ||
        (e = cudaMemsetAsync(s->oldw, 0, grid_bytes, s->stream)) != cudaSuccess ||
        (e = cudaMemsetAsync(s->d_cta_outlets, 0, (size_t)s->n_strips * s->n_chunks, s->stream)) != cudaSuccess ||
        (e = cudaMemsetAsync(s->flags, 0, kFlagsBytes + ev_bytes, s->stream)) != cudaSuccess)
        return cleanup(WDPM_E_CUDA, cudaGetErrorString(e));
    int rc = alloc_outlets(s, 1);  // the single total exists before any set is installed
    if (rc) { wdpm_destroy(s); return rc; }
    rc = s->dtype == WDPM_F64 ? fill_dem<double>(s) : fill_dem<float>(s);
    if (rc) { wdpm_destroy(s); return rc; }
    if ((e = cudaStreamSynchronize(s->stream)) != cudaSuccess) return cleanup(WDPM_E_CUDA, cudaGetErrorString(e));
    *out = s;
    return WDPM_OK;
}

int wdpm_destroy(wdpm_solver* s) {
    if (!s) return WDPM_OK;
    cudaSetDevice(s->device);
    if (s->stream) cudaStreamSynchronize(s->stream);
    if (s->ck_done) cudaEventSynchronize(s->ck_done);  // a capture may still be copying out of oldw
    if (s->ck_water) cudaFreeHost(s->ck_water);
    if (s->ck_totals) cudaFreeHost(s->ck_totals);
    if (s->d_ck_totals) cudaFree(s->d_ck_totals);
    if (s->ck_ready) cudaEventDestroy(s->ck_ready);
    if (s->ck_done) cudaEventDestroy(s->ck_done);
    if (s->ck_stream) cudaStreamDestroy(s->ck_stream);
    for (auto* peer : {&s->above, &s->below})
        if (peer->present && peer->ipc) {
            cudaIpcCloseMemHandle(peer->w[0]);
            cudaIpcCloseMemHandle(peer->w[1]);
            cudaIpcCloseMemHandle(peer->flags);
        }
    if (s->flags) cudaFree(s->flags);
    void* ptrs[] = {s->dem, s->w[0], s->w[1], s->oldw, s->totaldrain, s->ev_area, s->saved_elev, s->d_outlet_rc, s->d_outlet_pos, s->d_cta_outlets,
                    s->d_total, s->d_bad, s->partials, s->d_result, s->outlet_partials, s->d_outlet, s->d_dirty};
    for (void* p : ptrs)
        if (p) cudaFree(p);
    if (s->h_result) cudaFreeHost(s->h_result);
    if (s->h_halo_error) cudaFreeHost(s->h_halo_error);
    for (auto& evn : s->ev)
        if (evn) cudaEventDestroy(evn);
    if (s->own_stream) cudaStreamDestroy(s->own_stream);
    cudaGetLastError();
    delete s;
    return WDPM_OK;
}

int wdpm_set_stream(wdpm_solver* s, void* cuda_stream) {
    if (!s) return fail(WDPM_E_ARG, "null solver");
    CUDA_TRY(cudaSetDevice(s->device));
    CUDA_TRY(cudaStreamSynchronize(s->stream));
    s->stream = cuda_stream ? static_cast<cudaStream_t>(cuda_stream) : s->own_stream;
    return WDPM_OK;
}

int wdpm_synchronize(wdpm_solver* s) {
    if (!s) return fail(WDPM_E_ARG, "null solver");
    CUDA_TRY(cudaSetDevice(s->device));
    CUDA_TRY(cudaStreamSynchronize(s->stream));
    return WDPM_OK;
}

int wdpm_upload(wdpm_solver* s, const void* dem, const void* water) {
    if (!s || !dem) return fail(WDPM_E_ARG, "null argument");
    if (s->stripe) return fail(WDPM_E_STATE, "stripe solvers upload with wdpm_stripe_upload");
    CUDA_TRY(cudaSetDevice(s->device));
    int rc = upload_grid(s, s->dem, dem);
    if (rc) return rc;
    {   // store elevations masked: dem <= nodata -> sentinel (relax.cuh)
        const long long n = s->g.cells_dev();
        const int grid = grid_for(n, 256, s->sm_count);
        if (s->dtype == WDPM_F64) k_mask_dem<double><<<grid, 256, 0, s->stream>>>(static_cast<double*>(s->dem), n, s->cfg.nodata);
        else k_mask_dem<float><<<grid, 256, 0, s->stream>>>(static_cast<float*>(s->dem), n, (float)s->cfg.nodata);
        s->launches++;
        CUDA_TRY(cudaGetLastError());
    }
    s->have_dem = true;
    s->marks_applied = false;  // the upload replaced the marked cells
    rc = apply_outlet_marks(s, true);
    if (rc) return rc;
    return wdpm_upload_water(s, water);
}

int wdpm_upload_water(wdpm_solver* s, const void* water) {
    if (!s) return fail(WDPM_E_ARG, "null solver");
    if (s->stripe) return fail(WDPM_E_STATE, "stripe solvers upload with wdpm_stripe_upload");
    if (!s->have_dem) return fail(WDPM_E_STATE, "upload the DEM first");
    CUDA_TRY(cudaSetDevice(s->device));
    if (water) {
        int rc = upload_grid(s, s->w[s->cur], water);
        if (rc) return rc;
    } else {
        CUDA_TRY(cudaMemsetAsync(s->w[s->cur], 0, (size_t)s->g.cells_dev() * s->esize, s->stream));
    }
    return refresh_water_flags(s);
}

int wdpm_download_water(wdpm_solver* s, void* water) {
    if (!s || !water) return fail(WDPM_E_ARG, "null argument");
    if (!s->have_dem) return fail(WDPM_E_STATE, "nothing uploaded yet");
    CUDA_TRY(cudaSetDevice(s->device));
    int rows = 0;  // a stripe: the owned interior rows only
    const char* src = owned_interior(s, s->w[s->cur], &rows);
    CUDA_TRY(cudaMemcpy2DAsync(water, (size_t)s->g.C * s->esize, src, (size_t)s->g.pitch * s->esize, (size_t)s->g.C * s->esize,
                               (size_t)rows, cudaMemcpyDeviceToHost, s->stream));
    CUDA_TRY(cudaStreamSynchronize(s->stream));
    return WDPM_OK;
}

int wdpm_apply_add(wdpm_solver* s, double depth, double runoff_fraction) {
    if (!s) return fail(WDPM_E_ARG, "null solver");
    if (!s->have_dem) return fail(WDPM_E_STATE, "upload first");
    CUDA_TRY(cudaSetDevice(s->device));
    const long long n = s->g.cells_dev();
    const int grid = grid_for(n, 256, s->sm_count);
    if (s->dtype == WDPM_F64)
        k_apply_add<double><<<grid, 256, 0, s->stream>>>(static_cast<double*>(s->w[s->cur]), static_cast<const double*>(s->dem), n,
                                                         depth, depth * runoff_fraction);
    else
        k_apply_add<float><<<grid, 256, 0, s->stream>>>(static_cast<float*>(s->w[s->cur]), static_cast<const float*>(s->dem), n,
                                                        (float)depth, (float)(depth * runoff_fraction));
    s->water_clean = false;
    s->negzero_free = false;  // depth * runoff_fraction may be -0.0
    s->launches++;
    CUDA_TRY(cudaGetLastError());
    return WDPM_OK;
}

int wdpm_apply_subtract(wdpm_solver* s, double depth) {
    if (!s) return fail(WDPM_E_ARG, "null solver");
    if (!s->have_dem) return fail(WDPM_E_STATE, "upload first");
    CUDA_TRY(cudaSetDevice(s->device));
    const long long n = s->g.cells_dev();
    const int grid = grid_for(n, 256, s->sm_count);
    if (s->dtype == WDPM_F64)
        k_apply_subtract<double><<<grid, 256, 0, s->stream>>>(static_cast<double*>(s->w[s->cur]), static_cast<const double*>(s->dem),
                                                              n, depth);
    else
        k_apply_subtract<float><<<grid, 256, 0, s->stream>>>(static_cast<float*>(s->w[s->cur]), static_cast<const float*>(s->dem), n,
                                                             (float)depth);
    s->water_clean = false;
    s->negzero_free = true;  // every valid cell is now > 0 or +0
    s->launches++;
    CUDA_TRY(cudaGetLastError());
    return WDPM_OK;
}

int wdpm_find_outlet(wdpm_solver* s, int32_t* drainrow, int32_t* draincol, double* min_elevation) {
    if (!s) return fail(WDPM_E_ARG, "null solver");
    if (!s->have_dem) return fail(WDPM_E_STATE, "upload first");
    CUDA_TRY(cudaSetDevice(s->device));
    int rc = apply_outlet_marks(s, false);  // search the true elevations
    if (rc) return rc;
    if (s->dtype == WDPM_F64)
        k_find_outlet_stage1<double, 256><<<s->reduce_blocks, 256, 0, s->stream>>>(static_cast<const double*>(s->dem), s->g, s->outlet_partials);
    else
        k_find_outlet_stage1<float, 256><<<s->reduce_blocks, 256, 0, s->stream>>>(static_cast<const float*>(s->dem), s->g, s->outlet_partials);
    k_find_outlet_stage2<<<1, 32, 0, s->stream>>>(s->outlet_partials, s->reduce_blocks, s->d_outlet);
    s->launches += 2;
    CUDA_TRY(cudaGetLastError());
    OutletCand c;
    CUDA_TRY(cudaMemcpyAsync(&c, s->d_outlet, sizeof(c), cudaMemcpyDeviceToHost, s->stream));
    CUDA_TRY(cudaStreamSynchronize(s->stream));
    if (c.index < 0) { apply_outlet_marks(s, true); return fail(WDPM_E_STATE, "no cell with elevation > 0: no outlet"); }
    const int32_t row = (int32_t)(c.index / (s->g.C + 2)) + s->G, col = (int32_t)(c.index % (s->g.C + 2));
    if (drainrow) *drainrow = row;
    if (draincol) *draincol = col;
    if (min_elevation) *min_elevation = c.elev;
    if (s->module != WDPM_DRAIN) return WDPM_OK;  // a query only; no outlet to install
    return wdpm_set_outlets(s, 1, &row, &col);
}

int wdpm_set_outlet(wdpm_solver* s, int32_t drainrow, int32_t draincol) {
    if (s && s->module != WDPM_DRAIN) return WDPM_OK;  // only Drain kernels look at outlets
    return wdpm_set_outlets(s, 1, &drainrow, &draincol);
}

int wdpm_set_outlets(wdpm_solver* s, int32_t n, const int32_t* rows, const int32_t* cols) {
    if (!s || (n > 0 && (!rows || !cols))) return fail(WDPM_E_ARG, "null argument");
    if (s->module != WDPM_DRAIN) return fail(WDPM_E_STATE, "outlets belong to the Drain module");
    if (n < 1 || n > kMaxOutlets) return fail(WDPM_E_ARG, "number of outlets must be in 1..WDPM_MAX_OUTLETS");
    if (n > 1 && s->schedule == WDPM_SCHEDULE_SERIAL) return fail(WDPM_E_UNSUPPORTED, "the serial schedule has one outlet (the emptying of overlapping outlet neighbourhoods is not defined)");
    if (s->in_block) return fail(WDPM_E_STATE, "a block is open");
    for (int k = 0; k < n; k++)
        if (rows[k] < 1 || rows[k] > s->cfg.rows || cols[k] < 1 || cols[k] > s->g.C) return fail(WDPM_E_ARG, "outlet outside the DEM");
    // sort by (row, col): kernels find an outlet by binary search; order[i] = the caller's index of sorted outlet i
    std::vector<int> order((size_t)n);
    for (int k = 0; k < n; k++) order[k] = k;
    auto key = [&](int k) { return ((long long)rows[k] << 32) | (long long)cols[k]; };
    std::sort(order.begin(), order.end(), [&](int a, int b) { return key(a) < key(b); });
    for (int i = 1; i < n; i++)
        if (key(order[i]) == key(order[i - 1])) return fail(WDPM_E_ARG, "duplicate outlet");
    CUDA_TRY(cudaSetDevice(s->device));
    int rc = apply_outlet_marks(s, false);  // restore the cells of the previous set
    if (rc) return rc;
    rc = alloc_outlets(s, n);
    if (rc) { s->n_outlets = 0; s->have_outlet = false; return rc; }
    s->outlet_rc.resize((size_t)2 * n);
    s->outlet_pos.resize((size_t)n);
    for (int i = 0; i < n; i++) {
        s->outlet_rc[2 * i] = rows[order[i]] - s->G;  // kernels work in the stripe's local rows (may lie outside the stripe)
        s->outlet_rc[2 * i + 1] = cols[order[i]];
        s->outlet_pos[order[i]] = i;
    }
    s->n_outlets = n;
    s->have_outlet = true;
    CUDA_TRY(cudaMemcpyAsync(s->d_outlet_rc, s->outlet_rc.data(), sizeof(int) * 2 * n, cudaMemcpyHostToDevice, s->stream));
    CUDA_TRY(cudaMemcpyAsync(s->d_outlet_pos, s->outlet_pos.data(), sizeof(int) * n, cudaMemcpyHostToDevice, s->stream));
    CUDA_TRY(cudaMemsetAsync(s->ev_area, 0, event_area_bytes(n, s->ev_slots, s->esize), s->stream));
    if (s->events) CUDA_TRY(cudaMemsetAsync(s->events, 0, event_area_bytes(border_entries(s), s->ev_slots, s->esize), s->stream));
    rc = s->dtype == WDPM_F64 ? compute_cta_outlets<double>(s) : compute_cta_outlets<float>(s);
    if (rc) return rc;
    return s->have_dem ? apply_outlet_marks(s, true) : WDPM_OK;
}

int wdpm_set_total_drain(wdpm_solver* s, double value) {
    if (!s) return fail(WDPM_E_ARG, "null solver");
    CUDA_TRY(cudaSetDevice(s->device));
    double v64 = value;
    float v32 = (float)value;
    const size_t first = s->n_outlets > 0 ? (size_t)s->outlet_pos[0] : 0;  // the value goes to the first outlet's total
    CUDA_TRY(cudaMemsetAsync(s->totaldrain, 0, s->esize * s->outlet_cap, s->stream));
    CUDA_TRY(cudaMemcpyAsync(static_cast<char*>(s->totaldrain) + first * s->esize, s->dtype == WDPM_F64 ? (void*)&v64 : (void*)&v32, s->esize,
                             cudaMemcpyHostToDevice, s->stream));
    CUDA_TRY(cudaStreamSynchronize(s->stream));
    return WDPM_OK;
}

int wdpm_seed_outlet_drains(wdpm_solver* s) {
    if (!s) return fail(WDPM_E_ARG, "null solver");
    if (!s->have_dem) return fail(WDPM_E_STATE, "upload first");
    if (!s->have_outlet) return fail(WDPM_E_STATE, "no outlet installed");
    if (s->in_block) return fail(WDPM_E_STATE, "a block is open");
    CUDA_TRY(cudaSetDevice(s->device));
    const int blocks = (s->n_outlets + 255) / 256;
    if (s->dtype == WDPM_F64) k_seed_outlets<double><<<blocks, 256, 0, s->stream>>>(static_cast<const double*>(s->w[s->cur]), s->g, drain_state<double>(s));
    else k_seed_outlets<float><<<blocks, 256, 0, s->stream>>>(static_cast<const float*>(s->w[s->cur]), s->g, drain_state<float>(s));
    s->launches++;
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaStreamSynchronize(s->stream));
    return WDPM_OK;
}

int wdpm_get_outlet_drains(wdpm_solver* s, double* values, int32_t n) {
    if (!s || !values) return fail(WDPM_E_ARG, "null argument");
    if (n < 1 || n > s->outlet_cap) return fail(WDPM_E_ARG, "n out of range (at most the installed set's size)");
    CUDA_TRY(cudaSetDevice(s->device));
    const size_t m = (size_t)s->outlet_cap;
    std::vector<double> v64(s->dtype == WDPM_F64 ? m : 0);
    std::vector<float> v32(s->dtype == WDPM_F64 ? 0 : m);
    CUDA_TRY(cudaMemcpyAsync(s->dtype == WDPM_F64 ? (void*)v64.data() : (void*)v32.data(), s->totaldrain, s->esize * m, cudaMemcpyDeviceToHost, s->stream));
    CUDA_TRY(cudaStreamSynchronize(s->stream));
    for (int k = 0; k < n; k++) {  // back to the caller's order
        const size_t i = s->n_outlets > 0 ? (size_t)s->outlet_pos[k] : (size_t)k;
        values[k] = s->dtype == WDPM_F64 ? v64[i] : (double)v32[i];
    }
    return WDPM_OK;
}

int wdpm_get_total_drain(wdpm_solver* s, double* value) {
    if (!s || !value) return fail(WDPM_E_ARG, "null argument");
    CUDA_TRY(cudaSetDevice(s->device));
    if (s->dtype == WDPM_F64) k_sum_totals<double><<<1, 32, 0, s->stream>>>(static_cast<const double*>(s->totaldrain), s->d_outlet_pos, std::max(s->n_outlets, 1), s->d_total);
    else k_sum_totals<float><<<1, 32, 0, s->stream>>>(static_cast<const float*>(s->totaldrain), s->d_outlet_pos, std::max(s->n_outlets, 1), s->d_total);
    s->launches++;
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaMemcpyAsync(value, s->d_total, sizeof(double), cudaMemcpyDeviceToHost, s->stream));
    CUDA_TRY(cudaStreamSynchronize(s->stream));
    return WDPM_OK;
}

int wdpm_set_outlet_drains(wdpm_solver* s, const double* values, int32_t n) {
    if (!s || !values) return fail(WDPM_E_ARG, "null argument");
    if (s->module != WDPM_DRAIN) return fail(WDPM_E_STATE, "outlet totals belong to the Drain module");
    if (s->in_block) return fail(WDPM_E_STATE, "a block is open");
    if (n != std::max(s->n_outlets, 1)) return fail(WDPM_E_ARG, "n must be the installed outlet set's size");
    CUDA_TRY(cudaSetDevice(s->device));
    // sorted order; as wdpm_seed_outlet_drains: a total is kept by the solver that owns its outlet's row, 0 elsewhere
    std::vector<double> v64(s->dtype == WDPM_F64 ? (size_t)s->outlet_cap : 0, 0.0);
    std::vector<float> v32(s->dtype == WDPM_F64 ? 0 : (size_t)s->outlet_cap, 0.0f);
    for (int k = 0; k < n; k++) {
        const size_t i = s->n_outlets > 0 ? (size_t)s->outlet_pos[k] : 0;
        const bool owned = s->n_outlets == 0 || (s->outlet_rc[2 * i] >= 0 && s->outlet_rc[2 * i] < s->P);
        if (s->dtype == WDPM_F64) v64[i] = owned ? values[k] : 0.0;
        else v32[i] = owned ? (float)values[k] : 0.0f;
    }
    CUDA_TRY(cudaMemcpyAsync(s->totaldrain, s->dtype == WDPM_F64 ? (const void*)v64.data() : (const void*)v32.data(), s->esize * s->outlet_cap,
                             cudaMemcpyHostToDevice, s->stream));
    CUDA_TRY(cudaStreamSynchronize(s->stream));
    return WDPM_OK;
}

int wdpm_checkpoint_arm(wdpm_solver* s) {
    if (!s) return fail(WDPM_E_ARG, "null solver");
    if (!s->have_dem) return fail(WDPM_E_STATE, "upload first");
    if (s->in_block) return fail(WDPM_E_STATE, "a block is open: arm before wdpm_block_begin");
    CUDA_TRY(cudaSetDevice(s->device));
    if (!s->ck_stream) CUDA_TRY(cudaStreamCreateWithFlags(&s->ck_stream, cudaStreamNonBlocking));
    if (!s->ck_ready) CUDA_TRY(cudaEventCreateWithFlags(&s->ck_ready, cudaEventDisableTiming));
    if (!s->ck_done) CUDA_TRY(cudaEventCreateWithFlags(&s->ck_done, cudaEventDisableTiming));
    if (!s->ck_water) {
        int rows = 0;
        owned_interior(s, s->oldw, &rows);
        CUDA_TRY(cudaHostAlloc(&s->ck_water, (size_t)rows * s->g.C * s->esize, cudaHostAllocDefault));
    }
    s->ck_armed = true;
    s->ck_captured = false;
    return WDPM_OK;
}

int wdpm_checkpoint_wait(wdpm_solver* s, const void** water, const double** totals, int32_t* n) {
    if (!s) return fail(WDPM_E_ARG, "null solver");
    if (!s->ck_captured)
        return fail(WDPM_E_STATE, s->ck_armed ? "the armed capture is taken by the next wdpm_block_begin" : "no checkpoint capture armed");
    CUDA_TRY(cudaSetDevice(s->device));
    CUDA_TRY(cudaEventSynchronize(s->ck_done));
    if (water) *water = s->ck_water;
    if (totals) *totals = s->ck_totals;
    if (n) *n = s->ck_n;
    return WDPM_OK;
}

int wdpm_quantize_water(wdpm_solver* s) {
    if (!s) return fail(WDPM_E_ARG, "null solver");
    if (!s->have_dem) return fail(WDPM_E_STATE, "upload first");
    if (s->in_block) return fail(WDPM_E_STATE, "a block is open");
    CUDA_TRY(cudaSetDevice(s->device));
    const long long n = s->g.cells_dev();
    const int grid = grid_for(n, 256, s->sm_count);
    if (s->dtype == WDPM_F64) k_quantize_water<double><<<grid, 256, 0, s->stream>>>(static_cast<double*>(s->w[s->cur]), static_cast<const double*>(s->dem), n);
    else k_quantize_water<float><<<grid, 256, 0, s->stream>>>(static_cast<float*>(s->w[s->cur]), static_cast<const float*>(s->dem), n);
    s->launches++;
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaStreamSynchronize(s->stream));
    s->water_clean = false;
    s->negzero_free = false;  // a tiny negative value quantises to -0.0
    return WDPM_OK;
}

int wdpm_copy_state(wdpm_solver* dst, wdpm_solver* src, int32_t what) {
    if (!dst || !src) return fail(WDPM_E_ARG, "null solver");
    if (dst == src || !(what & (WDPM_COPY_DEM | WDPM_COPY_WATER))) return fail(WDPM_E_ARG, "nothing to copy");
    if (dst->stripe || src->stripe) return fail(WDPM_E_UNSUPPORTED, "stripe solvers take their grids from the host");
    if (dst->device != src->device || dst->dtype != src->dtype || dst->cfg.rows != src->cfg.rows || dst->g.C != src->g.C)
        return fail(WDPM_E_ARG, "solvers differ in device, precision or grid size");
    if (!src->have_dem) return fail(WDPM_E_STATE, "the source solver holds no grids");
    if (!(what & WDPM_COPY_DEM) && !dst->have_dem) return fail(WDPM_E_STATE, "the destination needs elevations first");
    if (dst->in_block || src->in_block) return fail(WDPM_E_STATE, "a block is open");
    CUDA_TRY(cudaSetDevice(dst->device));
    // the padded grid (halo ring included) sits at the same offset in both layouts; the pitches may differ
    const size_t off_d = ((size_t)kPadTop * dst->g.pitch + kPadLeft) * dst->esize, off_s = ((size_t)kPadTop * src->g.pitch + kPadLeft) * src->esize;
    const size_t width = (size_t)(src->g.C + 2) * src->esize, height = (size_t)(src->g.R + 2);
    if (what & WDPM_COPY_DEM) {
        int rc = apply_outlet_marks(src, false);  // the true elevations travel, not the source's outlet marks
        if (rc) return rc;
        CUDA_TRY(cudaStreamSynchronize(src->stream));
        CUDA_TRY(cudaMemcpy2DAsync(static_cast<char*>(dst->dem) + off_d, (size_t)dst->g.pitch * dst->esize, static_cast<const char*>(src->dem) + off_s,
                                   (size_t)src->g.pitch * src->esize, width, height, cudaMemcpyDeviceToDevice, dst->stream));
        CUDA_TRY(cudaStreamSynchronize(dst->stream));
        rc = apply_outlet_marks(src, true);
        if (rc) return rc;
        dst->have_dem = true;
        dst->marks_applied = false;
        rc = apply_outlet_marks(dst, true);
        if (rc) return rc;
    }
    if (what & WDPM_COPY_WATER) {
        CUDA_TRY(cudaStreamSynchronize(src->stream));
        CUDA_TRY(cudaMemcpy2DAsync(static_cast<char*>(dst->w[dst->cur]) + off_d, (size_t)dst->g.pitch * dst->esize,
                                   static_cast<const char*>(src->w[src->cur]) + off_s, (size_t)src->g.pitch * src->esize, width, height,
                                   cudaMemcpyDeviceToDevice, dst->stream));
    }
    CUDA_TRY(cudaStreamSynchronize(dst->stream));
    CUDA_TRY(cudaStreamSynchronize(src->stream));
    return refresh_water_flags(dst);  // a new DEM changes which cells are invalid, new water what they hold
}

int wdpm_get_cell_water(wdpm_solver* s, int32_t row, int32_t col, double* value) {
    if (!s || !value) return fail(WDPM_E_ARG, "null argument");
    row -= s->G;
    if (row < 0 || row > s->g.R + 1 || col < 0 || col > s->g.C + 1) return fail(WDPM_E_ARG, "cell outside this solver's padded rows");
    CUDA_TRY(cudaSetDevice(s->device));
    const size_t off = ((size_t)(row + kPadTop) * s->g.pitch + (size_t)(col + kPadLeft)) * s->esize;
    double v64 = 0;
    float v32 = 0;
    CUDA_TRY(cudaMemcpyAsync(s->dtype == WDPM_F64 ? (void*)&v64 : (void*)&v32, static_cast<char*>(s->w[s->cur]) + off, s->esize,
                             cudaMemcpyDeviceToHost, s->stream));
    CUDA_TRY(cudaStreamSynchronize(s->stream));
    *value = s->dtype == WDPM_F64 ? v64 : (double)v32;
    return WDPM_OK;
}

int wdpm_final_statistics(wdpm_solver* s, int64_t* valid_cells, int64_t* wet_above_1mm, double* max_depth) {
    if (!s) return fail(WDPM_E_ARG, "null solver");
    if (!s->have_dem) return fail(WDPM_E_STATE, "nothing uploaded yet");
    if (s->in_block) return fail(WDPM_E_STATE, "a block is open");
    CUDA_TRY(cudaSetDevice(s->device));
    const int lo = s->stripe ? std::max(s->G, 1) - s->G : 1;
    const int hi = s->stripe ? std::min(s->G + s->P, s->cfg.rows + 1) - s->G : s->g.R + 1;
    FinalStats* d_st = reinterpret_cast<FinalStats*>(s->partials);  // scratch, free between blocks
    FinalStats init{0ull, 0ull, 0.0};
    const long long lowest = (long long)0x8000000000000000ull;  // image of the most negative double: below every depth
    std::memcpy(&init.max_depth, &lowest, sizeof(lowest));
    CUDA_TRY(cudaMemcpyAsync(d_st, &init, sizeof(init), cudaMemcpyHostToDevice, s->stream));
    const int grid = std::max(1, std::min(hi - lo, s->sm_count * 8));
    if (s->dtype == WDPM_F64)
        k_final_stats<double><<<grid, 256, 0, s->stream>>>(static_cast<const double*>(s->w[s->cur]), static_cast<const double*>(s->dem), s->g, lo, hi - lo, d_st);
    else
        k_final_stats<float><<<grid, 256, 0, s->stream>>>(static_cast<const float*>(s->w[s->cur]), static_cast<const float*>(s->dem), s->g, lo, hi - lo, d_st);
    s->launches++;
    CUDA_TRY(cudaGetLastError());
    FinalStats out;
    CUDA_TRY(cudaMemcpyAsync(&out, d_st, sizeof(out), cudaMemcpyDeviceToHost, s->stream));
    CUDA_TRY(cudaStreamSynchronize(s->stream));
    long long bits;
    std::memcpy(&bits, &out.max_depth, sizeof(bits));
    bits = bits >= 0 ? bits : (long long)(0x8000000000000000ull - (unsigned long long)bits);  // the image is its own inverse
    double md;
    std::memcpy(&md, &bits, sizeof(md));
    if (valid_cells) *valid_cells = (int64_t)out.valid_cells;
    if (wet_above_1mm) *wet_above_1mm = (int64_t)out.wet_above_1mm;
    if (max_depth) *max_depth = out.valid_cells ? md : 0.0;
    return WDPM_OK;
}

int wdpm_water_checksum(wdpm_solver* s, uint64_t* checksum) {
    if (!s || !checksum) return fail(WDPM_E_ARG, "null argument");
    if (!s->have_dem) return fail(WDPM_E_STATE, "nothing uploaded yet");
    CUDA_TRY(cudaSetDevice(s->device));
    // owned interior rows in local padded coordinates (a stripe's first/last padded row may be the DEM's halo ring)
    const int lo = s->stripe ? std::max(s->G, 1) - s->G : 1;
    const int hi = s->stripe ? std::min(s->G + s->P, s->cfg.rows + 1) - s->G : s->g.R + 1;
    unsigned long long* d_sum = reinterpret_cast<unsigned long long*>(s->partials);  // scratch, free between blocks
    if (s->in_block) return fail(WDPM_E_STATE, "a block is open");
    CUDA_TRY(cudaMemsetAsync(d_sum, 0, sizeof(unsigned long long), s->stream));
    const int grid = std::max(1, std::min(hi - lo, s->sm_count * 8));
    if (s->dtype == WDPM_F64)
        k_water_checksum<double><<<grid, 256, 0, s->stream>>>(static_cast<const double*>(s->w[s->cur]), s->g, lo, hi - lo, s->G, s->cfg.cols, d_sum);
    else
        k_water_checksum<float><<<grid, 256, 0, s->stream>>>(static_cast<const float*>(s->w[s->cur]), s->g, lo, hi - lo, s->G, s->cfg.cols, d_sum);
    s->launches++;
    CUDA_TRY(cudaGetLastError());
    unsigned long long v = 0;
    CUDA_TRY(cudaMemcpyAsync(&v, d_sum, sizeof(v), cudaMemcpyDeviceToHost, s->stream));
    CUDA_TRY(cudaStreamSynchronize(s->stream));
    *checksum = (uint64_t)v;
    return WDPM_OK;
}

int wdpm_run_block(wdpm_solver* s, int32_t n_iters, wdpm_block_result* out) {
    if (!s) return fail(WDPM_E_ARG, "null solver");
    if (s->halo_failed) return fail(WDPM_E_HALO, "an earlier halo wait timed out: upload again");
    if (n_iters < 0) return fail(WDPM_E_ARG, "negative iteration count");
    if (!s->have_dem) return fail(WDPM_E_STATE, "upload first");
    if (s->module == WDPM_DRAIN && !s->have_outlet) return fail(WDPM_E_STATE, "Drain needs an outlet: call wdpm_find_outlet or wdpm_set_outlet");
    CUDA_TRY(cudaSetDevice(s->device));
    return s->dtype == WDPM_F64 ? run_block_t<double>(s, n_iters, out) : run_block_t<float>(s, n_iters, out);
}

int wdpm_block_begin(wdpm_solver* s) {
    if (!s) return fail(WDPM_E_ARG, "null solver");
    if (s->halo_failed) return fail(WDPM_E_HALO, "an earlier halo wait timed out: upload again");
    if (!s->have_dem) return fail(WDPM_E_STATE, "upload first");
    if (s->in_block) return fail(WDPM_E_STATE, "a block is already open");
    if (s->module == WDPM_DRAIN && !s->have_outlet) return fail(WDPM_E_STATE, "Drain needs an outlet: call wdpm_find_outlet or wdpm_set_outlet");
    CUDA_TRY(cudaSetDevice(s->device));
    return s->dtype == WDPM_F64 ? block_begin_t<double>(s) : block_begin_t<float>(s);
}

int wdpm_block_enqueue(wdpm_solver* s, int32_t n_iters) {
    if (!s) return fail(WDPM_E_ARG, "null solver");
    if (!s->in_block) return fail(WDPM_E_STATE, "no open block: call wdpm_block_begin");
    if (n_iters < 0) return fail(WDPM_E_ARG, "negative iteration count");
    CUDA_TRY(cudaSetDevice(s->device));
    const int rc = iterate(s, n_iters);
    if (rc == WDPM_OK) s->blk_iters += n_iters;
    return rc;
}

int wdpm_block_end(wdpm_solver* s, wdpm_block_result* out) {
    if (!s) return fail(WDPM_E_ARG, "null solver");
    if (!s->in_block) return fail(WDPM_E_STATE, "no open block: call wdpm_block_begin");
    CUDA_TRY(cudaSetDevice(s->device));
    return s->dtype == WDPM_F64 ? block_end_t<double>(s, out) : block_end_t<float>(s, out);
}

int wdpm_iterate(wdpm_solver* s, int32_t n_iters) {
    if (!s) return fail(WDPM_E_ARG, "null solver");
    if (s->halo_failed) return fail(WDPM_E_HALO, "an earlier halo wait timed out: upload again");
    if (n_iters < 0) return fail(WDPM_E_ARG, "negative iteration count");
    if (!s->have_dem) return fail(WDPM_E_STATE, "upload first");
    if (s->module == WDPM_DRAIN && !s->have_outlet) return fail(WDPM_E_STATE, "Drain needs an outlet");
    CUDA_TRY(cudaSetDevice(s->device));
    return iterate(s, n_iters);
}

int wdpm_subpass(wdpm_solver* s, int32_t oi, int32_t oj) {
    if (!s) return fail(WDPM_E_ARG, "null solver");
    if (oi < 1 || oi > 3 || oj < 1 || oj > 3) return fail(WDPM_E_ARG, "oi and oj must be 1..3");
    if (!s->have_dem) return fail(WDPM_E_STATE, "upload first");
    CUDA_TRY(cudaSetDevice(s->device));
    return s->dtype == WDPM_F64 ? colour_subpass<double>(s, oi, oj) : colour_subpass<float>(s, oi, oj);
}

int wdpm_get_info(wdpm_solver* s, wdpm_info* info) {
    if (!s || !info) return fail(WDPM_E_ARG, "null argument");
    std::memset(info, 0, sizeof(*info));
    info->device_bytes = s->device_bytes;
    info->kernel_launches = s->launches;
    info->kernel = s->kernel;
    info->sm_count = s->sm_count;
    int W, TWV, K, nt; size_t smem; bool wa;
    if (s->dtype == WDPM_F64) { const auto& v = fused_variants<double>()[s->variant]; W = v.W; TWV = v.TWV; K = v.K; nt = v.nthreads; smem = v.smem; wa = v.wa; }
    else { const auto& v = fused_variants<float>()[s->variant]; W = v.W; TWV = v.TWV; K = v.K; nt = v.nthreads; smem = v.smem; wa = v.wa; }
    info->warp_autonomous = (s->kernel == WDPM_KERNEL_FUSED && wa) ? 1 : 0;
    info->strip_cols = TWV;
    info->window_cols = W;
    info->chunk_rows = 3 * s->chunk_triples;
    info->grid_ctas = s->n_strips * s->n_chunks;
    info->cta_threads = nt;
    info->smem_bytes = (int32_t)smem;
    info->iters_per_launch = s->kernel == WDPM_KERNEL_FUSED ? K : 1;
    if (s->kernel == WDPM_KERNEL_RESIDENT) {  // the resident kernel's tiling instead
        info->strip_cols = s->res_TC;
        info->window_cols = s->res_TC + kResHaloLeft + kResHaloRight;
        info->chunk_rows = s->res_TR;
        info->grid_ctas = s->res_ntx * s->res_nty;
        info->cta_threads = kResidentThreads;
        info->smem_bytes = (int32_t)s->res_smem;
        info->iters_per_launch = 0;  // a whole block of iterations per launch
    }
    return WDPM_OK;
}

int wdpm_stripe_band(wdpm_solver* s, int32_t* band_row0, int32_t* band_rows, int32_t* owned_row0, int32_t* owned_rows) {
    if (!s) return fail(WDPM_E_ARG, "null solver");
    if (!s->stripe) return fail(WDPM_E_STATE, "not a stripe solver");
    const int R = s->cfg.rows;
    // padded rows -> interior (0-based) rows: interior = padded - 1, clipped to [1, R]
    const int blo = std::max(s->G - kHaloAbove, 1), bhi = std::min(s->G + s->P + kHaloBelow, R + 1);
    const int olo = std::max(s->G, 1), ohi = std::min(s->G + s->P, R + 1);
    if (band_row0) *band_row0 = blo - 1;
    if (band_rows) *band_rows = bhi - blo;
    if (owned_row0) *owned_row0 = olo - 1;
    if (owned_rows) *owned_rows = ohi - olo;
    return WDPM_OK;
}

int wdpm_stripe_upload(wdpm_solver* s, const void* dem_band, const void* water_band, int32_t band_row0, int32_t band_rows) {
    if (!s || !dem_band) return fail(WDPM_E_ARG, "null argument");
    if (!s->stripe) return fail(WDPM_E_STATE, "not a stripe solver");
    int32_t b0, bn;
    wdpm_stripe_band(s, &b0, &bn, nullptr, nullptr);
    if (band_row0 != b0 || band_rows != bn) return fail(WDPM_E_ARG, "band must be exactly the rows wdpm_stripe_band reports");
    CUDA_TRY(cudaSetDevice(s->device));
    const size_t grid_bytes = (size_t)s->g.cells_dev() * s->esize;
    const int local0 = band_row0 + 1 - s->G;  // local padded row of the band's first row (>= -kHaloAbove)
    const size_t off = ((size_t)(local0 + kPadTop) * s->g.pitch + (size_t)(1 + kPadLeft)) * s->esize;
    int rc = s->dtype == WDPM_F64 ? fill_dem<double>(s) : fill_dem<float>(s);
    if (rc) return rc;
    CUDA_TRY(cudaMemcpy2DAsync(static_cast<char*>(s->dem) + off, (size_t)s->g.pitch * s->esize, dem_band, (size_t)s->g.C * s->esize,
                               (size_t)s->g.C * s->esize, (size_t)band_rows, cudaMemcpyHostToDevice, s->stream));
    {
        const long long n = s->g.cells_dev();
        const int grid = grid_for(n, 256, s->sm_count);
        if (s->dtype == WDPM_F64) k_mask_dem<double><<<grid, 256, 0, s->stream>>>(static_cast<double*>(s->dem), n, s->cfg.nodata);
        else k_mask_dem<float><<<grid, 256, 0, s->stream>>>(static_cast<float*>(s->dem), n, (float)s->cfg.nodata);
        s->launches++;
        CUDA_TRY(cudaGetLastError());
    }
    CUDA_TRY(cudaMemsetAsync(s->w[0], 0, grid_bytes, s->stream));
    CUDA_TRY(cudaMemsetAsync(s->w[1], 0, grid_bytes, s->stream));
    s->cur = 0;  // neighbours must agree on which buffer is current
    if (water_band)
        CUDA_TRY(cudaMemcpy2DAsync(static_cast<char*>(s->w[s->cur]) + off, (size_t)s->g.pitch * s->esize, water_band,
                                   (size_t)s->g.C * s->esize, (size_t)s->g.C * s->esize, (size_t)band_rows, cudaMemcpyHostToDevice,
                                   s->stream));
    CUDA_TRY(cudaMemsetAsync(s->flags, 0, sizeof(HaloFlags), s->stream));
    s->epoch = 0;
    s->launch_slot = 0;  // neighbours must agree on the event buffer rotation as well
    CUDA_TRY(cudaMemsetAsync(s->ev_area, 0, event_area_bytes(s->outlet_cap, s->ev_slots, s->esize), s->stream));
    if (s->events) CUDA_TRY(cudaMemsetAsync(s->events, 0, event_area_bytes(border_entries(s), s->ev_slots, s->esize), s->stream));
    s->halo_failed = false;
    *s->h_halo_error = 0;
    s->have_dem = true;
    s->marks_applied = false;  // the upload replaced the marked cells
    {
        const int rc = apply_outlet_marks(s, true);
        if (rc) return rc;
    }
    return refresh_water_flags(s);
}

int wdpm_stripe_export(wdpm_solver* s, wdpm_stripe_endpoint* self) {
    if (!s || !self) return fail(WDPM_E_ARG, "null argument");
    if (!s->stripe) return fail(WDPM_E_STATE, "not a stripe solver");
    CUDA_TRY(cudaSetDevice(s->device));
    std::memset(self, 0, sizeof(*self));
    static_assert(sizeof(cudaIpcMemHandle_t) == WDPM_IPC_HANDLE_BYTES, "IPC handle size");
    CUDA_TRY(cudaIpcGetMemHandle(reinterpret_cast<cudaIpcMemHandle_t*>(self->water_a), s->w[0]));
    CUDA_TRY(cudaIpcGetMemHandle(reinterpret_cast<cudaIpcMemHandle_t*>(self->water_b), s->w[1]));
    CUDA_TRY(cudaIpcGetMemHandle(reinterpret_cast<cudaIpcMemHandle_t*>(self->flags), s->flags));
    self->device = s->device;
    self->stripe_row0 = s->G;
    self->stripe_rows = s->P;
    self->pitch = s->g.pitch;
    self->pid = (int64_t)getpid();
    self->local_ptr = (uint64_t)(uintptr_t)s;
    return WDPM_OK;
}

static int connect_side(wdpm_solver* s, wdpm_solver::Peer& peer, const wdpm_stripe_endpoint* ep, bool is_above) {
    peer = wdpm_solver::Peer();
    if (!ep) return WDPM_OK;
    if (ep->pitch != s->g.pitch) return fail(WDPM_E_ARG, "neighbour stripe has a different row pitch (cols / variant mismatch)");
    if (is_above ? (ep->stripe_row0 + ep->stripe_rows != s->G) : (s->G + s->P != ep->stripe_row0))
        return fail(WDPM_E_ARG, "neighbour stripe is not adjacent");
    peer.P = ep->stripe_rows;
    if (ep->pid == (int64_t)getpid()) {
        wdpm_solver* o = reinterpret_cast<wdpm_solver*>((uintptr_t)ep->local_ptr);
        if (o->device != s->device) {
            int can = 0;
            CUDA_TRY(cudaDeviceCanAccessPeer(&can, s->device, o->device));
            if (!can) return fail(WDPM_E_UNSUPPORTED, "no peer access between the stripes' devices");
            cudaError_t e = cudaDeviceEnablePeerAccess(o->device, 0);
            if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) return fail(WDPM_E_CUDA, cudaGetErrorString(e));
            cudaGetLastError();
        }
        peer.w[0] = o->w[0];
        peer.w[1] = o->w[1];
        peer.flags = o->flags;
        peer.events = o->events;
        peer.ipc = false;
    } else {
        cudaIpcMemHandle_t h;
        std::memcpy(&h, ep->water_a, sizeof(h));
        CUDA_TRY(cudaIpcOpenMemHandle(&peer.w[0], h, cudaIpcMemLazyEnablePeerAccess));
        std::memcpy(&h, ep->water_b, sizeof(h));
        CUDA_TRY(cudaIpcOpenMemHandle(&peer.w[1], h, cudaIpcMemLazyEnablePeerAccess));
        std::memcpy(&h, ep->flags, sizeof(h));
        void* f = nullptr;
        CUDA_TRY(cudaIpcOpenMemHandle(&f, h, cudaIpcMemLazyEnablePeerAccess));
        peer.flags = static_cast<HaloFlags*>(f);
        peer.events = static_cast<char*>(f) + kFlagsBytes;
        peer.ipc = true;
    }
    peer.present = true;
    return WDPM_OK;
}

int wdpm_stripe_connect(wdpm_solver* s, const wdpm_stripe_endpoint* above, const wdpm_stripe_endpoint* below) {
    if (!s) return fail(WDPM_E_ARG, "null solver");
    if (!s->stripe) return fail(WDPM_E_STATE, "not a stripe solver");
    CUDA_TRY(cudaSetDevice(s->device));
    int rc = connect_side(s, s->above, above, true);
    if (rc) return rc;
    return connect_side(s, s->below, below, false);
}

int wdpm_stripe_phase(wdpm_solver* s, int32_t phase) {
    if (!s) return fail(WDPM_E_ARG, "null solver");
    if (!s->stripe) return fail(WDPM_E_STATE, "not a stripe solver");
    if (!s->have_dem) return fail(WDPM_E_STATE, "upload first");
    CUDA_TRY(cudaSetDevice(s->device));
    if (phase == 0) return s->dtype == WDPM_F64 ? fused_launch_only<double>(s) : fused_launch_only<float>(s);
    if (phase == 1) return s->dtype == WDPM_F64 ? fold_last_launch<double>(s) : fold_last_launch<float>(s);
    return fail(WDPM_E_ARG, "phase must be 0 or 1");
}

#ifdef WDPM_TEST_HOOKS
int wdpm_debug_counters(int32_t* out4) {
    CUDA_TRY(cudaDeviceSynchronize());
    CUDA_TRY(cudaMemcpyFromSymbol(out4, g_dbg_counters, sizeof(int) * 4));
    return WDPM_OK;
}
#endif

#ifdef WDPM_TIMELINE
// Developer probe (scripts/timeline.py builds a separate library with -DWDPM_TIMELINE).
int wdpm_debug_timeline(int32_t cta, int32_t step0, long long* out, int32_t n) {
    if (out) {
        CUDA_TRY(cudaDeviceSynchronize());
        CUDA_TRY(cudaMemcpyFromSymbol(out, g_timeline, sizeof(long long) * (size_t)n));
        return WDPM_OK;
    }
    CUDA_TRY(cudaMemcpyToSymbol(g_timeline_cta, &cta, sizeof(int)));
    CUDA_TRY(cudaMemcpyToSymbol(g_timeline_step0, &step0, sizeof(int)));
    return WDPM_OK;
}
#endif

}  // extern "C"
