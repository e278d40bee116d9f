"""GPU (-m gpu): the production path as AUTO runs it, and the order-free outputs against exact host values.

* A: AUTO's three size bands (resident kernel, small k_fused tilings, k_fused_wa) x Add / Subtract / Drain x fp64 /
  fp32 through wdpm_run_block with a zero threshold > 0, so that every block after the first runs the clean launch
  (solver.cu, pick_launch); block by block against the oracle.
* B: k_fused_wa's geometry (production variants 17 / 16) on small grids: strip, warp and lane boundaries, heights of
  every residue mod 3, chunkings with a short last chunk, guarded (iterate, threshold 0) and clean (run_block).
* C: water_checksum, final_statistics and find_outlet against values computed exactly on the host.
* D: three in-process row stripes on the production tiling with AUTO chunking, free-running and in lockstep.
* E: one grid of more than 2^31 elements (47 000^2 fp32).

Every test asserts from Solver.info() that it ran the kernel and tiling it claims to cover, so a change of AUTO turns
it red instead of moving it to another path. The pure-numpy references (exact checksum, reduction bound, outlet-set
block) are plain functions here; tests/test_exact_refs_cpu.py checks them on hand-computed grids.
"""
import math

import numpy as np
import pytest

from conftest import random_case

pytestmark = pytest.mark.gpu

NODATA = -99999.0
THRES = 4e-3
U = 2.0 ** -53          # unit roundoff of the double accumulators
TWV = {np.float64: 348, np.float32: 720}   # strip_cols of the production k_fused_wa tilings (mw_schedule.h, WaCfg)
WA_VARIANT = {np.float64: 17, np.float32: 16}
SMALL_VARIANT = {np.float64: 5, np.float32: 7}
WA_WARP_STRIDE, WA_LANE_COLS, WA_HL = 186, 6, 12


# ---- pure-numpy references --------------------------------------------------------------------------------------

def exact_checksum(w, global_row0=0, dem_cols=None, rows_per_chunk=None):
    """The value wdpm_water_checksum defines, computed exactly on the host: sum over the cells of bits(w) * (2 * idx + 1)
    mod 2^64, idx = (global_row0 + i) * dem_cols + j the cell's row-major position in the whole DEM (0-based interior
    coordinates; `w` holds the owned interior rows, its first row being DEM row global_row0). fp32 bit patterns are
    zero-extended to 64 bits. numpy's uint64 arithmetic wraps, which is the mod 2^64."""
    w = np.ascontiguousarray(w)
    dem_cols = w.shape[1] if dem_cols is None else dem_cols
    bits = w.view(np.uint64) if w.dtype == np.float64 else w.view(np.uint32)
    step = rows_per_chunk or max(1, (1 << 22) // max(1, w.shape[1]))
    j = np.arange(w.shape[1], dtype=np.uint64)
    acc = 0
    for r0 in range(0, w.shape[0], step):
        b = bits[r0:r0 + step].astype(np.uint64)
        i = np.arange(global_row0 + r0, global_row0 + r0 + b.shape[0], dtype=np.uint64)[:, None]
        weight = (i * np.uint64(dem_cols) + j) * np.uint64(2) + np.uint64(1)
        acc = (acc + int((b * weight).sum(dtype=np.uint64))) % (1 << 64)
    return acc


def reduction_chain(padded_rows, padded_cols, sm_count):
    """L, the longest chain of floating-point additions behind one masked_sum of k_block_reduce_stage1/2 over a grid of
    padded_rows x padded_cols cells with reduce_blocks = 8 * sm_count:

        L = ceil(padded_rows / reduce_blocks) * ceil(padded_cols / 256)   sequential additions per thread
            + 5                                                           shuffle levels of a warp
            + 8                                                           warp partials of a block
            + reduce_blocks                                               stage 2, one thread

    Every partial sum is rounded once per addition, so |masked_sum - exact| <= L * 2^-53 * sum(|w_valid|)."""
    rb = 8 * sm_count
    return -(-padded_rows // rb) * -(-padded_cols // 256) + 5 + 8 + rb


def sum_bound(chain, w_valid):
    return chain * U * math.fsum(np.abs(w_valid.astype(np.float64)))


def oracle_block_outlets(oracle, w, d, thres, n_iters, outlets, totals):
    """One convergence block of Drain with an outlet set, in place on the padded grid w (the block of WDPMCL.c:1054-1268
    with oracle.iterate_outlets for the iterations): threshold pass w < thres -> 0 over the whole padded grid,
    snapshot, n_iters iterations, then reductions over the valid cells (d > NODATA).
    Returns (max_diff, exact masked sum (fsum), wet cells, per-outlet totals in the caller's order)."""
    dt = w.dtype.type
    w[w < dt(thres)] = 0
    old = w.copy()
    totals = oracle.iterate_outlets(w, d, NODATA, n_iters, outlets, totals=totals)
    valid = d > dt(NODATA)
    md = float(np.max(np.abs(w[valid] - old[valid]), initial=dt(0)))
    return md, math.fsum(w[valid].astype(np.float64)), int(np.count_nonzero(w[valid] > 0)), totals


def ordered_sum(v, dt):
    """Totals added in outlet order in the solver's precision (what a block's total_drain reports for a set)."""
    acc = dt(v[0])
    for x in v[1:]:
        acc = dt(acc + dt(x))
    return acc


# ---- helpers ----------------------------------------------------------------------------------------------------

def _bits(x, dt):
    a = np.asarray(x, dtype=dt)
    return a.view(np.uint64 if dt == np.float64 else np.uint32)


def _same_bits(a, b, dt):
    return np.array_equal(_bits(a, dt), _bits(b, dt))


def _code(dt):
    from wdpm_b200 import F32, F64
    return F64 if dt == np.float64 else F32


def _tiling(i):
    return {k: i[k] for k in ("window_cols", "strip_cols", "cta_threads", "smem_bytes")}


def _variant_tiling(variant, dt):
    from wdpm_b200 import solver
    return _tiling(solver.fused_variant_info(variant, _code(dt)))


def _assert_band(info, band, dt):
    """The kernel and tiling AUTO is meant to pick for this size band."""
    from wdpm_b200 import KERNEL_FUSED, KERNEL_RESIDENT
    if band == "resident":
        assert info["kernel"] == KERNEL_RESIDENT, info
        return
    assert info["kernel"] == KERNEL_FUSED, info
    if band == "small":
        assert info["warp_autonomous"] == 0 and _tiling(info) == _variant_tiling(SMALL_VARIANT[dt], dt), info
    else:
        assert info["warp_autonomous"] == 1 and _tiling(info) == _variant_tiling(WA_VARIANT[dt], dt), info
        assert info["strip_cols"] == TWV[dt]


def _border_cell(info, rows, cols, dt):
    """A cell on an ownership border of the tiling in use: the first owned row of the second chunk (resident kernel:
    tile row) and the first (fp64) or second (fp32) owned column of the second strip, inside the grid."""
    r = info["chunk_rows"] if info["chunk_rows"] <= rows else rows // 2 + 1
    c = info["strip_cols"] + (0 if dt == np.float64 else 1)
    return max(r, 1), (c if c <= cols else cols // 2 + 1)


def _check_block(r, a, D, dt, md, chain):
    """One block's reductions against the oracle grid `a` after the block: max_diff exactly, wet cells exactly,
    masked_sum within the rounding bound of the device's fixed-order sum around the exact sum."""
    valid = D > dt(NODATA)
    assert r.max_diff == md, (r.max_diff, md)
    assert r.wet_cells == int(np.count_nonzero((a > 0) & valid))
    wv = a[valid]
    exact = math.fsum(wv.astype(np.float64))
    assert abs(r.masked_sum - exact) <= sum_bound(chain, wv), (r.masked_sum, exact)


def _case(seed, rows, cols, dt):
    rng = np.random.default_rng(seed)
    D, W = random_case(rng, rows, cols, dt, nodata_fraction=0.05, wet_fraction=0.6, depth=0.05)
    return rng, D, W


# ---- A: AUTO bands x modules x precisions through run_block -----------------------------------------------------

A_SHAPES = [
    ("resident", 1022, 1022),   # (R+2)(C+2) = 2^20 exactly
    ("resident", 700, 1490),    # 1 047 384 cells, not square
    ("small", 1023, 1022),      # 2^20 + 1024
    ("small", 2046, 2045),      # 2^22 - 2048
    ("wa", 2046, 2046),         # 2^22 exactly
    ("wa", 1200, 3600),         # partial last strip (fp64: 3602 mod 348 = 122 columns)
    ("wa", 8000, 530),          # tall and narrow: many AUTO chunks
    ("wa", 520, 8200),          # short and wide: many strips
]
BLOCK_ITERS = (5, 7, 5)


@pytest.mark.parametrize("band,rows,cols", A_SHAPES, ids=[f"{b}-{r}x{c}" for b, r, c in A_SHAPES])
@pytest.mark.parametrize("mod", [0, 1, 2], ids=["add", "subtract", "drain"])
@pytest.mark.parametrize("dt", [np.float64, np.float32], ids=["f64", "f32"])
def test_auto_blocks_match_oracle(cuda_lib, oracle, dt, mod, band, rows, cols):
    """AUTO, zero threshold > 0, a water file with the NODATA value on invalid cells: the first block's prologue clears
    them, so the first block runs guarded and the later ones the clean launch. Water grid bit for bit, max_diff and
    wet_cells exactly, total_drain bit for bit, masked_sum within the bound around the exact sum. Drain: the
    reference's single outlet, found by find_outlet on a minimum planted on a chunk and a strip border."""
    from wdpm_b200 import Solver, ascgrid
    _, D, W = _case(1000 + 7 * rows + cols + mod, rows, cols, dt)
    s = Solver(rows, cols, NODATA, mod, dtype=_code(dt), zero_threshold=THRES)
    info = s.info()
    _assert_band(info, band, dt)
    outlet, td = (0, 0), 0.0
    if mod == 2:
        outlet = _border_cell(info, rows, cols, dt)
        D[outlet] = dt(1.0)   # the lowest cell with dem > 0
        W[outlet] = dt(0.03)
    W[D <= NODATA] = dt(NODATA)   # as a water file written by the Add module has it
    s.upload(D[1:-1, 1:-1], W[1:-1, 1:-1])
    if mod == 2:
        r, c, e = s.find_outlet()
        assert (r, c) == outlet == oracle.find_outlet(D) and e == 1.0
        td = max(s.get_cell_water(r, c), 0.0)   # the reference's seed (WDPMCL.c:1029)
        s.set_total_drain(td)
    chain = reduction_chain(rows + 2, cols + 2, info["sm_count"])
    a = W.copy()
    for n in BLOCK_ITERS:
        md, _, td = oracle.block(a, D, NODATA, mod, dt(THRES), n, outlet=outlet, totaldrain=td)
        res = s.run_block(n)
        _check_block(res, a, D, dt, md, chain)
        if mod == 2:
            assert _same_bits(res.total_drain, td, dt), (res.total_drain, td)
    b = ascgrid.pad_grid(s.download_water(), dt(0))
    _assert_band(s.info(), band, dt)   # still the same path (AUTO's resident kernel may fall back at run time)
    s.close()
    assert _same_bits(a, b, dt), int((a != b).sum())


@pytest.mark.parametrize("mod", [0, 1, 2], ids=["add", "subtract", "drain"])
@pytest.mark.parametrize("dt", [np.float64, np.float32], ids=["f64", "f32"])
def test_auto_water_on_nodata_cells_stays_guarded(cuda_lib, oracle, dt, mod):
    """Positive water on NODATA cells survives every threshold pass, so the water is never clean and every block must
    keep the guarded launch of k_fused_wa: the unguarded step would move water out of an invalid centre."""
    from wdpm_b200 import Solver, ascgrid
    rows, cols = 2046, 2046
    rng, D, W = _case(2000 + mod, rows, cols, dt)
    s = Solver(rows, cols, NODATA, mod, dtype=_code(dt), zero_threshold=THRES)
    info = s.info()
    _assert_band(info, "wa", dt)
    outlet, td = (0, 0), 0.0
    if mod == 2:
        outlet = _border_cell(info, rows, cols, dt)
        D[outlet] = dt(1.0)
    invalid = D <= NODATA
    W[invalid] = dt(NODATA)
    W[invalid & (rng.uniform(size=D.shape) < 0.5)] = dt(0.25)
    W[0, :] = W[-1, :] = W[:, 0] = W[:, -1] = 0   # the upload covers the interior only
    s.upload(D[1:-1, 1:-1], W[1:-1, 1:-1])
    if mod == 2:
        assert s.find_outlet()[:2] == outlet
        td = max(s.get_cell_water(*outlet), 0.0)
        s.set_total_drain(td)
    chain = reduction_chain(rows + 2, cols + 2, info["sm_count"])
    a = W.copy()
    for n in BLOCK_ITERS:
        md, _, td = oracle.block(a, D, NODATA, mod, dt(THRES), n, outlet=outlet, totaldrain=td)
        res = s.run_block(n)
        _check_block(res, a, D, dt, md, chain)
        if mod == 2:
            assert _same_bits(res.total_drain, td, dt)
    b = ascgrid.pad_grid(s.download_water(), dt(0))
    s.close()
    assert np.count_nonzero(a[invalid] == dt(0.25)) > 1000   # the water on invalid cells is still there
    assert _same_bits(a[1:-1, 1:-1], b[1:-1, 1:-1], dt), int((a != b).sum())


def _border_outlets(info, rows, cols, rng, n_random=4):
    """About 20 outlets: on chunk and strip borders (first owned rows / columns and their neighbours) and on the rim."""
    cr, sc = info["chunk_rows"], info["strip_cols"]
    want = [(1, 1), (1, cols), (rows, 1), (rows, cols), (1, cols // 2), (rows // 2, 1), (rows // 2 + 1, cols), (rows, cols // 3),
            (cr, sc), (cr, sc + 1), (cr - 1, sc - 1), (cr + 1, 2 * sc), (2 * cr, sc), (2 * cr, 2 * sc + 1), (cr, 5), (7, sc),
            (3 * cr - 1, sc + 2)]
    want += [(int(rng.integers(1, rows + 1)), int(rng.integers(1, cols + 1))) for _ in range(n_random)]
    out = []
    for r, c in want:
        if 1 <= r <= rows and 1 <= c <= cols and (r, c) not in out:
            out.append((r, c))
    return out


@pytest.mark.parametrize("band,rows,cols", [("resident", 1022, 1022), ("wa", 1200, 3600)], ids=["resident", "wa-1200x3600"])
@pytest.mark.parametrize("dt", [np.float64, np.float32], ids=["f64", "f32"])
def test_auto_outlet_set_blocks_match_oracle(cuda_lib, oracle, dt, band, rows, cols):
    """An outlet set on chunk / strip borders and the rim through AUTO and run_block: the grid, every outlet's total
    and max_diff / wet_cells exactly; total_drain is the outlet-order sum of the totals in the solver's precision."""
    from wdpm_b200 import Solver, ascgrid
    rng, D, W = _case(3000 + rows, rows, cols, dt)
    s = Solver(rows, cols, NODATA, 2, dtype=_code(dt), zero_threshold=THRES)
    info = s.info()
    _assert_band(info, band, dt)
    outlets = _border_outlets(info, rows, cols, rng)
    assert len(outlets) >= 18
    for rc in outlets:
        D[rc] = dt(480.0)   # outlets lie on valid cells
    W[D <= NODATA] = dt(NODATA)
    s.upload(D[1:-1, 1:-1], W[1:-1, 1:-1])
    s.set_outlets(outlets)
    s.seed_outlet_drains()
    totals = np.array([max(W[rc], dt(0)) for rc in outlets], dtype=dt)
    chain = reduction_chain(rows + 2, cols + 2, info["sm_count"])
    a = W.copy()
    for n in BLOCK_ITERS:
        md, _, wet, totals = oracle_block_outlets(oracle, a, D, THRES, n, outlets, totals)
        res = s.run_block(n)
        _check_block(res, a, D, dt, md, chain)
        assert res.wet_cells == wet
        assert _same_bits(s.get_outlet_drains(len(outlets)).astype(dt), totals, dt)
        assert _same_bits(res.total_drain, ordered_sum(totals, dt), dt)
    b = ascgrid.pad_grid(s.download_water(), dt(0))
    _assert_band(s.info(), band, dt)
    s.close()
    assert _same_bits(a, b, dt), int((a != b).sum())


# ---- B: k_fused_wa geometry sweep -------------------------------------------------------------------------------

def _wa_widths(dt):
    """Padded widths around the strip, warp and lane boundaries of the production k_fused_wa tiling: a window starts at
    padded column st*TWV - 12, its warps 186 columns apart, lanes 6 apart (lane 31 stores nothing)."""
    twv = TWV[dt]
    kw = 2 if dt == np.float64 else 4   # warps per row triple
    widths = [k * twv + d for k in (1, 2, 3) for d in (-2, -1, 0, 1, 2)]
    for st in (0, 1):
        x0 = st * twv - WA_HL
        for j in range(1, kw):
            last = x0 + WA_WARP_STRIDE * j   # a warp's first column is the last column of the grid
            widths += [last, last + 1, last + 2]
        for lane in (1, 30, 31):
            widths += [x0 + WA_LANE_COLS * lane + 1, x0 + WA_WARP_STRIDE + WA_LANE_COLS * lane + 2]
    widths += list(range(3, 41))
    return sorted({w for w in widths if w >= 3})


def _chunk_leaving(total_triples, last):
    """Forced chunk rows that leave a last chunk of `last` row triples (0 = AUTO's chunking)."""
    if last == 0:
        return 0
    for ct in range(last + 1, total_triples):
        if total_triples % ct == last:
            return 3 * ct
    return 0


@pytest.mark.parametrize("mod", [0, 1, 2], ids=["add", "subtract", "drain"])
@pytest.mark.parametrize("dt", [np.float64, np.float32], ids=["f64", "f32"])
def test_wa_geometry_sweep_matches_oracle(cuda_lib, oracle, dt, mod):
    """The production k_fused_wa variant on small grids: every padded width of _wa_widths, heights of every residue
    mod 3 and one below the ring depth (36 rows), chunkings whose last chunk holds 1, 2 or 3 row triples; each grid
    through iterate at threshold 0 (guarded launch) and through two blocks of run_block at a threshold > 0 (clean
    launch). Drain: outlets in the last column of a strip and in the first row of the last chunk."""
    from wdpm_b200 import KERNEL_FUSED, Solver, ascgrid
    code, variant, twv = _code(dt), WA_VARIANT[dt], TWV[dt]
    assert _variant_tiling(variant, dt)["strip_cols"] == twv
    heights = (62, 61, 60, 20)     # padded rows: residues 2, 1, 0 mod 3, and fewer than the 36 ring rows
    rng = np.random.default_rng(4000 + 10 * mod + (dt == np.float32))
    for k, pw in enumerate(_wa_widths(dt)):
        ph = heights[k % 4]
        rows, cols = ph - 2, pw - 2
        chunk = _chunk_leaving((ph + 2) // 3, (k // 4) % 4)
        D, W = random_case(rng, rows, cols, dt, nodata_fraction=0.05, wet_fraction=0.7, depth=0.05)
        outlets = []
        for thres in (0.0, THRES):
            s = Solver(rows, cols, NODATA, mod, dtype=code, zero_threshold=thres, kernel=KERNEL_FUSED, fused_variant=variant,
                       fused_chunk_rows=chunk)
            info = s.info()
            n_strips = -(-pw // twv)
            assert info["warp_autonomous"] == 1 and info["strip_cols"] == twv
            assert info["grid_ctas"] % n_strips == 0 and (chunk == 0 or info["chunk_rows"] == chunk), (info, chunk)
            if mod == 2 and not outlets:
                last_chunk_row = (info["grid_ctas"] // n_strips - 1) * info["chunk_rows"]
                strip_end = (cols + 1) // twv * twv - 1 if cols + 1 >= twv else cols
                outlets = [(min(max(ph // 2, 1), rows), max(strip_end, 1)), (min(max(last_chunk_row, 1), rows), min(twv // 2, cols))]
                outlets = list(dict.fromkeys(outlets))
                for rc in outlets:
                    D[rc] = dt(480.0)
                    W[rc] = dt(0.02)
            s.upload(D[1:-1, 1:-1], W[1:-1, 1:-1])
            a = W.copy()
            if mod == 2:
                s.set_outlets(outlets)
                s.seed_outlet_drains()
                totals = np.array([max(W[rc], dt(0)) for rc in outlets], dtype=dt)
            if thres == 0.0:
                s.iterate(5)
                if mod == 2:
                    totals = oracle.iterate_outlets(a, D, NODATA, 5, outlets, totals=totals)
                else:
                    oracle.iterate(a, D, NODATA, mod, 5)
            else:
                for n in (3, 4):
                    res = s.run_block(n)
                    if mod == 2:
                        md, _, wet, totals = oracle_block_outlets(oracle, a, D, thres, n, outlets, totals)
                    else:
                        md, _, _ = oracle.block(a, D, NODATA, mod, dt(thres), n)
                        wet = int(np.count_nonzero((a > 0) & (D > dt(NODATA))))
                    assert res.max_diff == md and res.wet_cells == wet, (pw, ph, chunk, thres)
            b = ascgrid.pad_grid(s.download_water(), dt(0))
            tb = s.get_outlet_drains(len(outlets)).astype(dt) if mod == 2 else None
            s.close()
            assert _same_bits(a, b, dt), (pw, ph, chunk, thres, int((a != b).sum()))
            if mod == 2:
                assert _same_bits(tb, totals, dt), (pw, ph, chunk, thres)


# ---- C: order-free outputs against exact host values ------------------------------------------------------------

@pytest.mark.parametrize("dt", [np.float64, np.float32], ids=["f64", "f32"])
def test_water_checksum_is_the_exact_sum(cuda_lib, dt):
    """wdpm_water_checksum recomputed from the downloaded grid with exact integer arithmetic, for a single solver and
    for three in-process stripes (each stripe's part, and their sum); and its sensitivity to one cell's bits."""
    from wdpm_b200 import Solver
    from wdpm_b200.stripes import StripeSolver, connect_in_process, plan_stripes
    rows, cols = 301, 1103
    rng, D, W = _case(5000, rows, cols, dt)
    dem, w0 = D[1:-1, 1:-1], W[1:-1, 1:-1]
    s = Solver(rows, cols, NODATA, 0, dtype=_code(dt), zero_threshold=THRES)
    s.upload(dem, w0)
    s.run_block(4)
    w = s.download_water()
    assert s.water_checksum() == exact_checksum(w)
    plan = plan_stripes(rows, 3)
    ss = [StripeSolver(rows, cols, NODATA, 0, st, dtype=_code(dt), zero_threshold=THRES) for st in plan]
    connect_in_process(ss)
    for t, st in zip(ss, plan):
        t.upload_band(dem[st.band_row0:st.band_row0 + st.band_rows], w0[st.band_row0:st.band_row0 + st.band_rows])
    for t in ss:
        t.block_begin()
    for t in ss:
        t.block_enqueue(4)
    for t in ss:
        t.block_end()
    parts = [t.water_checksum() for t in ss]
    owned = [t.download_owned() for t in ss]
    for t in ss:
        t.close()
    for p, o, st in zip(parts, owned, plan):
        assert p == exact_checksum(o, st.owned_row0, cols), st
    assert np.array_equal(np.concatenate(owned).view(np.uint8), w.view(np.uint8))
    assert sum(parts) % (1 << 64) == exact_checksum(w)

    # sensitivity, on the uploaded grid
    base = np.ascontiguousarray(w0)
    s.upload(dem, base)
    c0 = s.water_checksum()
    assert c0 == exact_checksum(base)
    i, j = 17, 611
    idx = i * cols + j
    uint = np.uint64 if dt == np.float64 else np.uint32
    v = base.copy()
    v.view(uint)[i, j] ^= uint(1)   # lowest mantissa bit
    s.upload_water(v)
    delta = (s.water_checksum() - c0) % (1 << 64)
    assert delta in ((2 * idx + 1) % (1 << 64), (-(2 * idx + 1)) % (1 << 64))
    pz, nz = base.copy(), base.copy()
    pz[i, j], nz[i, j] = dt(0.0), dt(-0.0)
    s.upload_water(pz)
    cp = s.water_checksum()
    s.upload_water(nz)
    cn = s.water_checksum()
    sign = 1 << (63 if dt == np.float64 else 31)
    assert (cn - cp) % (1 << 64) == sign * (2 * idx + 1) % (1 << 64)
    if dt == np.float64:
        assert (cn - cp) % (1 << 64) == 1 << 63
    sw = base.copy()
    sw[3, 4], sw[200, 900] = dt(0.125), dt(0.375)
    s.upload_water(sw)
    c1 = s.water_checksum()
    sw[3, 4], sw[200, 900] = sw[200, 900], sw[3, 4]
    s.upload_water(sw)
    assert s.water_checksum() != c1
    s.close()


def _final_stats_ref(dem, w, marked=()):
    valid = dem > NODATA
    for rc in marked:
        valid[rc] = True
    if not valid.any():
        return 0, 0, 0.0
    w64 = w.astype(np.float64)
    return int(valid.sum()), int(np.count_nonzero((w64 > 0.001) & valid)), float(w64[valid].max())


@pytest.mark.parametrize("dt", [np.float64, np.float32], ids=["f64", "f32"])
def test_final_statistics_edge_inputs(cuda_lib, dt):
    """No valid cell, an all-dry grid, water at exactly 0.001 and one ulp either side (the comparison is made in double:
    fp32 0.001 is above it), and outlet-marked cells, which count as valid."""
    from wdpm_b200 import Solver
    rows, cols = 90, 400
    rng, D, W = _case(6000, rows, cols, dt)
    dem, w = D[1:-1, 1:-1].copy(), W[1:-1, 1:-1].copy()
    with Solver(rows, cols, NODATA, 0, dtype=_code(dt)) as s:
        s.upload(np.full_like(dem, NODATA), w)
        assert s.final_statistics() == (0, 0, 0.0)
        s.upload(dem, np.zeros_like(w))
        assert s.final_statistics() == _final_stats_ref(dem, np.zeros_like(w)) and s.final_statistics()[1:] == (0, 0.0)
        mm = dt(0.001)
        edge = np.where(dem > NODATA, rng.choice(np.array([np.nextafter(mm, dt(0)), mm, np.nextafter(mm, dt(1))], dtype=dt), dem.shape), dt(0))
        s.upload(dem, edge)
        got = s.final_statistics()
        assert got == _final_stats_ref(dem, edge), got
        # fp64: only the value above 0.001 counts; fp32: 0.001f is 0.0010000000475 in double and counts too
        exact = (dem > NODATA) & (edge == mm)
        assert got[1] == int(np.count_nonzero((dem > NODATA) & (edge > mm))) + (int(exact.sum()) if dt == np.float32 else 0)
        s.upload(dem, w)
        assert s.final_statistics() == _final_stats_ref(dem, w)
    with Solver(rows, cols, NODATA, 2, dtype=_code(dt)) as s:
        marked = [(0, 0), (5, 7), (40, 399), (89, 200)]
        d2 = dem.copy()
        for rc in marked:
            d2[rc] = dt(450.0)
        w2 = w.copy()
        w2[5, 7] = dt(9.5)   # the deepest water sits on an outlet
        s.upload(d2, w2)
        s.set_outlets([(r + 1, c + 1) for r, c in marked])
        assert s.final_statistics() == _final_stats_ref(d2, w2, marked) and s.final_statistics()[2] == 9.5


def _outlet_dems(dt, rows, cols, rng):
    """DEMs for the outlet search, with the expected (padded) outlet or None."""
    base = (500 + 3 * rng.standard_normal((rows, cols))).astype(dt)
    base[rng.uniform(size=base.shape) < 0.05] = dt(NODATA)
    out = []
    d = base.copy()   # a plateau of equal minimum elevation over rows far apart (other stage-1 blocks)
    for r, c in ((1900, 3), (611, 2000), (611, 1999), (2045, 0), (40, 1500), (1024, 1024)):
        d[r, c] = dt(3.25)
    out.append(("plateau", d, (41, 1501)))
    d = base.copy()
    tiny = np.nextafter(dt(0), dt(1))   # smallest positive subnormal
    d[1500, 17], d[200, 9] = tiny, dt(2 * tiny)
    out.append(("subnormal", d, (1501, 18)))
    d = base.copy()
    d[3, 3], d[4, 4], d[5, 5] = dt(0.0), dt(-0.0), dt(-1.0)
    d[1200, 1200] = dt(0.5)
    out.append(("signed_zero", d, (1201, 1201)))
    d = np.full((rows, cols), dt(2e8), dtype=dt)
    d[100, 100] = dt(1e8)                         # not below the reference's starting minimum
    d[900, 5] = np.nextafter(dt(1e8), dt(0))      # just below it
    out.append(("near_1e8", d, (901, 6)))
    d = np.full((rows, cols), dt(-5.0), dtype=dt)
    d[::7, ::5] = dt(1e8)
    d[10, 10], d[11, 11] = dt(3e9), dt(0.0)
    out.append(("none_below_1e8", d, None))
    d = base.copy()
    d[rows - 1, cols - 7] = dt(0.75)
    out.append(("last_row", d, (rows, cols - 6)))
    return out


@pytest.mark.parametrize("dt", [np.float64, np.float32], ids=["f64", "f32"])
def test_find_outlet_ties_and_edges(cuda_lib, oracle, dt):
    """find_outlet on an AUTO-size grid (stage 1 runs 8 x SMs blocks) against oracle.find_outlet: ties across blocks
    (first in row-major order wins), the smallest subnormal, signed zeros, the 1e8 limit, no outlet, the last row."""
    from wdpm_b200 import Solver, WdpmError, ascgrid
    rows, cols = 2046, 2046
    rng = np.random.default_rng(7000)
    with Solver(rows, cols, NODATA, 0, dtype=_code(dt)) as s:
        _assert_band(s.info(), "wa", dt)
        for name, d, want in _outlet_dems(dt, rows, cols, rng):
            D = ascgrid.pad_grid(d, dt(NODATA))
            assert oracle.find_outlet(D) == want, name
            s.upload(d, None)
            if want is None:
                with pytest.raises(WdpmError):
                    s.find_outlet()
                continue
            r, c, e = s.find_outlet()
            assert (r, c) == want, name
            assert _same_bits(e, D[r, c], dt), name


# ---- D: production stripes --------------------------------------------------------------------------------------

def _stripes_lockstep(ss, n):
    for _ in range(n):
        for t in ss:
            t.phase(0)
        for t in ss:
            t.synchronize()
        for t in ss:
            t.phase(1)
        for t in ss:
            t.synchronize()


@pytest.mark.parametrize("mod", [0, 1, 2], ids=["add", "subtract", "drain"])
@pytest.mark.parametrize("dt", [np.float64, np.float32], ids=["f64", "f32"])
def test_production_stripes_match_oracle(cuda_lib, oracle, monkeypatch, dt, mod):
    """Three in-process stripes on the production k_fused_wa tiling with AUTO chunking and a zero threshold > 0,
    free-running (block_begin / enqueue / end) and in lockstep (phase 0 / phase 1): the assembled grid, the combined
    block results and the summed checksum against the oracle and the exact checksum. Drain: an outlet on the first
    owned row of the middle stripe and on a strip border, so centres of two stripes drain it."""
    from wdpm_b200.stripes import StripeSolver, combine_block_results, connect_in_process, plan_stripes
    monkeypatch.setenv("WDPM_B200_HALO_TIMEOUT_MS", "20000")   # a stuck wait ends as WDPM_E_HALO
    rows, cols = 600, 1500
    _, D, W = _case(8000 + mod, rows, cols, dt)
    plan = plan_stripes(rows, 3)
    outlet = (plan[1].row0, TWV[dt])
    if mod == 2:
        D[outlet] = dt(1.0)
        W[outlet] = dt(0.04)
    W[D <= NODATA] = dt(NODATA)
    dem, w0 = D[1:-1, 1:-1], W[1:-1, 1:-1]
    ss = [StripeSolver(rows, cols, NODATA, mod, st, dtype=_code(dt), zero_threshold=THRES) for st in plan]
    for t in ss:
        i = t.info()
        assert i["warp_autonomous"] == 1 and _tiling(i) == _variant_tiling(WA_VARIANT[dt], dt), i
    connect_in_process(ss)
    sm = ss[0].info()["sm_count"]
    chain = max(reduction_chain(st.rows, cols + 2, sm) for st in plan) + len(plan)

    def upload():
        for t, st in zip(ss, plan):
            t.upload_band(dem[st.band_row0:st.band_row0 + st.band_rows], w0[st.band_row0:st.band_row0 + st.band_rows])
            if mod == 2:
                t.set_outlet(*outlet)
                t.seed_outlet_drains()

    for mode in ("free", "lockstep"):
        upload()
        a, td = W.copy(), max(W[outlet], dt(0)) if mod == 2 else 0.0
        for n in BLOCK_ITERS:
            md, _, td = oracle.block(a, D, NODATA, mod, dt(THRES), n, outlet=outlet if mod == 2 else (0, 0), totaldrain=td)
            for t in ss:
                t.block_begin()
            if mode == "free":
                for t in ss:
                    t.block_enqueue(n)
            else:
                _stripes_lockstep(ss, n)
            res = combine_block_results([t.block_end() for t in ss])
            _check_block(res, a, D, dt, md, chain)
            if mod == 2:
                assert _same_bits(res.total_drain, td, dt), (mode, res.total_drain, td)
        full = np.concatenate([t.download_owned() for t in ss])
        assert _same_bits(full, a[1:-1, 1:-1], dt), (mode, int((full != a[1:-1, 1:-1]).sum()))
        assert sum(t.water_checksum() for t in ss) % (1 << 64) == exact_checksum(a[1:-1, 1:-1]), mode
    for t in ss:
        t.close()


# ---- E: one grid beyond 2^31 elements ---------------------------------------------------------------------------

def test_grid_beyond_2_31_elements(cuda_lib):
    """47 000^2 fp32 Add (padded 2.209e9 cells, every device grid > 2^31 elements): AUTO (k_fused_wa) equals the colour
    kernel bit for bit after 2 iterations; a crop at the last rows and columns equals the oracle; run_block(0)'s
    reductions, the checksum and find_outlet (minimum in the last row, padded index > 2^31) against host values."""
    import psutil
    import torch
    from oracle import pyoracle
    from wdpm_b200 import F32, KERNEL_COLOUR, KERNEL_FUSED, Solver, ascgrid
    if torch.cuda.get_device_properties(0).total_memory < 100e9 or psutil.virtual_memory().available < 60e9:
        pytest.skip("needs a device with >= 100 GB and >= 60 GB of free host memory (47 000^2 fp32: ~36 GB on the device, ~30 GB on the host)")
    n, dt = 47000, np.float32
    g = torch.Generator(device="cuda")
    g.manual_seed(47)
    dem_t = 500 + 3 * torch.randn((n, n), generator=g, device="cuda", dtype=torch.float32)
    dem_t[torch.rand((n, n), generator=g, device="cuda") < 0.02] = NODATA
    dem = dem_t.cpu().numpy()
    del dem_t
    torch.cuda.empty_cache()
    low = (n - 1, n - 20)
    dem[low] = dt(0.5)
    outs = []
    for kernel in (0, KERNEL_COLOUR):
        s = Solver(n, n, NODATA, 0, dtype=F32, kernel=kernel)
        info = s.info()
        assert info["device_bytes"] > 4 * 4 * (1 << 31)   # four grids (dem, two water buffers, snapshot) of > 2^31 fp32
        if kernel == 0:
            assert info["kernel"] == KERNEL_FUSED and info["warp_autonomous"] == 1 and _tiling(info) == _variant_tiling(16, dt)
        s.upload(dem, None)
        s.apply_add(0.1, 1.0)
        s.iterate(2)
        if kernel == 0:
            r, c, e = s.find_outlet()
            assert (r, c) == (low[0] + 1, low[1] + 1) and e == 0.5
            assert r * (n + 2) + c > 1 << 31
            blk = s.run_block(0)
        outs.append(s.download_water())
        if kernel == 0:
            chk = s.water_checksum()
        s.close()
    w = outs[0]
    assert np.array_equal(w.view(np.uint32), outs[1].view(np.uint32))
    del outs
    # reductions of run_block(0) (threshold 0 on water >= 0 is a no-op) against per-band float64 sums
    parts, absparts, wet = [], [], 0
    for r0 in range(0, n, 1000):
        wb, vb = w[r0:r0 + 1000], dem[r0:r0 + 1000] > NODATA
        x = wb[vb].astype(np.float64)
        parts.append(float(x.sum()))
        absparts.append(float(np.abs(x).sum()))
        wet += int(np.count_nonzero(x > 0))
    assert blk.wet_cells == wet and blk.max_diff == 0.0
    ref, absum = math.fsum(parts), math.fsum(absparts)
    chain = reduction_chain(n + 2, n + 2, torch.cuda.get_device_properties(0).multi_processor_count) + 64  # + the band sums' own
    assert abs(blk.masked_sum - ref) <= chain * U * absum, (blk.masked_sum, ref)
    assert chk == exact_checksum(w)
    # oracle on a 320^2 crop ending at the last row and column: the crop's bottom and right margins are the DEM's own,
    # so only cells within 18 * n_it + 4 of its top and left cuts can differ; the origin keeps the colours (multiple of 3)
    m, k = 18 * 2 + 4, 320
    r0 = c0 = 3 * ((n - k) // 3)
    assert r0 + k == n
    Dc = ascgrid.pad_grid(dem[r0:, c0:], dt(NODATA))
    Wc = np.where(Dc > NODATA, dt(0.1), dt(0)).astype(dt)
    pyoracle.Oracle().iterate(Wc, Dc, NODATA, 0, 2)
    assert np.array_equal(Wc[1 + m:-1, 1 + m:-1], w[r0 + m:, c0 + m:])
