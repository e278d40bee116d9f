"""Module driver: the host logic of WDPM's Add / Subtract / Drain runs around the solver.

Python twin of the command-line host (wdpm_b200/host/wdpm_host.c), used by the
tests and the benchmark. It keeps on the host exactly what the reference keeps
there - module set-up, the 1000-iteration block cadence, the stop tests and the
final statistics (/root/reference/src/WDPMCL.c:654-1034, :1054-1377, :1379-1467)
- and delegates each block to a backend with the `wdpm_b200.Solver` interface
(the CUDA library). Tests pass an oracle-backed object with the same methods to
check this logic on a machine without a GPU; the product never does.
"""
from __future__ import annotations

import dataclasses
from typing import Callable

import numpy as np

from . import solver as _solver

BLOCK_ITERS = 1000  # IterationNum, hard-coded at WDPMCL.c:597


@dataclasses.dataclass
class ModuleParams:
    module: str                 # "add" | "subtract" | "drain"
    depth_mm: float = 0.0       # add / subtract depth
    runoff_fraction: float = 1.0
    elevation_tol_mm: float = 1.0
    drain_tol_m3: float = 0.0
    zero_threshold_mm: float = 0.0
    iteration_limit: int = 0    # 0 = none; otherwise rounded up to a block (WDPMCL.c:1285-1287)
    block_iters: int = BLOCK_ITERS


@dataclasses.dataclass
class BlockLine:
    iterations: int
    max_diff: float
    vol_change: float | None
    water_left: float | None
    seconds: float


@dataclasses.dataclass
class RunReport:
    water: np.ndarray           # rows x cols, NODATA cells = nodata (what write_gis writes)
    iterations: int
    blocks: list
    initial_vol: float
    final_vol: float
    drain_vol: float
    water_frac: float
    mean_water: float
    drain_depth: float
    max_depth_mm: float
    outlet: tuple | None        # the reference's single outlet (None when a set was given)
    min_elevation: float | None  # its elevation, or the lowest outlet elevation of a set
    solver_ms: float
    launches: int
    outlet_totals: np.ndarray | None = None  # a set: every outlet's drained depth in m (x cellarea = m3), in outlet order


def default_backend(dtype=_solver.F64, **kw) -> Callable:
    def make(rows, cols, nodata, module, zero_threshold):
        return _solver.Solver(rows, cols, nodata, module, dtype=dtype, zero_threshold=zero_threshold, **kw)
    return make


def run_module(dem: np.ndarray, nodata: float, cellsize: float, params: ModuleParams, water: np.ndarray | None = None,
               backend: Callable | None = None, resume: bool = False, on_block: Callable | None = None,
               outlets=None) -> RunReport:
    """Run one module to its stop criterion.

    `water` is the water-file contents (None = "NULL"/absent). `resume=True` means
    `water` came from a scratch file: the module's add/subtract step is skipped
    (WDPMCL.c:668-673, :824-829). `outlets` (Drain only): None for the reference's
    single outlet, a list of 1-based (row, col), or "rim" (ascgrid.rim_outlets) -
    the water then leaves through every outlet of the set, each with its own total.
    """
    import time

    module = _solver.MODULES[params.module]
    rows, cols = dem.shape
    cellarea = cellsize * cellsize
    thres = params.zero_threshold_mm / 1000
    eltol = params.elevation_tol_mm / 1000.0
    make = backend or default_backend()
    be = make(rows, cols, nodata, module, thres)
    np_dtype = getattr(be, "np_dtype", np.float64)
    dem_t = np.ascontiguousarray(dem, dtype=np_dtype)
    valid = dem > nodata

    if water is None:
        if params.module == "drain":
            raise FileNotFoundError("Error water file missing")  # WDPMCL.c:971-972, exit code 42
        w0 = np.zeros_like(dem_t)
    else:
        w0 = np.ascontiguousarray(water, dtype=np_dtype)

    # Initial volume as the reference prints it (SURVEY appendix A, quirk 8): Add and Subtract sum
    # water[][] before any file has been read on the no-scratch path (WDPMCL.c:656-664, :812-821),
    # so they report 0; Drain sums the water file over valid cells (WDPMCL.c:1019-1028).
    if params.module == "drain":
        initial_vol = float(np.sum(np.where(valid, w0.astype(np.float64), 0.0))) * cellarea
    else:
        initial_vol = 0.0

    be.upload(dem_t, w0)
    if not resume:
        if params.module == "add":
            be.apply_add(params.depth_mm / 1000.0, params.runoff_fraction)
        elif params.module == "subtract":
            be.apply_subtract(params.depth_mm / 1000)

    outlet = None
    min_elev = None
    if outlets is not None and params.module == "drain":
        from .ascgrid import rim_outlets
        outlets = rim_outlets(dem, nodata) if isinstance(outlets, str) and outlets == "rim" else [(int(r), int(c)) for r, c in outlets]
        if not outlets:
            raise ValueError("the outlet set is empty")
        be.set_outlets(outlets)
        be.seed_outlet_drains()
        min_elev = min(float(dem[r - 1, c - 1]) for r, c in outlets)
    elif params.module == "drain":
        r, c, min_elev = be.find_outlet()
        outlet = (r, c)
        w_out = be.get_cell_water(r, c)
        be.set_total_drain(max(w_out, 0.0))  # WDPMCL.c:1029

    blocks = []
    k = 0
    total_drain = be.get_total_drain() if params.module == "drain" else 0.0
    solver_ms = 0.0
    launches = 0
    t0 = time.time()
    while True:
        old_drain = total_drain
        res = be.run_block(params.block_iters)
        k += params.block_iters
        solver_ms += res.block_ms
        launches += res.launches
        total_drain = res.total_drain
        if params.module == "drain":
            diffdrain = abs(total_drain - old_drain) * cellarea
            final_vol_blk = res.masked_sum * cellarea
            line = BlockLine(k, res.max_diff, diffdrain, final_vol_blk, time.time() - t0)
            done = res.max_diff <= eltol or diffdrain < params.drain_tol_m3  # WDPMCL.c:1287, :1303
        else:
            line = BlockLine(k, res.max_diff, None, None, time.time() - t0)
            done = res.max_diff <= eltol  # WDPMCL.c:1324, :1350
        if params.iteration_limit > 0 and k >= params.iteration_limit:
            done = True
        blocks.append(line)
        if on_block:
            on_block(line)
        if done:
            break

    w = be.download_water().astype(np.float64)
    outlet_totals = be.get_outlet_drains(len(outlets)) if outlets is not None and params.module == "drain" else None
    if hasattr(be, "close"):
        be.close()

    # final statistics, WDPMCL.c:1379-1459
    w = np.where(valid, w, nodata)
    watercount = int(np.count_nonzero((w > 0.001) & valid))
    watertotal = float(np.sum(w[valid]))  # row-major order
    final_vol = watertotal * cellarea
    basincount = int(np.count_nonzero(valid))
    with np.errstate(divide="ignore", invalid="ignore"):
        mean_water = watertotal / float(np.float32(watercount)) if watercount else float("nan")
        water_frac = float(np.float32(watercount) / np.float32(basincount)) if basincount else float("nan")
    drain_vol = total_drain * cellarea if params.module == "drain" else 0.0
    drain_depth = (drain_vol / (float(np.float32(basincount)) * cellarea)) * 1000 if params.module == "drain" else 0.0
    max_depth_mm = float(np.max(w)) * 1000  # scans every cell, NODATA included (WDPMCL.c:1451-1459)
    return RunReport(w, k, blocks, initial_vol, final_vol, drain_vol, water_frac, mean_water, drain_depth, max_depth_mm,
                     outlet, min_elev, solver_ms, launches, outlet_totals)
