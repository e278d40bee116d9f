"""Row-stripe partition of one DEM across GPUs (host side).

New work relative to the reference, which is single-device (/root/reference/src/WDPMCL.c:98-118).
`plan_stripes` is pure arithmetic (also exercised by CPU tests); `StripedSolver` wires one
`wdpm_b200.Solver` per rank through torch.distributed: CUDA IPC handles are all-gathered once, after
which halos travel GPU to GPU over NVLink inside the library (include/wdpm_b200.h, "row-stripe
partition") and only the per-block scalars cross the host (an all_gather of three numbers).
"""
from __future__ import annotations

import ctypes as C
import dataclasses

import numpy as np

from . import solver as _solver

HALO_ABOVE, HALO_BELOW = 3, 6  # rows; WDPM_STRIPE_HALO_* in include/wdpm_b200.h


@dataclasses.dataclass(frozen=True)
class Stripe:
    row0: int        # first owned PADDED row (multiple of 3)
    rows: int        # owned padded rows
    band_row0: int   # first INTERIOR row (0-based) the stripe must be given (owned + halos, clipped)
    band_rows: int
    owned_row0: int  # first interior row it owns
    owned_rows: int


def plan_stripes(rows: int, n: int) -> list[Stripe]:
    """Cut padded rows 0..rows+1 into n contiguous bands starting at multiples of 3, as equal as possible.
    Every band gets at least 9 rows (HALO_ABOVE + HALO_BELOW), which needs 9 * n padded rows: 3 * n row triples are
    not enough when the last one is partial, the last band would get 7 or 8 rows."""
    padded = rows + 2
    triples = (padded + 2) // 3
    if n < 1 or padded < 9 * n:
        raise ValueError(f"{rows} rows are too few for {n} stripes")
    out = []
    for r in range(n):
        t0, t1 = (triples * r) // n, (triples * (r + 1)) // n
        g0, g1 = 3 * t0, min(3 * t1, padded)
        blo, bhi = max(g0 - HALO_ABOVE, 1), min(g1 + HALO_BELOW, rows + 1)
        olo, ohi = max(g0, 1), min(g1, rows + 1)
        out.append(Stripe(g0, g1 - g0, blo - 1, bhi - blo, olo - 1, ohi - olo))
    return out


class _Endpoint(C.Structure):
    _fields_ = [("water_a", C.c_uint8 * 64), ("water_b", C.c_uint8 * 64), ("flags", C.c_uint8 * 64), ("device", C.c_int32),
                ("stripe_row0", C.c_int32), ("stripe_rows", C.c_int32), ("pitch", C.c_int32), ("pid", C.c_int64),
                ("local_ptr", C.c_uint64)]


class StripeSolver(_solver.Solver):
    """A Solver that owns one band of padded rows (mirror of a stripe wdpm_solver)."""

    def __init__(self, rows: int, cols: int, nodata: float, module: int, stripe: Stripe, **kw):
        self.stripe = stripe
        super().__init__(rows, cols, nodata, module, _stripe=(stripe.row0, stripe.rows), **kw)

    def upload_band(self, dem_band, water_band=None):
        st = self.stripe
        d = np.ascontiguousarray(dem_band, dtype=self.np_dtype)
        assert d.shape == (st.band_rows, self.cols), (d.shape, st)
        w = None if water_band is None else np.ascontiguousarray(water_band, dtype=self.np_dtype)
        _solver._check(self._lib.wdpm_stripe_upload(self._h, d.ctypes.data_as(C.c_void_p),
                                                    None if w is None else w.ctypes.data_as(C.c_void_p),
                                                    C.c_int32(st.band_row0), C.c_int32(st.band_rows)))

    def upload_band_ptr(self, dem_ptr: int, water_ptr: int | None):
        st = self.stripe
        _solver._check(self._lib.wdpm_stripe_upload(self._h, C.c_void_p(dem_ptr), C.c_void_p(water_ptr) if water_ptr else None,
                                                    C.c_int32(st.band_row0), C.c_int32(st.band_rows)))

    def download_owned(self, out=None) -> np.ndarray:
        st = self.stripe
        if out is None:
            out = np.empty((st.owned_rows, self.cols), dtype=self.np_dtype)
        _solver._check(self._lib.wdpm_download_water(self._h, out.ctypes.data_as(C.c_void_p)))
        return out

    def export(self) -> _Endpoint:
        ep = _Endpoint()
        _solver._check(self._lib.wdpm_stripe_export(self._h, C.byref(ep)))
        return ep

    def connect(self, above: _Endpoint | None, below: _Endpoint | None):
        _solver._check(self._lib.wdpm_stripe_connect(self._h, C.byref(above) if above is not None else None,
                                                     C.byref(below) if below is not None else None))

    def phase(self, which: int):
        _solver._check(self._lib.wdpm_stripe_phase(self._h, C.c_int32(which)))


def connect_in_process(stripes: list[StripeSolver]):
    eps = [s.export() for s in stripes]
    for i, s in enumerate(stripes):
        s.connect(eps[i - 1] if i > 0 else None, eps[i + 1] if i + 1 < len(stripes) else None)


def combine_block_results(results: list) -> _solver.BlockResult:
    """Whole-DEM block result from per-stripe results, in stripe order (deterministic sum)."""
    md = max(r.max_diff for r in results)
    ms = 0.0
    for r in results:
        ms += r.masked_sum
    td = 0.0
    for r in results:
        td += r.total_drain
    return _solver.BlockResult(md, ms, td, sum(r.wet_cells for r in results), results[0].iterations,
                               sum(r.launches for r in results), max(r.block_ms for r in results),
                               max(r.iterate_ms for r in results))


class DistributedSolver:
    """One stripe per rank of an initialised torch.distributed group (NCCL or gloo for the scalars)."""

    def __init__(self, rows: int, cols: int, nodata: float, module: int, device: int, **kw):
        import torch.distributed as dist
        self.dist = dist
        self.rank, self.world = dist.get_rank(), dist.get_world_size()
        self.plan = plan_stripes(rows, self.world)
        self.stripe = self.plan[self.rank]
        self.solver = StripeSolver(rows, cols, nodata, module, self.stripe, device=device, **kw)
        eps = [None] * self.world
        dist.all_gather_object(eps, bytes(self.solver.export()))
        eps = [_Endpoint.from_buffer_copy(b) for b in eps]
        self.solver.connect(eps[self.rank - 1] if self.rank > 0 else None,
                            eps[self.rank + 1] if self.rank + 1 < self.world else None)
        dist.barrier()

    def upload_band(self, dem_band, water_band=None):
        self.solver.upload_band(dem_band, water_band)
        self.dist.barrier()  # nobody iterates (and pushes halos) before every stripe has reset its flags

    def upload_band_ptr(self, dem_ptr, water_ptr):
        self.solver.upload_band_ptr(dem_ptr, water_ptr)
        self.dist.barrier()

    def run_block(self, n_iters: int = 1000) -> _solver.BlockResult:
        r = self.solver.run_block(n_iters)
        allr = [None] * self.world
        self.dist.all_gather_object(allr, r)
        out = combine_block_results(allr)
        n = getattr(self.solver, "n_outlets", 0)
        if self.solver.module == _solver.DRAIN and n > 1:
            # an outlet set: the single-solver total is the per-outlet totals added in outlet order, in the solver's
            # precision (include/wdpm_b200.h); each total lives on one stripe, so gather them and add in that order
            acc = self.solver.np_dtype(0)
            for v in self.outlet_drains(n).astype(self.solver.np_dtype):
                acc = self.solver.np_dtype(acc + v)
            out.total_drain = float(acc)
        return out

    def set_outlets(self, outlets):
        """Every stripe takes the whole set (padded (row, col) of the whole DEM)."""
        self.solver.set_outlets(outlets)

    def seed_outlet_drains(self):
        self.solver.seed_outlet_drains()

    def set_outlet_drains(self, values):
        """Every stripe takes the whole array; the one that owns an outlet's row keeps its total."""
        self.solver.set_outlet_drains(values)

    def checkpoint_arm(self):
        self.solver.checkpoint_arm()

    def checkpoint_wait(self):
        """This rank's capture: its owned rows and its share of the totals (0 for outlets of other stripes)."""
        return self.solver.checkpoint_wait()

    def outlet_drains(self, n: int) -> np.ndarray:
        """Per-outlet totals of the whole DEM: each is kept by the stripe that owns the outlet's row (0 elsewhere),
        so the element-wise sum over the stripes is exact."""
        mine = self.solver.get_outlet_drains(n)
        parts = [None] * self.world
        self.dist.all_gather_object(parts, mine)
        return np.sum(parts, axis=0)

    def close(self):
        self.dist.barrier()
        self.solver.close()
