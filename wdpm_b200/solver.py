"""ctypes mirror of include/wdpm_b200.h.

Host-side plumbing only: every method forwards to the C ABI of
libwdpm_b200.so, which owns the device memory and launches the CUDA kernels.
There is no fallback: if the library is missing or no GPU is present the calls
raise.
"""
from __future__ import annotations

import ctypes as C
import dataclasses
from pathlib import Path

import numpy as np

ADD, SUBTRACT, DRAIN = 0, 1, 2
F32, F64 = 0, 1
KERNEL_AUTO, KERNEL_COLOUR, KERNEL_FUSED, KERNEL_RESIDENT = 0, 1, 2, 3
# update schedule (WDPM_SCHEDULE_* in include/wdpm_b200.h): the reference's OpenCL branch, or its serial branch
SCHED_OPENCL, SCHED_SERIAL = 0, 1
MAX_OUTLETS = 1 << 20  # WDPM_MAX_OUTLETS: the largest outlet set wdpm_set_outlets takes
MODULES = {"add": ADD, "subtract": SUBTRACT, "drain": DRAIN}
# the tiling AUTO picks for large fp64 Add/Subtract grids (kDefaultVariantF64 in csrc/solver.cu); tests and
# smoke() name it to exercise the production kernel on small grids
PRODUCTION_FUSED_VARIANT_F64 = 17   # warp-autonomous kernel (k_fused_wa), all three modules
PRODUCTION_FUSED_VARIANT_F32 = 16

_PKG = Path(__file__).resolve().parent


class WdpmError(RuntimeError):
    def __init__(self, code: int, message: str):
        super().__init__(f"wdpm_b200 error {code}: {message}")
        self.code = code


class _Config(C.Structure):
    _fields_ = [("struct_size", C.c_uint32), ("rows", C.c_int32), ("cols", C.c_int32), ("nodata", C.c_double),
                ("dtype", C.c_int32), ("module", C.c_int32), ("zero_threshold", C.c_double), ("device", C.c_int32),
                ("kernel", C.c_int32), ("stripe_row0", C.c_int32), ("stripe_rows", C.c_int32),
                ("iters_per_launch", C.c_int32), ("fused_variant", C.c_int32), ("fused_chunk_rows", C.c_int32),
                ("schedule", C.c_int32), ("reserved", C.c_int32 * 4)]


class _BlockResult(C.Structure):
    _fields_ = [("max_diff", C.c_double), ("masked_sum", C.c_double), ("total_drain", C.c_double),
                ("wet_cells", C.c_int64), ("iterations", C.c_int32), ("launches", C.c_int32),
                ("block_ms", C.c_float), ("iterate_ms", C.c_float)]


class _Info(C.Structure):
    _fields_ = [("device_bytes", C.c_int64), ("kernel_launches", C.c_int64), ("kernel", C.c_int32),
                ("strip_cols", C.c_int32), ("window_cols", C.c_int32), ("chunk_rows", C.c_int32),
                ("grid_ctas", C.c_int32), ("cta_threads", C.c_int32), ("smem_bytes", C.c_int32),
                ("iters_per_launch", C.c_int32), ("sm_count", C.c_int32), ("warp_autonomous", C.c_int32), ("reserved", C.c_int32 * 6)]


@dataclasses.dataclass
class BlockResult:
    max_diff: float
    masked_sum: float
    total_drain: float
    wet_cells: int
    iterations: int
    launches: int
    block_ms: float
    iterate_ms: float


_lib = None


def library_path() -> Path:
    # WDPM_B200_LIB: developer hook (scripts/timeline.py loads an instrumented build of the same sources)
    import os
    return Path(os.environ.get("WDPM_B200_LIB") or (_PKG / "libwdpm_b200.so"))


def load_library() -> C.CDLL:
    """Load libwdpm_b200.so (build it with `python -m wdpm_b200.build`). Fails loudly if absent."""
    global _lib
    if _lib is None:
        path = library_path()
        if not path.exists():
            raise FileNotFoundError(f"{path} is missing: run `python -m wdpm_b200.build` (no CPU fallback exists)")
        lib = C.CDLL(str(path))
        lib.wdpm_last_error.restype = C.c_char_p
        _lib = lib
    return _lib


def _check(rc: int):
    if rc != 0:
        raise WdpmError(rc, load_library().wdpm_last_error().decode())


def _np_dtype(dtype: int):
    return np.float64 if dtype == F64 else np.float32


def fused_variant_info(variant: int, dtype: int) -> dict | None:
    lib = load_library()
    vals = [C.c_int32() for _ in range(5)]
    rc = lib.wdpm_fused_variant_info(C.c_int32(variant), C.c_int32(dtype), *[C.byref(v) for v in vals])
    if rc != 0:
        return None
    keys = ("window_cols", "strip_cols", "iters_per_launch", "cta_threads", "smem_bytes")
    return dict(zip(keys, (v.value for v in vals)))


class Solver:
    """One GPU-resident redistribution solver (mirror of wdpm_solver)."""

    def __init__(self, rows: int, cols: int, nodata: float, module: int, dtype: int = F64, zero_threshold: float = 0.0,
                 device: int = 0, kernel: int = KERNEL_AUTO, iters_per_launch: int = 0, fused_variant: int = 0,
                 fused_chunk_rows: int = 0, schedule: int = SCHED_OPENCL, _stripe: tuple | None = None):
        self._lib = load_library()
        self._h = C.c_void_p()
        cfg = _Config()
        cfg.struct_size = C.sizeof(_Config)
        cfg.rows, cfg.cols, cfg.nodata = rows, cols, nodata
        cfg.dtype, cfg.module, cfg.zero_threshold = dtype, module, zero_threshold
        cfg.device, cfg.kernel = device, kernel
        cfg.stripe_row0, cfg.stripe_rows = _stripe if _stripe else (0, 0)
        cfg.iters_per_launch, cfg.fused_variant, cfg.fused_chunk_rows = iters_per_launch, fused_variant, fused_chunk_rows
        cfg.schedule = schedule
        _check(self._lib.wdpm_create(C.byref(cfg), C.byref(self._h)))
        self.rows, self.cols, self.dtype, self.module, self.nodata = rows, cols, dtype, module, nodata
        self.schedule = schedule
        self.np_dtype = _np_dtype(dtype)
        self.owned_rows = self.stripe.owned_rows if _stripe else rows  # interior rows download_water returns

    # -- lifetime ---------------------------------------------------------
    def close(self):
        if getattr(self, "_h", None) and self._h.value:
            self._lib.wdpm_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    # -- data -------------------------------------------------------------
    def _host(self, a, name):
        a = np.ascontiguousarray(a, dtype=self.np_dtype)
        if a.shape != (self.rows, self.cols):
            raise ValueError(f"{name} must be {self.rows}x{self.cols}, got {a.shape}")
        return a

    def upload(self, dem, water=None):
        d = self._host(dem, "dem")
        w = None if water is None else self._host(water, "water")
        _check(self._lib.wdpm_upload(self._h, d.ctypes.data_as(C.c_void_p), None if w is None else w.ctypes.data_as(C.c_void_p)))

    def upload_ptr(self, dem_ptr: int, water_ptr: int | None):
        """Upload from raw host addresses (e.g. pinned torch tensors)."""
        _check(self._lib.wdpm_upload(self._h, C.c_void_p(dem_ptr), C.c_void_p(water_ptr) if water_ptr else None))

    def upload_water(self, water=None):
        w = None if water is None else self._host(water, "water")
        _check(self._lib.wdpm_upload_water(self._h, None if w is None else w.ctypes.data_as(C.c_void_p)))

    def download_water(self, out: np.ndarray | None = None) -> np.ndarray:
        if out is None:
            out = np.empty((self.rows, self.cols), dtype=self.np_dtype)
        assert out.flags.c_contiguous and out.dtype == self.np_dtype and out.shape == (self.rows, self.cols)
        _check(self._lib.wdpm_download_water(self._h, out.ctypes.data_as(C.c_void_p)))
        return out

    def download_water_ptr(self, ptr: int):
        _check(self._lib.wdpm_download_water(self._h, C.c_void_p(ptr)))

    # -- module set-up ----------------------------------------------------
    def apply_add(self, depth_m: float, runoff_fraction: float):
        _check(self._lib.wdpm_apply_add(self._h, C.c_double(depth_m), C.c_double(runoff_fraction)))

    def apply_subtract(self, depth_m: float):
        _check(self._lib.wdpm_apply_subtract(self._h, C.c_double(depth_m)))

    def find_outlet(self):
        r, c, e = C.c_int32(), C.c_int32(), C.c_double()
        _check(self._lib.wdpm_find_outlet(self._h, C.byref(r), C.byref(c), C.byref(e)))
        return r.value, c.value, e.value

    def set_outlet(self, drainrow: int, draincol: int):
        _check(self._lib.wdpm_set_outlet(self._h, C.c_int32(drainrow), C.c_int32(draincol)))
        self.n_outlets = 1

    def set_outlets(self, outlets):
        """A set of outlet cells [(row, col), ...] in padded coordinates of the whole DEM (extension;
        one outlet is the reference's Drain)."""
        rows = (C.c_int32 * len(outlets))(*[int(o[0]) for o in outlets])
        cols = (C.c_int32 * len(outlets))(*[int(o[1]) for o in outlets])
        _check(self._lib.wdpm_set_outlets(self._h, C.c_int32(len(outlets)), rows, cols))
        self.n_outlets = len(outlets)

    def seed_outlet_drains(self):
        """Every outlet's total = max(water at the outlet, 0) (WDPMCL.c:1029 per outlet); on row stripes only the
        stripe that owns the outlet's row keeps a non-zero seed."""
        _check(self._lib.wdpm_seed_outlet_drains(self._h))

    def get_outlet_drains(self, n: int) -> np.ndarray:
        out = np.zeros(n, dtype=np.float64)
        _check(self._lib.wdpm_get_outlet_drains(self._h, out.ctypes.data_as(C.POINTER(C.c_double)), C.c_int32(n)))
        return out

    def set_outlet_drains(self, values):
        """Restore every outlet's total, in the caller's order (on row stripes only the stripe that owns the outlet's
        row keeps it)."""
        v = np.ascontiguousarray(values, dtype=np.float64)
        _check(self._lib.wdpm_set_outlet_drains(self._h, v.ctypes.data_as(C.POINTER(C.c_double)), C.c_int32(v.size)))

    def checkpoint_arm(self):
        """Capture the state the next block starts from (wdpm_checkpoint_arm)."""
        _check(self._lib.wdpm_checkpoint_arm(self._h))

    def checkpoint_wait(self):
        """(water, totals) of the last capture, as copies: the owned interior rows in the solver's precision and the
        outlet totals in the caller's order."""
        w, t, n = C.c_void_p(), C.POINTER(C.c_double)(), C.c_int32()
        _check(self._lib.wdpm_checkpoint_wait(self._h, C.byref(w), C.byref(t), C.byref(n)))
        cells = self.owned_rows * self.cols
        raw = (C.c_char * (cells * np.dtype(self.np_dtype).itemsize)).from_address(w.value)
        water = np.frombuffer(raw, dtype=self.np_dtype).reshape(self.owned_rows, self.cols).copy()
        return water, np.ctypeslib.as_array(t, shape=(n.value,)).copy()

    def quantize_water(self):
        """What a "%f" file hand-over does to the water grid (module chaining; include/wdpm_quantize.h)."""
        _check(self._lib.wdpm_quantize_water(self._h))

    def copy_state_from(self, src: "Solver", dem: bool = True, water: bool = True):
        """Take the elevations and/or the current water grid of another solver of the same DEM, inside HBM."""
        _check(self._lib.wdpm_copy_state(self._h, src._h, C.c_int32((1 if dem else 0) | (2 if water else 0))))

    def set_total_drain(self, v: float):
        _check(self._lib.wdpm_set_total_drain(self._h, C.c_double(v)))

    def get_total_drain(self) -> float:
        v = C.c_double()
        _check(self._lib.wdpm_get_total_drain(self._h, C.byref(v)))
        return v.value

    def get_cell_water(self, row: int, col: int) -> float:
        v = C.c_double()
        _check(self._lib.wdpm_get_cell_water(self._h, C.c_int32(row), C.c_int32(col), C.byref(v)))
        return v.value

    def final_statistics(self):
        """(valid cells, cells with more than 1 mm of water, deepest water in m) over the owned interior cells -
        the order-free part of the reference's final report (WDPMCL.c:1394-1459), computed on the device."""
        nv, nw, md = C.c_int64(), C.c_int64(), C.c_double()
        _check(self._lib.wdpm_final_statistics(self._h, C.byref(nv), C.byref(nw), C.byref(md)))
        return nv.value, nw.value, md.value

    def water_checksum(self) -> int:
        """Order-free 64-bit checksum of the owned interior water cells (position-weighted bit patterns, mod 2^64)."""
        v = C.c_uint64()
        _check(self._lib.wdpm_water_checksum(self._h, C.byref(v)))
        return int(v.value)

    # -- the hot path -----------------------------------------------------
    def run_block(self, n_iters: int = 1000) -> BlockResult:
        r = _BlockResult()
        _check(self._lib.wdpm_run_block(self._h, C.c_int32(n_iters), C.byref(r)))
        return BlockResult(r.max_diff, r.masked_sum, r.total_drain, r.wet_cells, r.iterations, r.launches, r.block_ms, r.iterate_ms)

    def block_begin(self):
        """Threshold + snapshot, non-blocking (hosts that feed several stripe solvers round-robin)."""
        _check(self._lib.wdpm_block_begin(self._h))

    def block_enqueue(self, n_iters: int):
        _check(self._lib.wdpm_block_enqueue(self._h, C.c_int32(n_iters)))

    def block_end(self) -> BlockResult:
        r = _BlockResult()
        _check(self._lib.wdpm_block_end(self._h, C.byref(r)))
        return BlockResult(r.max_diff, r.masked_sum, r.total_drain, r.wet_cells, r.iterations, r.launches, r.block_ms, r.iterate_ms)

    def iterate(self, n_iters: int):
        _check(self._lib.wdpm_iterate(self._h, C.c_int32(n_iters)))

    def subpass(self, oi: int, oj: int):
        _check(self._lib.wdpm_subpass(self._h, C.c_int32(oi), C.c_int32(oj)))

    def set_stream(self, cuda_stream: int | None):
        _check(self._lib.wdpm_set_stream(self._h, C.c_void_p(cuda_stream) if cuda_stream else None))

    def synchronize(self):
        _check(self._lib.wdpm_synchronize(self._h))

    def info(self) -> dict:
        i = _Info()
        _check(self._lib.wdpm_get_info(self._h, C.byref(i)))
        return {k: getattr(i, k) for k, _ in _Info._fields_ if k != "reserved"}
