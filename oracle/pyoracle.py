"""TEST INFRASTRUCTURE - ctypes bindings for the CPU oracle and the reference shims.

* `Oracle`   : oracle/_build/libwdpm_oracle.so - this repo's C restatement
               (oracle/wdpm_oracle_impl.h), padded ROW-major grids.
* `RefCL`    : oracle/_ref/librunoffcl_ref.so - the verbatim reference kernel file
               compiled as C (oracle/ref_shim), padded COLUMN-major grids exactly
               as WDPMCL.c:1129-1134 flattens them. Present only when the oracle
               was built with a checkout of the reference (CentreForHydrology/WDPM)
               at reference_dir(); the repository does not carry its sources.
* `ref_binary()`: path of oracle/_ref/WDPMCL_ref, the unmodified reference host
               linked against the minicl stand-in runtime.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
from pathlib import Path

import numpy as np

HERE = Path(__file__).resolve().parent
ADD, SUBTRACT, DRAIN = 0, 1, 2
SCHED_OPENCL, SCHED_SERIAL = 0, 1
MODULES = {"add": ADD, "subtract": SUBTRACT, "drain": DRAIN}


def reference_dir() -> Path | None:
    """The reference checkout: WDPM_REFERENCE if set, else a directory `reference` beside this repository.
    None when it is absent or cannot be read (an unreadable location is no reference, not an error)."""
    ref = Path(os.environ.get("WDPM_REFERENCE") or HERE.parent.parent / "reference")
    try:
        return ref if (ref / "src" / "runoff.cl").is_file() else None
    except OSError:
        return None


def build(force: bool = False) -> None:
    """Compile the oracle (and oracle/_ref when the reference checkout, reference_dir(), is there)."""
    target = HERE / "_build" / "libwdpm_oracle.so"
    ref = reference_dir()
    if force or not target.exists() or ref is not None:
        subprocess.run(["make", "-C", str(HERE), f"REF={ref or ''}"], check=True, capture_output=True)


def _sfx(dtype) -> tuple[str, type]:
    dtype = np.dtype(dtype)
    if dtype == np.float64:
        return "_f64", C.c_double
    if dtype == np.float32:
        return "_f32", C.c_float
    raise TypeError(dtype)


def _ptr(a: np.ndarray):
    assert a.flags.c_contiguous
    return a.ctypes.data_as(C.c_void_p)


class Oracle:
    def __init__(self):
        path = HERE / "_build" / "libwdpm_oracle.so"
        if not path.exists():
            build()
        self.lib = C.CDLL(str(path))
        self.lib.wdpm_oracle_num_threads.restype = C.c_int

    @property
    def threads(self) -> int:
        return int(self.lib.wdpm_oracle_num_threads())

    def iterate(self, w: np.ndarray, d: np.ndarray, nodata: float, module: int, n_iters: int,
                schedule: int = SCHED_OPENCL, outlet=(0, 0), totaldrain: float = 0.0) -> float:
        """In place on padded row-major `w`; returns the updated totaldrain."""
        sfx, ct = _sfx(w.dtype)
        assert d.dtype == w.dtype and w.shape == d.shape
        R, Cc = w.shape[0] - 2, w.shape[1] - 2
        td = np.array([totaldrain], dtype=w.dtype)
        fn = getattr(self.lib, "wdpm_oracle_iterate" + sfx)
        fn.restype = None
        fn(_ptr(w), _ptr(d), C.c_int(R), C.c_int(Cc), ct(nodata), C.c_int(module), C.c_int(schedule),
           C.c_int(n_iters), C.c_int(outlet[0]), C.c_int(outlet[1]), _ptr(td))
        return float(td[0])

    def subpass(self, w, d, nodata, module, oi, oj, schedule=SCHED_OPENCL, outlet=(0, 0),
                totaldrain: float = 0.0) -> float:
        sfx, ct = _sfx(w.dtype)
        R, Cc = w.shape[0] - 2, w.shape[1] - 2
        td = np.array([totaldrain], dtype=w.dtype)
        fn = getattr(self.lib, "wdpm_oracle_subpass" + sfx)
        fn.restype = None
        fn(_ptr(w), _ptr(d), C.c_int(R), C.c_int(Cc), ct(nodata), C.c_int(module), C.c_int(schedule),
           C.c_int(oi), C.c_int(oj), C.c_int(outlet[0]), C.c_int(outlet[1]), _ptr(td))
        return float(td[0])

    def block(self, w, d, nodata, module, thres, n_iters, schedule=SCHED_OPENCL, outlet=(0, 0),
              totaldrain: float = 0.0):
        """One convergence block in place; returns (max_diff, masked_sum, totaldrain)."""
        sfx, ct = _sfx(w.dtype)
        R, Cc = w.shape[0] - 2, w.shape[1] - 2
        old = np.empty_like(w)
        td = np.array([totaldrain], dtype=w.dtype)
        md, ms = C.c_double(0), C.c_double(0)
        fn = getattr(self.lib, "wdpm_oracle_block" + sfx)
        fn.restype = None
        fn(_ptr(w), _ptr(old), _ptr(d), C.c_int(R), C.c_int(Cc), ct(nodata), C.c_int(module),
           C.c_int(schedule), ct(thres), C.c_int(n_iters), C.c_int(outlet[0]), C.c_int(outlet[1]),
           _ptr(td), C.byref(md), C.byref(ms))
        return md.value, ms.value, float(td[0])

    def iterate_outlets(self, w: np.ndarray, d: np.ndarray, nodata: float, n_iters: int, outlets, totals=None):
        """Drain with a SET of outlets (extension; one outlet = the reference). In place on w; returns the
        per-outlet totals (dtype of w)."""
        sfx, ct = _sfx(w.dtype)
        R, Cc = w.shape[0] - 2, w.shape[1] - 2
        rows = np.ascontiguousarray([o[0] for o in outlets], dtype=np.int32)
        cols = np.ascontiguousarray([o[1] for o in outlets], dtype=np.int32)
        td = np.zeros(len(outlets), dtype=w.dtype) if totals is None else np.ascontiguousarray(totals, dtype=w.dtype).copy()
        fn = getattr(self.lib, "wdpm_oracle_iterate_outlets" + sfx)
        fn.restype = C.c_int
        rc = fn(_ptr(w), _ptr(d), C.c_int(R), C.c_int(Cc), ct(nodata), C.c_int(n_iters), C.c_int(len(outlets)),
                _ptr(rows), _ptr(cols), _ptr(td))
        assert rc == 0
        return td

    def find_outlet(self, d):
        sfx, _ = _sfx(d.dtype)
        R, Cc = d.shape[0] - 2, d.shape[1] - 2
        r, c = C.c_int(0), C.c_int(0)
        fn = getattr(self.lib, "wdpm_oracle_find_outlet" + sfx)
        fn.restype = C.c_int
        ok = fn(_ptr(d), C.c_int(R), C.c_int(Cc), C.byref(r), C.byref(c))
        return (r.value, c.value) if ok else None


class RefCL:
    """Verbatim runoff.cl. Arrays passed in are padded ROW-major; they are flattened
    column-major for the kernels (as WDPMCL.c:1129-1134 does) and restored after."""

    PATH = HERE / "_ref" / "librunoffcl_ref.so"

    @classmethod
    def available(cls) -> bool:
        return cls.PATH.exists()

    def __init__(self):
        self.lib = C.CDLL(str(self.PATH))

    def iterate(self, w: np.ndarray, d: np.ndarray, nodata: float, module: int, n_iters: int,
                outlet=(0, 0), totaldrain: float = 0.0) -> float:
        sfx, ct = _sfx(w.dtype)
        R, Cc = w.shape[0] - 2, w.shape[1] - 2
        wf = np.ascontiguousarray(w.T)  # element (row i, col j) at i + (R+2)*j
        df = np.ascontiguousarray(d.T)
        td = np.array([totaldrain], dtype=w.dtype)
        fn = getattr(self.lib, "refcl_iterate" + sfx)
        fn.restype = None
        fn(C.c_int(module), _ptr(wf), _ptr(df), ct(nodata), C.c_int(R), C.c_int(Cc), C.c_int(n_iters),
           _ptr(td), C.c_int(outlet[0]), C.c_int(outlet[1]))
        w[...] = wf.T
        return float(td[0])


def ref_binary() -> Path | None:
    p = HERE / "_ref" / "WDPMCL_ref"
    return p if p.exists() else None
