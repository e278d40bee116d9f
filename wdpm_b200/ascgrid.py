"""ESRI ASCII (.asc) grids, as WDPM reads and writes them.

Test/bench-side helper (numpy). The drop-in command-line host has its own C
reader/writer (wdpm_b200/host/); this module mirrors the same format rules so
Python tests can produce and inspect the files the reference consumes:

* six header lines "NAME value", taken positionally as ncols, nrows, xll, yll,
  cellsize, nodata (/root/reference/src/WDPMCL.c:542-555);
* data in row-major order, any whitespace (fscanf "%lf", :1569-1574);
* output header formats %d %d %14.6f %14.6f %9.6f %14.6f and every value written
  as "%f " with a newline per row (:1538-1552).
"""
from __future__ import annotations

import dataclasses
import gzip
import io
from pathlib import Path

import numpy as np


@dataclasses.dataclass
class AscHeader:
    names: list[str]
    ncols: int
    nrows: int
    xll: float
    yll: float
    cellsize: float
    nodata: float

    @staticmethod
    def default(nrows: int, ncols: int, cellsize: float = 10.0, nodata: float = -99999.0) -> "AscHeader":
        return AscHeader(["NCOLS", "NROWS", "XLLCORNER", "YLLCORNER", "CELLSIZE", "NODATA_VALUE"],
                         ncols, nrows, 0.0, 0.0, cellsize, nodata)


def _open_text(path):
    path = Path(path)
    if path.suffix == ".gz":
        return io.TextIOWrapper(gzip.open(path, "rb"))
    return open(path, "r")


def read_asc(path, dtype=np.float64) -> tuple[AscHeader, np.ndarray]:
    with _open_text(path) as f:
        tokens = f.read().split()
    names = [tokens[2 * i] for i in range(6)]
    vals = [float(tokens[2 * i + 1]) for i in range(6)]
    hdr = AscHeader(names, int(vals[0]), int(vals[1]), vals[2], vals[3], vals[4], vals[5])
    data = np.array(tokens[12:12 + hdr.nrows * hdr.ncols], dtype=np.float64)
    if data.size != hdr.nrows * hdr.ncols:
        raise ValueError(f"{path}: expected {hdr.nrows * hdr.ncols} values, found {data.size}")
    return hdr, data.reshape(hdr.nrows, hdr.ncols).astype(dtype, copy=False)


def write_asc(path, hdr: AscHeader, grid: np.ndarray) -> None:
    """Byte-compatible with write_gis (/root/reference/src/WDPMCL.c:1533-1554)."""
    out = io.StringIO()
    out.write("%s %d\n" % (hdr.names[0], hdr.ncols))
    out.write("%s %d\n" % (hdr.names[1], hdr.nrows))
    out.write("%s %14.6f\n" % (hdr.names[2], hdr.xll))
    out.write("%s %14.6f\n" % (hdr.names[3], hdr.yll))
    out.write("%s %9.6f\n" % (hdr.names[4], hdr.cellsize))
    out.write("%s %14.6f\n" % (hdr.names[5], hdr.nodata))
    g = np.asarray(grid, dtype=np.float64)
    for row in g:
        out.write("".join("%f " % v for v in row))
        out.write("\n")
    Path(path).write_text(out.getvalue())


def rim_outlets(dem: np.ndarray, nodata: float) -> list[tuple[int, int]]:
    """The outlet set "rim" of the command-line host (WDPM_B200_OUTLETS=rim): every cell with dem > nodata in the
    first or last row or column of the (unpadded) DEM, in row-major order, as 1-based padded (row, col)."""
    R, C = dem.shape
    on_rim = np.zeros((R, C), dtype=bool)
    on_rim[0, :] = on_rim[-1, :] = on_rim[:, 0] = on_rim[:, -1] = True
    r, c = np.nonzero(on_rim & (dem > nodata))
    return list(zip((r + 1).tolist(), (c + 1).tolist()))


def pad_grid(a: np.ndarray, fill) -> np.ndarray:
    """(R, C) -> (R+2, C+2) with a one-cell border of `fill` (WDPMCL.c:795-807)."""
    out = np.full((a.shape[0] + 2, a.shape[1] + 2), fill, dtype=a.dtype)
    out[1:-1, 1:-1] = a
    return out
