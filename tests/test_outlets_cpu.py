"""Drain outlet sets without a GPU: the rim order, the ctypes mirror against the header, and the command-line
host's checks of WDPM_B200_OUTLETS, which refuse a bad set before any solver is created."""
import os
import re
import subprocess
from pathlib import Path

import numpy as np
import pytest

from conftest import gunzip_to

ROOT = Path(__file__).resolve().parent.parent
NODATA = -99999.0


def test_rim_outlets_order_and_validity():
    from wdpm_b200 import ascgrid
    rng = np.random.default_rng(9)
    d = rng.uniform(1, 2, (7, 9))
    d[0, 3] = d[6, 0] = d[4, 8] = d[3, 4] = NODATA
    want = [(i + 1, j + 1) for i in range(7) for j in range(9)
            if (i in (0, 6) or j in (0, 8)) and d[i, j] > NODATA]
    assert ascgrid.rim_outlets(d, NODATA) == want
    assert (1, 4) not in want and (5, 9) not in want and len(want) == 2 * 9 + 2 * 5 - 3


def test_mirror_declares_the_outlet_entry_points():
    from wdpm_b200 import MAX_OUTLETS, Solver
    header = (ROOT / "include" / "wdpm_b200.h").read_text()
    m = re.search(r"#define WDPM_MAX_OUTLETS (\d+)", header)
    assert m and int(m.group(1)) == MAX_OUTLETS == 1 << 20
    assert "int wdpm_seed_outlet_drains(wdpm_solver *s);" in header
    assert "wdpm_seed_outlet_drains" in (ROOT / "wdpm_b200" / "solver.py").read_text()
    assert callable(getattr(Solver, "seed_outlet_drains", None))


@pytest.fixture(scope="module")
def host_bin():
    from wdpm_b200 import build
    build.build_library()
    return build.build_host()


def _grid(path, rows, cols, values, nodata=-9999.0):
    from wdpm_b200 import ascgrid
    ascgrid.write_asc(path, ascgrid.AscHeader.default(rows, cols, nodata=nodata), values)
    return path


def _drain(host_bin, tmp_path, spec):
    dem = gunzip_to("basin5.asc.gz", tmp_path / "basin5.asc")
    env = dict(os.environ, WDPM_B200_OUTLETS=str(spec))
    argv = ["drain", str(dem), str(dem), str(tmp_path / "o.asc"), "NULL", "0.1", "1.0", "1", "1", "0.005", "0"]
    return subprocess.run([str(host_bin)] + argv, capture_output=True, text=True, env=env, timeout=120)


@pytest.fixture(scope="module")
def basin5_dem():
    from wdpm_b200 import ascgrid
    from conftest import GOLDEN
    return ascgrid.read_asc(GOLDEN / "basin5.asc.gz")


def test_cli_refuses_an_outlet_grid_of_another_size(host_bin, tmp_path, basin5_dem):
    hdr, d = basin5_dem
    res = _drain(host_bin, tmp_path, _grid(tmp_path / "g.asc", hdr.nrows + 1, hdr.ncols, np.ones((hdr.nrows + 1, hdr.ncols))))
    assert res.returncode == 1 and "ncols and nrows differ" in res.stderr
    assert "solver" not in res.stdout + res.stderr  # refused before any solver exists


def test_cli_outlet_grid_rules(host_bin, tmp_path, basin5_dem):
    """Only values > 0 that are not the grid's NODATA mark outlets; an outlet on a DEM NODATA cell is refused."""
    hdr, d = basin5_dem
    g = np.zeros_like(d)
    g[:5, :5] = -9999.0   # the grid's NODATA
    g[5:9, :5] = -1.0     # not > 0
    res = _drain(host_bin, tmp_path, _grid(tmp_path / "none.asc", hdr.nrows, hdr.ncols, g))
    assert res.returncode == 1 and "no outlet" in res.stderr
    i, j = map(int, np.argwhere(d <= hdr.nodata)[0])
    g[i, j] = 2.0
    res = _drain(host_bin, tmp_path, _grid(tmp_path / "bad.asc", hdr.nrows, hdr.ncols, g))
    assert res.returncode == 1 and "dem <= nodata" in res.stderr
