import gzip
import shutil
import sys
from pathlib import Path

import numpy as np
import pytest

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(Path(__file__).resolve().parent))
GOLDEN = Path(__file__).resolve().parent / "golden"


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


@pytest.fixture(scope="session")
def oracle():
    from oracle import pyoracle
    pyoracle.build()
    return pyoracle.Oracle()


@pytest.fixture(scope="session")
def refcl():
    from oracle import pyoracle
    pyoracle.build()
    if not pyoracle.RefCL.available():
        pytest.skip("oracle/_ref/librunoffcl_ref.so not built (needs the reference checkout at build time: ../reference or $WDPM_REFERENCE)")
    return pyoracle.RefCL()


@pytest.fixture(scope="session")
def basin5():
    from wdpm_b200 import ascgrid
    return ascgrid.read_asc(GOLDEN / "basin5.asc.gz")


@pytest.fixture(scope="session")
def cuda_lib():
    """Build (if stale) and load the CUDA library; GPU tests use it through wdpm_b200.Solver."""
    from wdpm_b200 import build, solver
    build.build_library()
    return solver.load_library()


def golden_text(name: str) -> str:
    with gzip.open(GOLDEN / name, "rt") as f:
        return f.read()


def gunzip_to(name: str, dst: Path) -> Path:
    with gzip.open(GOLDEN / name, "rb") as f, open(dst, "wb") as g:
        shutil.copyfileobj(f, g)
    return dst


def random_case(rng, rows, cols, dtype, nodata=-99999.0, wet_fraction=0.7, nodata_fraction=0.08, depth=0.5):
    """Padded (dem, water) pair with relief, NODATA holes and dry patches."""
    from wdpm_b200 import ascgrid
    d = (500 + 3 * rng.standard_normal((rows, cols))).round(4)
    d[rng.uniform(size=d.shape) < nodata_fraction] = nodata
    D = ascgrid.pad_grid(d.astype(dtype), dtype(nodata))
    W = np.where(D > nodata, rng.uniform(0, depth, D.shape), 0).astype(dtype)
    W[rng.uniform(size=D.shape) > wet_fraction] = 0
    return D, W
