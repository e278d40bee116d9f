"""GPU (-m gpu): bench.py --dump-outputs writes what the last timed step computed, the same in every run."""
import json
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = Path(__file__).resolve().parent.parent
SCALARS = ["masked_sum.npy", "max_diff.npy", "total_drain.npy", "wet_cells.npy"]


def _bench(out: Path, warmup: int, steps: int, size: int = 4096) -> dict:
    res = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--size", str(size), "--steps", str(steps), "--warmup", str(warmup),
                          "--no-cpu-baseline", "--dump-outputs", str(out)], capture_output=True, text=True, timeout=900)
    assert res.returncode == 0, res.stdout[-1000:] + res.stderr[-2000:]
    return json.loads(res.stdout.strip().splitlines()[-1])


def _same(a: Path, b: Path) -> bool:
    names = sorted(p.name for p in a.iterdir())
    return names == sorted(p.name for p in b.iterdir()) and all(np.array_equal(np.load(a / n), np.load(b / n)) for n in names)


def test_dump_outputs_are_the_last_timed_step(cuda_lib, tmp_path):
    """4096^2 is above bench.DUMP_CELLS (the sampled form). Same arguments: same files. Warm-up 1 + 3 timed steps and
    warm-up 2 + 2 timed steps end the timed loop in the same state but run different end-to-end phases after it (one
    block per timed step, at most 5), so equal files show the dump is taken when the timed steps end."""
    sys.path.insert(0, str(ROOT))
    import bench
    a, b, c, d = (tmp_path / x for x in "abcd")
    la, lb, lc, ld = _bench(a, 1, 2), _bench(b, 1, 2), _bench(c, 1, 3), _bench(d, 2, 2)
    assert la["steps"] == lb["steps"] == ld["steps"] == 2 and lc["steps"] == 3
    assert sorted(p.name for p in a.iterdir()) == sorted(SCALARS + ["water_sample.npy"])
    assert sum(p.stat().st_size for p in a.iterdir()) <= 64 << 20
    assert _same(a, b) and la["state"]["checksum"] == lb["state"]["checksum"]
    assert lc["e2e"]["steps"] != ld["e2e"]["steps"]
    assert _same(c, d) and lc["state"]["checksum"] == ld["state"]["checksum"]
    assert not _same(a, c)  # one more timed step moves the water
    water = np.load(a / "water_sample.npy")
    assert water.dtype == np.float64 and water.shape == bench.sample_cells(4096, 4096).shape
    assert np.load(a / "max_diff.npy")[0] == la["state"]["max_diff"]
    assert np.load(a / "wet_cells.npy")[0] == round(la["state"]["wet_fraction"] * 4096 * 4096)


def test_dump_outputs_whole_grid_when_small(cuda_lib, tmp_path):
    """At or below bench.DUMP_CELLS the whole water grid is written, in the run's precision."""
    line = _bench(tmp_path, 1, 1, size=2048)
    assert sorted(p.name for p in tmp_path.iterdir()) == sorted(SCALARS + ["water.npy"])
    water = np.load(tmp_path / "water.npy")
    assert water.dtype == np.float64 and water.shape == (2048, 2048)
    assert int(np.count_nonzero(water > 0)) == round(line["state"]["wet_fraction"] * 2048 * 2048)
