"""CPU: the reference arm of bench.py (the unmodified reference program on a bounded sample) - no GPU needed."""
import json
import os
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

ROOT = Path(__file__).resolve().parent.parent


def _ref_binary():
    sys.path.insert(0, str(ROOT))
    from oracle import pyoracle
    pyoracle.build()
    return pyoracle.ref_binary()


def test_reference_arm_runs_the_unmodified_program_on_all_cores():
    """Under torch.distributed.run OMP_NUM_THREADS is 1 (VERDICT r1: the N >= 2 reference numbers ran on one thread);
    the arm must set the thread count itself, keep the workload's config and say what it sampled."""
    if _ref_binary() is None:
        pytest.skip("oracle/_ref/WDPMCL_ref not built (needs the reference checkout at build time: ../reference or $WDPM_REFERENCE)")
    env = dict(os.environ, OMP_NUM_THREADS="1", RANK="0", WORLD_SIZE="2")
    res = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "0",
                          "--sample-size-ref", "96"], capture_output=True, text=True, env=env, timeout=600)
    assert res.returncode == 0, res.stderr[-2000:]
    line = json.loads(res.stdout.strip().splitlines()[-1])
    cores = len(os.sched_getaffinity(0))
    assert line["impl"] == "reference" and line["cpu_baseline"]["kind"] == "reference"
    assert line["cpu_baseline"]["cores"] == cores
    assert line["config"]["rows"] == 32768 and "2 row stripes" in line["config"]["partition"]  # the workload's config, as our arm prints it
    assert "96x96" in line["sample"] and "UNMODIFIED" in line["sample"]
    assert line["value"] > 0 and line["e2e"]["h2d_bytes_per_step"] == 0 and line["gpu_launches"] == 0


def test_dump_sample_is_fixed_and_fits_the_budget():
    """bench.py --dump-outputs: the sampled cells are the same in every run, and what is written stays under 64 MB."""
    sys.path.insert(0, str(ROOT))
    import bench
    small = bench.sample_cells(300, 500)
    assert np.array_equal(small, np.arange(300 * 500))
    a, b = bench.sample_cells(32768, 32768), bench.sample_cells(32768, 32768)
    assert np.array_equal(a, b)
    assert len(a) > 0.99 * bench.DUMP_CELLS and np.all(np.diff(a) > 0) and a[0] >= 0 and a[-1] < 32768 * 32768
    assert len(a) * 8 + 4 * 8 <= 64 << 20


@pytest.mark.parametrize("n_stripes", [1, 3, 8])
def test_dump_sample_gathered_from_stripes_is_the_whole_grid_sample(n_stripes):
    """With row stripes each rank takes the sampled cells of its owned rows; rank 0 concatenates them in row order."""
    sys.path.insert(0, str(ROOT))
    import bench
    from wdpm_b200.stripes import plan_stripes
    rows = cols = 2100  # above DUMP_CELLS: the sampled form
    grid = np.random.default_rng(2).random((rows, cols))
    idx = bench.sample_cells(rows, cols)
    assert len(idx) < rows * cols
    parts = [(st.owned_row0, bench.sampled_rows(idx, cols, st.owned_row0, grid[st.owned_row0:st.owned_row0 + st.owned_rows]))
             for st in plan_stripes(rows, n_stripes)]
    water = np.concatenate([p[1] for p in sorted(parts, key=lambda p: p[0])])
    assert np.array_equal(water, grid.ravel()[idx])


def test_reference_arm_other_ranks_stay_silent():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2")
    res = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "0"],
                         capture_output=True, text=True, env=env, timeout=120)
    assert res.returncode == 0 and res.stdout.strip() == ""
