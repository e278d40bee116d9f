"""Launched by tests/test_gpu_serial_schedule.py (one process, one GPU).

The serial schedule (WDPM_SCHEDULE_SERIAL) on N in-process stripe solvers of the SAME device running FREE
(wdpm_block_begin / enqueue / end on their own streams - the host never waits between iterations): what orders
their iterations, and the emptying of a Drain outlet's 3x3 neighbourhood after each of them, is only the
device-side halo protocol. The outlet sits on the first stripe border, so the nine cells it empties span two
stripes. The assembled grid, the block's max difference, the wet-cell count and the drained total must equal
those of a single serial-schedule solver bit for bit.

usage: stripes_freerun_serial_check.py N_STRIPES MODULE CHUNK_ROWS ITERS [DTYPE]   -> prints FREERUN_EQUAL or FREERUN_DIFFER <n>
"""
import sys
from pathlib import Path

import numpy as np

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
sys.path.insert(0, str(Path(__file__).resolve().parent))

from conftest import random_case  # noqa: E402
from wdpm_b200 import F32, F64, SCHED_SERIAL, Solver  # noqa: E402
from wdpm_b200.stripes import StripeSolver, connect_in_process, plan_stripes  # noqa: E402

NODATA = -99999.0


def main():
    n_stripes, module, chunk_rows, iters = (int(x) for x in sys.argv[1:5])
    dt = np.float32 if len(sys.argv) > 5 and sys.argv[5] == "f32" else np.float64
    code = F64 if dt == np.float64 else F32
    rng = np.random.default_rng(4242)
    rows, cols = 250, 330
    D, W = random_case(rng, rows, cols, dt, nodata_fraction=0.03, wet_fraction=0.9)
    plan = plan_stripes(rows, n_stripes)
    outlet = (plan[1].row0, cols // 2)
    D[outlet] = dt(480.0)
    dem, w0 = D[1:-1, 1:-1], W[1:-1, 1:-1]

    with Solver(rows, cols, NODATA, module, dtype=code, zero_threshold=1e-4, kernel=2, fused_variant=2, schedule=SCHED_SERIAL) as s:
        s.upload(dem, w0)
        if module == 2:
            s.set_outlet(*outlet)
            s.set_total_drain(0.0)
        ref_res = s.run_block(iters)
        ref = s.download_water()

    ss = [StripeSolver(rows, cols, NODATA, module, st, dtype=code, zero_threshold=1e-4, fused_variant=2, fused_chunk_rows=chunk_rows,
                       schedule=SCHED_SERIAL) for st in plan]
    connect_in_process(ss)
    for s, st in zip(ss, plan):
        s.upload_band(dem[st.band_row0:st.band_row0 + st.band_rows], w0[st.band_row0:st.band_row0 + st.band_rows])
        if module == 2:
            s.set_outlet(*outlet)
            s.set_total_drain(0.0)
    for s in ss:
        s.block_begin()
    done = 0
    while done < iters:  # small slices, round-robin: nothing here blocks
        n = min(5, iters - done)
        for s in ss:
            s.block_enqueue(n)
        done += n
    res = [s.block_end() for s in ss]
    full = np.concatenate([s.download_owned() for s in ss], axis=0)
    for s in ss:
        s.close()
    ndiff = int((full != ref).sum())
    md = max(r.max_diff for r in res)
    td = dt(sum(r.total_drain for r in res))  # the stripes that do not own the outlet's row hold 0
    if (ndiff == 0 and md == ref_res.max_diff and sum(r.wet_cells for r in res) == ref_res.wet_cells
            and td == dt(ref_res.total_drain)):
        print("FREERUN_EQUAL")
    else:
        print(f"FREERUN_DIFFER {ndiff}")


if __name__ == "__main__":
    main()
