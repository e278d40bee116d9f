"""GPU (-m gpu): row stripes at the partition's limits, against the oracle.

A stripe needs at least 9 padded rows, kHaloAbove + kHaloBelow: in a 9-row middle stripe every owned row is exported
(rows 0-5 to the stripe above, rows 6-8 to the stripe below), and with AUTO chunking one chunk of CTAs both exports
upwards and reads the bottom halo, so it counts towards both arrival flags. 9N - 2 rows give N stripes of exactly
9 rows; 9N - 1 and 9N + 1 rows leave a last stripe of 10 and 12 rows (a partial row triple, and a whole extra one).

1. Geometry sweep on one GPU, in-process stripes: N = 2, 3, 4, 8 at those heights and 8 unequal stripes on 203 rows;
   the small k_fused test window (variant 2, AUTO chunking), the production k_fused_wa tiling with one row triple per
   CTA, and AUTO; rows that cross two strip borders; Add / Subtract / Drain in fp64 and fp32; blocks of 5, 7 and 5
   iterations at a zero threshold > 0 (the clean launch) and 12 iterations at threshold 0 (the guarded launch), free
   running and in lockstep. Grid bit for bit, block results, summed checksum and final statistics against exact
   host values.
2. Drain on thin stripes: an outlet set on, above and below every border row and on strip borders; the serial
   schedule's single outlet on each border row of an 8-stripe plan (its 3x3 emptying spans the border), and serial
   Subtract; and the first free-running Drain block of a fresh process, whose kernels must not be loaded behind a
   spinning halo wait.
3. Checkpoints captured on 8 nine-row stripes resume on one solver and on 3 stripes, and the reverse.
4. Several real GPUs, when present: tests/dist_stripes_check.py on nine-row stripes, and the command line with
   WDPM_B200_GPUS=8 against one GPU, on a DEM that takes 8 stripes and on one too small for them.

Every test asserts from info() the kernel and tiling each stripe runs. WDPM_B200_HALO_TIMEOUT_MS is set so that a halo
that never arrives ends as WDPM_E_HALO instead of a wait.
"""
import os
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

from conftest import random_case
from test_cli import _normalise
from test_gpu_checkpoint import CASES, Run, _kernels, _setup
from test_gpu_checkpoint import _case as _ck_case
from test_gpu_production_path import (BLOCK_ITERS, NODATA, THRES, WA_VARIANT, _check_block, _code, _final_stats_ref, _same_bits,
                                      _stripes_lockstep, _tiling, _variant_tiling, exact_checksum, ordered_sum, oracle_block_outlets,
                                      reduction_chain)

pytestmark = pytest.mark.gpu

HALO_TIMEOUT_MS = "20000"
GEOMETRIES = [(n, 9 * n + d) for n in (2, 3, 4, 8) for d in (-2, -1, 1)] + [(8, 203)]
TILINGS = ("small", "wa", "auto")


@pytest.fixture(autouse=True)
def _halo_timeout(monkeypatch):
    monkeypatch.setenv("WDPM_B200_HALO_TIMEOUT_MS", HALO_TIMEOUT_MS)


def _variant(tiling, dt):
    return 2 if tiling == "small" else WA_VARIANT[dt]


def _tiling_kw(tiling, dt):
    """small: the k_fused test window with AUTO chunking; wa: the production k_fused_wa tiling, one row triple per
    CTA (many CTAs export upwards); auto: the solver's own choice for a stripe."""
    if tiling == "small":
        return dict(fused_variant=2)
    if tiling == "wa":
        return dict(fused_variant=WA_VARIANT[dt], fused_chunk_rows=3)
    return {}


def _cols(tiling, dt):
    """A row crosses two strip borders of the tiling: three strips, the last one partial."""
    return 2 * _variant_tiling(_variant(tiling, dt), dt)["strip_cols"] + 5


def _assert_stripe_tiling(t, tiling, dt):
    from wdpm_b200 import KERNEL_FUSED
    i, st = t.info(), t.stripe
    sc = i["strip_cols"]
    assert i["kernel"] == KERNEL_FUSED and _tiling(i) == _variant_tiling(_variant(tiling, dt), dt), (tiling, i)
    assert i["warp_autonomous"] == (tiling != "small"), i
    n_strips, triples = -(-(t.cols + 2) // sc), (st.rows + 2) // 3
    assert n_strips == 3, i
    assert i["grid_ctas"] == n_strips * -(-triples // (i["chunk_rows"] // 3)), (st, i)
    if tiling == "wa":
        assert i["chunk_rows"] == 3, i
    elif st.rows <= 12:
        assert i["chunk_rows"] >= st.rows, (st, i)   # one chunk exports upwards and reads the bottom halo


class Stripes:
    """N in-process stripe solvers on one GPU."""

    def __init__(self, rows, cols, mod, dt, n, thres, tiling, schedule=0):
        from wdpm_b200.stripes import StripeSolver, connect_in_process, plan_stripes
        self.plan, self.dt, self.cols = plan_stripes(rows, n), dt, cols
        self.ss = [StripeSolver(rows, cols, NODATA, mod, st, dtype=_code(dt), zero_threshold=thres, schedule=schedule,
                                **_tiling_kw(tiling, dt)) for st in self.plan]
        for t in self.ss:
            _assert_stripe_tiling(t, tiling, dt)
        connect_in_process(self.ss)

    def upload(self, D, W, outlets=None):
        dem, w = D[1:-1, 1:-1], W[1:-1, 1:-1]
        for t, st in zip(self.ss, self.plan):
            sl = slice(st.band_row0, st.band_row0 + st.band_rows)
            t.upload_band(dem[sl], w[sl])
            if outlets:
                t.set_outlets(outlets)
                t.seed_outlet_drains()

    def block(self, n, mode):
        for t in self.ss:
            t.block_begin()
        if mode == "free":
            for done in range(0, n, 3):
                for t in self.ss:
                    t.block_enqueue(min(3, n - done))
        else:
            _stripes_lockstep(self.ss, n)
        return [t.block_end() for t in self.ss]

    def iterate(self, n, mode):
        if mode == "free":
            for t in self.ss:
                t.iterate(n)
            for t in self.ss:
                t.synchronize()
        else:
            _stripes_lockstep(self.ss, n)

    def water(self):
        return np.concatenate([t.download_owned() for t in self.ss])

    def totals(self, n):
        return sum(t.get_outlet_drains(n) for t in self.ss)

    def checksum(self):
        return sum(t.water_checksum() for t in self.ss) % (1 << 64)

    def final_statistics(self):
        parts = [t.final_statistics() for t in self.ss]
        return sum(p[0] for p in parts), sum(p[1] for p in parts), max(p[2] for p in parts)

    def close(self):
        for t in self.ss:
            t.close()


def _chain(plan, cols, sm):
    """Rounding bound of the stripes' masked sums added on the host (one more addition per stripe)."""
    return max(reduction_chain(st.rows, cols + 2, sm) for st in plan) + len(plan)


# ---- 1. geometry sweep ------------------------------------------------------------------------------------------

@pytest.mark.parametrize("n,rows", GEOMETRIES, ids=[f"{n}x{r}" for n, r in GEOMETRIES])
@pytest.mark.parametrize("tiling", TILINGS)
@pytest.mark.parametrize("mod", [0, 1, 2], ids=["add", "subtract", "drain"])
@pytest.mark.parametrize("dt", [np.float64, np.float32], ids=["f64", "f32"])
def test_stripe_geometry_matches_oracle(cuda_lib, oracle, dt, mod, tiling, n, rows):
    from wdpm_b200.stripes import combine_block_results
    cols = _cols(tiling, dt)
    sc = (cols - 5) // 2
    rng = np.random.default_rng(10000 + 97 * rows + 13 * mod + 3 * TILINGS.index(tiling) + (dt == np.float32))
    D, W = random_case(rng, rows, cols, dt, nodata_fraction=0.05, wet_fraction=0.6, depth=0.05)
    S = Stripes(rows, cols, mod, dt, n, THRES, tiling)
    plan = S.plan
    if rows < 100:
        assert [st.rows for st in plan] == [9] * (n - 1) + [{-2: 9, -1: 10, 1: 12}[rows - 9 * n]], plan
    else:
        assert len({st.rows for st in plan}) > 1, plan
    # Drain: the reference's single outlet, on the first owned row of a middle stripe and on a strip border
    outlet = (plan[n // 2].row0, sc) if mod == 2 else (0, 0)
    if mod == 2:
        D[outlet], W[outlet] = dt(1.0), dt(0.04)
    Wb = W.copy()
    Wb[D <= NODATA] = dt(NODATA)   # as a water file written by the Add module has it; the first prologue clears them
    chain = _chain(plan, cols, S.ss[0].info()["sm_count"])
    S0 = None
    try:
        for mode in ("free", "lockstep"):
            S.upload(D, Wb, [outlet] if mod == 2 else None)
            a, td = Wb.copy(), max(Wb[outlet], dt(0)) if mod == 2 else 0.0
            for nb in BLOCK_ITERS:
                md, _, td = oracle.block(a, D, NODATA, mod, dt(THRES), nb, outlet=outlet, totaldrain=td)
                res = combine_block_results(S.block(nb, mode))
                _check_block(res, a, D, dt, md, chain)
                if mod == 2:
                    assert _same_bits(res.total_drain, td, dt), (mode, res.total_drain, td)
            full, ref = S.water(), a[1:-1, 1:-1]
            bad = np.argwhere(_bits_differ(full, ref))
            assert bad.size == 0, (mode, _where(bad, plan))
            assert S.checksum() == exact_checksum(ref), mode
            assert S.final_statistics() == _final_stats_ref(D[1:-1, 1:-1], ref), mode

        # zero threshold 0 through iterate: the guarded launch on every iteration
        S0 = Stripes(rows, cols, mod, dt, n, 0.0, tiling)
        for mode in ("free", "lockstep"):
            S0.upload(D, W, [outlet] if mod == 2 else None)
            a = W.copy()
            td = oracle.iterate(a, D, NODATA, mod, 12, outlet=outlet, totaldrain=max(W[outlet], dt(0)) if mod == 2 else 0.0)
            S0.iterate(5, mode)
            S0.iterate(7, mode)
            full, ref = S0.water(), a[1:-1, 1:-1]
            bad = np.argwhere(_bits_differ(full, ref))
            assert bad.size == 0, (mode, _where(bad, plan))
            assert S0.checksum() == exact_checksum(ref), mode
            assert S0.final_statistics() == _final_stats_ref(D[1:-1, 1:-1], ref), mode
            if mod == 2:
                assert _same_bits(S0.totals(1)[0], td, dt), (mode, S0.totals(1), td)
    finally:
        for s in (S, S0):
            if s is not None:
                s.close()


def _bits_differ(a, b):
    u = np.uint64 if a.dtype == np.float64 else np.uint32
    return np.ascontiguousarray(a).view(u) != np.ascontiguousarray(b).view(u)


def _where(bad, plan, k=8):
    """The first differing cells as (padded row, col, stripe, row relative to the stripe's first row P0)."""
    out = []
    for i, j in bad[:k]:
        r = int(i) + 1
        s = next(q for q, st in enumerate(plan) if st.row0 <= r < st.row0 + st.rows)
        out.append((r, int(j) + 1, s, r - plan[s].row0))
    return len(bad), out


# ---- 2. Drain on thin stripes -----------------------------------------------------------------------------------

def _border_outlets(plan, rows, cols, sc):
    """On every stripe border row, the rows on either side of it, at strip borders and in between; and the rim."""
    want = [(1, 1), (1, cols), (rows, 1), (rows, cols)]
    for k, st in enumerate(plan[1:]):
        b = st.row0
        for r in (b - 1, b, b + 1):
            want += [(r, sc - 1), (r, sc), (r, sc + 1), (r, 2 * sc), (r, 3 + (5 * k + r) % (cols - 3))]
    return list(dict.fromkeys(rc for rc in want if 1 <= rc[0] <= rows and 1 <= rc[1] <= cols))


@pytest.mark.parametrize("n,rows", [(8, 70), (8, 73), (4, 34)], ids=["8x70", "8x73", "4x34"])
@pytest.mark.parametrize("tiling", TILINGS)
@pytest.mark.parametrize("dt", [np.float64, np.float32], ids=["f64", "f32"])
def test_outlet_set_on_thin_stripes(cuda_lib, oracle, dt, tiling, n, rows):
    """The grid, every outlet's total and max_diff / wet_cells exactly; each stripe's block total is its own totals
    (0 for the outlets of other stripes) added in outlet order in the solver's precision."""
    from wdpm_b200.stripes import combine_block_results
    cols = _cols(tiling, dt)
    sc = (cols - 5) // 2
    rng = np.random.default_rng(20000 + rows + 7 * TILINGS.index(tiling) + (dt == np.float32))
    D, W = random_case(rng, rows, cols, dt, nodata_fraction=0.03, wet_fraction=0.9, depth=0.05)
    S = Stripes(rows, cols, 2, dt, n, THRES, tiling)
    try:
        plan = S.plan
        outlets = _border_outlets(plan, rows, cols, sc)
        assert len(outlets) >= 12 * (n - 1)
        for rc in outlets:
            D[rc] = dt(480.0)   # outlets lie on valid cells
        W[D <= NODATA] = dt(NODATA)
        chain = _chain(plan, cols, S.ss[0].info()["sm_count"])
        for mode in ("free", "lockstep"):
            S.upload(D, W, outlets)
            totals = np.array([max(W[rc], dt(0)) for rc in outlets], dtype=dt)
            assert _same_bits(S.totals(len(outlets)).astype(dt), totals, dt), mode   # the seed: each total on one stripe
            a = W.copy()
            for nb in BLOCK_ITERS:
                md, _, wet, totals = oracle_block_outlets(oracle, a, D, THRES, nb, outlets, totals)
                parts = S.block(nb, mode)
                res = combine_block_results(parts)
                _check_block(res, a, D, dt, md, chain)
                assert res.wet_cells == wet
                got = [t.get_outlet_drains(len(outlets)) for t in S.ss]
                for r, g, st in zip(parts, got, plan):
                    assert _same_bits(r.total_drain, ordered_sum(g.astype(dt), dt), dt), (mode, st)
                assert _same_bits(sum(got).astype(dt), totals, dt), (mode, nb)
                assert _same_bits(ordered_sum(sum(got).astype(dt), dt), ordered_sum(totals, dt), dt)
            full, ref = S.water(), a[1:-1, 1:-1]
            bad = np.argwhere(_bits_differ(full, ref))
            assert bad.size == 0, (mode, _where(bad, plan))
            assert S.final_statistics() == _final_stats_ref(D[1:-1, 1:-1], ref, [(r - 1, c - 1) for r, c in outlets]), mode
    finally:
        S.close()


@pytest.mark.parametrize("tiling", ["small", "auto"])
@pytest.mark.parametrize("mod", [1, 2], ids=["subtract", "drain"])
@pytest.mark.parametrize("dt", [np.float64, np.float32], ids=["f64", "f32"])
def test_serial_schedule_on_eight_nine_row_stripes(cuda_lib, oracle, dt, mod, tiling):
    """The serial schedule on 8 stripes of 9 rows against the oracle's serial schedule. Drain: the single outlet on
    each border row in turn (and once on the row above the middle border), so the 3x3 it empties after every iteration
    spans two stripes; free running and in lockstep."""
    from oracle import pyoracle as po
    from wdpm_b200 import SCHED_SERIAL
    from wdpm_b200.stripes import combine_block_results, plan_stripes
    rows, n = 70, 8
    cols = _cols(tiling, dt)
    sc = (cols - 5) // 2
    plan = plan_stripes(rows, n)
    rng = np.random.default_rng(30000 + 5 * mod + (dt == np.float32))
    D0, W0 = random_case(rng, rows, cols, dt, nodata_fraction=0.03, wet_fraction=0.9, depth=0.05)
    places = [(st.row0, (sc, sc + 1, cols // 2)[k % 3]) for k, st in enumerate(plan[1:])] + [(plan[4].row0 - 1, sc)]
    if mod == 2:
        for rc in places:   # every place is a valid cell: an upload re-marks the outlet installed before it
            D0[rc] = dt(480.0)
    D, W = D0, np.where(D0 > NODATA, W0, dt(0)).astype(dt)
    S = Stripes(rows, cols, mod, dt, n, THRES, tiling, schedule=SCHED_SERIAL)
    chain = _chain(plan, cols, S.ss[0].info()["sm_count"])
    try:
        for outlet in (places if mod == 2 else [(0, 0)]):
            for mode in ("free", "lockstep"):
                S.upload(D, W, [outlet] if mod == 2 else None)
                a, td = W.copy(), max(W[outlet], dt(0)) if mod == 2 else 0.0
                for nb in BLOCK_ITERS:
                    md, _, td = oracle.block(a, D, NODATA, mod, dt(THRES), nb, schedule=po.SCHED_SERIAL, outlet=outlet, totaldrain=td)
                    res = combine_block_results(S.block(nb, mode))
                    _check_block(res, a, D, dt, md, chain)
                    if mod == 2:
                        assert _same_bits(res.total_drain, td, dt), (outlet, mode, res.total_drain, td)
                full, ref = S.water(), a[1:-1, 1:-1]
                bad = np.argwhere(_bits_differ(full, ref))
                assert bad.size == 0, (outlet, mode, _where(bad, plan))
    finally:
        S.close()


_FIRST_BLOCK = r"""
import sys
import numpy as np
sys.path[:0] = sys.argv[1:3]
from conftest import random_case
from wdpm_b200 import F32, F64, WdpmError
from wdpm_b200.stripes import StripeSolver, connect_in_process, plan_stripes
dt, code = (np.float64, F64) if sys.argv[3] == "f64" else (np.float32, F32)
rows, cols = 16, 53
D, W = random_case(np.random.default_rng(5), rows, cols, dt)
plan = plan_stripes(rows, 2)
outlet = (plan[1].row0, 24)
D[outlet] = dt(1.0)
ss = [StripeSolver(rows, cols, -99999.0, 2, st, dtype=code, zero_threshold=4e-3, fused_variant=2, schedule=int(sys.argv[4]))
      for st in plan]
connect_in_process(ss)
for t, st in zip(ss, plan):
    sl = slice(st.band_row0, st.band_row0 + st.band_rows)
    t.upload_band(D[1:-1, 1:-1][sl], W[1:-1, 1:-1][sl])
    t.set_outlets([outlet])
    t.seed_outlet_drains()
for t in ss:
    t.block_begin()
for t in ss:
    t.block_enqueue(1)
try:
    for t in ss:
        t.block_end()
    print("FIRST_BLOCK_OK")
except WdpmError as e:
    print("FIRST_BLOCK_FAILED", e)
"""


@pytest.mark.parametrize("schedule", [0, 1], ids=["opencl", "serial"])
@pytest.mark.parametrize("dt", ["f64", "f32"])
def test_first_drain_block_in_a_fresh_process(cuda_lib, dt, schedule):
    """The first free-running Drain block of a process: each stripe enqueues its fold (serial schedule: its outlet
    emptying) behind a halo wait that spins until the neighbour's kernel has run, before the host has launched that
    kernel. No kernel may be loaded for the first time there (solver.cu, preload_stripe_kernels): the load could wait
    for the spinning wait, and the block would end in WDPM_E_HALO. A fresh process, so that no earlier test has loaded
    the kernels already."""
    here = Path(__file__).resolve().parent
    res = subprocess.run([sys.executable, "-c", _FIRST_BLOCK, str(here.parent), str(here), dt, str(schedule)], capture_output=True,
                         text=True, timeout=300, env=dict(os.environ, WDPM_B200_HALO_TIMEOUT_MS="5000"))
    assert "FIRST_BLOCK_OK" in res.stdout, res.stdout[-1000:] + res.stderr[-2000:]


# ---- 3. checkpoints across stripe counts ------------------------------------------------------------------------

CHECKPOINTS = [  # (case, dtype, capturing run, resuming run); a run = (stripes, driver, kernel name of test_gpu_checkpoint)
    ("drain-rim", np.float64, (8, "free", "fused-production"), (0, None, "fused-production")),
    ("drain-rim", np.float32, (8, "lockstep", "fused-small"), (3, "free", "fused-production")),
    ("drain-ref", np.float64, (8, "lockstep", "fused-production"), (3, "lockstep", "fused-small")),
    ("sub", np.float64, (8, "free", "fused-small"), (0, None, "resident")),
    ("drain-serial", np.float32, (8, "free", "fused-small"), (0, None, "fused-production")),
    ("add", np.float32, (0, None, "fused-production"), (8, "free", "fused-production")),
    ("drain-rim", np.float64, (3, "free", "fused-small"), (8, "lockstep", "fused-small")),
    ("drain-rim", np.float32, (0, None, "resident"), (8, "free", "fused-small")),
    ("drain-ref", np.float32, (3, "lockstep", "fused-production"), (8, "free", "fused-production")),
]


@pytest.mark.parametrize("case,dt,first,second", CHECKPOINTS,
                         ids=[f"{c}-{'f64' if d == np.float64 else 'f32'}-{a[0]}to{b[0]}" for c, d, a, b in CHECKPOINTS])
def test_checkpoint_across_stripe_counts(cuda_lib, case, dt, first, second):
    """Capture at the start of block B on one partition, resume in fresh solvers on another: the resumed blocks, grid
    and outlet totals equal those of one uninterrupted single solver (colour kernel) bit for bit; so does the
    capturing run, which goes on after its capture."""
    module, schedule = CASES[case]
    rows, cols, B, nit = 70, 300, 3, 9
    dem, w = _ck_case(dt, rows=rows, cols=cols, seed=17)
    runs = []

    def run(spec):
        r = Run(rows, cols, module, dt, n_stripes=spec[0], driver=spec[1], schedule=schedule, **_kernels(dt)[spec[2]])
        runs.append(r)
        if spec[0]:
            for t in r.ss:
                i = t.info()
                assert i["warp_autonomous"] == (spec[2] == "fused-production") and i["iters_per_launch"] == 1, i
            if spec[0] == 8:
                assert {st.rows for st in r.plan} == {9}
        return r

    try:
        ref = run((0, None, "colour"))
        outlets = _setup(ref, case, dem, w)
        one = outlets[0] if outlets and case != "drain-rim" else None
        rr = [ref.block(nit) for _ in range(2 * B)]
        wr, tr = ref.water(), ref.totals()

        a = run(first)
        _setup(a, case, dem, w, outlet=one)
        ra = []
        for b in range(2 * B):
            if b == B:
                a.arm()
            ra.append(a.block(nit))
        cw, ct = a.capture()
        wa, ta = a.water(), a.totals()

        c = run(second)
        _setup(c, case, dem, cw, resume=True, totals=ct if module == 2 else None, outlet=one)
        rc = [c.block(nit) for _ in range(B)]
        wc, tc = c.water(), c.totals()
    finally:
        for r in runs:
            r.close()
    for got, name in ((ra, "capturing run"), (ra[:B] + rc, "resumed run")):
        for k, (x, y) in enumerate(zip(got, rr)):
            assert (x.max_diff, x.total_drain, x.wet_cells) == (y.max_diff, y.total_drain, y.wet_cells), (name, k)
            assert abs(x.masked_sum - y.masked_sum) <= 1e-12 * abs(y.masked_sum), (name, k)
    for wx, tx, name in ((wa, ta, "capturing run"), (wc, tc, "resumed run")):
        assert _same_bits(wx, wr, dt), (name, int(_bits_differ(wx, wr).sum()))
        if module == 2:
            assert _same_bits(tx, tr, np.float64), name


# ---- 4. several real GPUs ---------------------------------------------------------------------------------------

def _device_count():
    import torch
    return torch.cuda.device_count()


def test_distributed_nine_row_stripes(cuda_lib):
    """One rank per GPU over CUDA IPC: 70 rows make 9-row stripes at world 8; below 8 GPUs a 9 * world - 2 row DEM
    does the same."""
    n = _device_count()
    if n < 2:
        pytest.skip("needs at least 2 GPUs")
    world = min(8, n)
    shapes = [(70, 900)] + ([(9 * world - 2, 900)] if world < 8 else [])
    script = Path(__file__).resolve().parent / "dist_stripes_check.py"
    for port, (rows, cols) in zip((29571, 29572), shapes):
        res = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}",
                              "--master-addr", "127.0.0.1", "--master-port", str(port), str(script), str(rows), str(cols)],
                             capture_output=True, text=True, timeout=900, env=dict(os.environ, WDPM_B200_HALO_TIMEOUT_MS=HALO_TIMEOUT_MS))
        assert "STRIPES_OK" in res.stdout, (rows, world, res.stdout[-2000:] + res.stderr[-3000:])


@pytest.fixture(scope="module")
def host_bin(cuda_lib):
    from wdpm_b200 import build
    return build.build_host()


@pytest.mark.parametrize("rows", [70, 20])
def test_cli_on_eight_gpus_equals_one(host_bin, tmp_path, rows):
    """WDPM_B200_GPUS=8 writes the same files and prints the same report numbers as one GPU: Add, then Drain with the
    reference's outlet and with the rim as an outlet set (per-outlet totals too). 70 rows make eight 9-row stripes;
    20 rows are too few for 8 stripes, and the host must lower the count (to 2) instead of failing."""
    from wdpm_b200 import ascgrid
    if _device_count() < 2:
        pytest.skip("needs at least 2 GPUs")
    rng = np.random.default_rng(40000 + rows)
    cols = 90
    d = (500 + 3 * rng.standard_normal((rows, cols))).round(4)
    d[rng.uniform(size=d.shape) < 0.05] = NODATA
    dem = tmp_path / "dem.asc"
    ascgrid.write_asc(dem, ascgrid.AscHeader.default(rows, cols), d)
    outs = {}
    for gpus in ("1", "8"):
        o = tmp_path / f"gpus{gpus}"
        o.mkdir()
        add, drain, rim = o / "add.asc", o / "drain.asc", o / "rim.asc"
        runs = [(["add", dem, "NULL", add, "NULL", "10", "1.0", "1.0", "1", "1", "0.005", "3000"], {}),
                (["drain", dem, add, drain, "NULL", "0.1", "1.0", "1", "1", "0.005", "2000"], {}),
                (["drain", dem, add, rim, "NULL", "0.1", "1.0", "1", "1", "0.005", "2000"],
                 {"WDPM_B200_OUTLETS": "rim", "WDPM_B200_OUTLET_TOTALS": str(o / "rim.csv")})]
        reports = []
        for argv, env in runs:
            res = subprocess.run([str(host_bin)] + [str(x) for x in argv], capture_output=True, text=True, timeout=600,
                                 env=dict(os.environ, WDPM_B200_GPUS=gpus, WDPM_B200_HALO_TIMEOUT_MS=HALO_TIMEOUT_MS, **env))
            assert res.returncode == 0, (gpus, res.stdout[-800:] + res.stderr)
            reports.append(_normalise(res.stdout))
        outs[gpus] = ([p.read_bytes() for p in (add, drain, rim, o / "rim.csv")], reports)
    for k, name in enumerate(("add", "drain", "rim drain", "rim totals")):
        assert outs["8"][0][k] == outs["1"][0][k], name
    for k, name in enumerate(("add", "drain", "rim drain")):
        assert outs["8"][1][k] == outs["1"][1][k], name
