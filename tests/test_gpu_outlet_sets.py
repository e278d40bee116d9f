"""Drain outlet sets above the old cap of 1024: rim sets against the oracle on every kernel, the seed entry point,
stripes, the limits of wdpm_set_outlets, and WDPM_B200_OUTLETS in the command-line host."""
import os
import subprocess
import time

import numpy as np
import pytest

from conftest import GOLDEN, gunzip_to, random_case

NODATA = -99999.0
pytestmark = pytest.mark.gpu


def _ordered_sum(v, dt):
    acc = dt(v[0])
    for x in v[1:]:
        acc = dt(acc + dt(x))
    return acc


def _seeded(W, outlets, dt):
    return np.array([max(W[r, c], dt(0)) for r, c in outlets], dtype=dt)


@pytest.mark.parametrize("dt", [np.float64, np.float32])
@pytest.mark.parametrize("kernel,variant", [(1, 0), (2, 1), (2, 2), (2, 3), (2, 17), (2, 18), (3, 0)])
def test_rim_set_above_the_old_cap_matches_oracle(cuda_lib, oracle, dt, kernel, variant):
    """About 2 000 rim outlets on a 400 x 700 grid with 4 % NODATA: water grid and every per-outlet total bit for
    bit, totals seeded by wdpm_seed_outlet_drains as the oracle is given them."""
    from wdpm_b200 import F32, F64, Solver, ascgrid
    code = F64 if dt == np.float64 else F32
    rng = np.random.default_rng(501)
    rows, cols, n_it = 400, 700, 5
    D, W = random_case(rng, rows, cols, dt, nodata_fraction=0.04, wet_fraction=0.9)
    outlets = ascgrid.rim_outlets(D[1:-1, 1:-1], NODATA)
    assert len(outlets) > 1024
    a = W.copy()
    ta = oracle.iterate_outlets(a, D, NODATA, n_it, outlets, totals=_seeded(W, outlets, dt))
    s = Solver(rows, cols, NODATA, 2, dtype=code, kernel=kernel, fused_variant=variant)
    s.upload(D[1:-1, 1:-1], W[1:-1, 1:-1])
    s.set_outlets(outlets)
    s.seed_outlet_drains()
    s.iterate(n_it)
    b = ascgrid.pad_grid(s.download_water(), dt(0))
    tb = s.get_outlet_drains(len(outlets)).astype(dt)
    total = s.get_total_drain()
    blk = s.run_block(0)
    s.close()
    assert np.array_equal(a, b), int((a != b).sum())
    assert np.array_equal(ta, tb), int((ta != tb).sum())
    assert dt(total) == _ordered_sum(ta, dt) and blk.total_drain == total


def test_fractal_rim_set_matches_oracle(cuda_lib, oracle):
    """2048^2 fractal DEM, its whole rim (8 188 outlets), on the production fp64 kernel."""
    from wdpm_b200 import F64, Solver, ascgrid, synth
    n = 2048
    d = synth.fractal_dem(n, n, seed=5).numpy()
    D = ascgrid.pad_grid(d, NODATA)
    W = np.where(D > NODATA, 0.05, 0.0)
    outlets = ascgrid.rim_outlets(d, NODATA)
    assert len(outlets) == 8188
    a = W.copy()
    ta = oracle.iterate_outlets(a, D, NODATA, 20, outlets, totals=_seeded(W, outlets, np.float64))
    s = Solver(n, n, NODATA, 2, dtype=F64)
    s.upload(d, W[1:-1, 1:-1])
    s.set_outlets(outlets)
    s.seed_outlet_drains()
    blk = s.run_block(20)
    b = ascgrid.pad_grid(s.download_water(), 0.0)
    tb = s.get_outlet_drains(len(outlets))
    s.close()
    assert np.array_equal(a, b) and np.array_equal(ta, tb)
    assert blk.total_drain == _ordered_sum(ta, np.float64)


@pytest.mark.parametrize("dt", [np.float64, np.float32])
def test_seed_is_max_of_water_and_zero(cuda_lib, dt):
    from wdpm_b200 import F32, F64, Solver
    code = F64 if dt == np.float64 else F32
    rng = np.random.default_rng(502)
    D, W = random_case(rng, 60, 80, dt, nodata_fraction=0.0)
    W[1:-1, 1:-1] -= dt(0.2)  # negative water under some outlets
    outlets = [(r, c) for r in range(1, 61, 7) for c in range(1, 81, 9)]
    s = Solver(60, 80, NODATA, 2, dtype=code, kernel=2)
    s.upload(D[1:-1, 1:-1], W[1:-1, 1:-1])
    s.set_outlets(outlets)
    s.seed_outlet_drains()
    got = s.get_outlet_drains(len(outlets)).astype(dt)
    assert np.array_equal(got, _seeded(W, outlets, dt))
    # one outlet: the host sequence get_cell_water + set_total_drain(max(w, 0)), bit for bit
    for rc in outlets[:6]:
        s.set_outlets([rc])
        s.seed_outlet_drains()
        seeded = s.get_total_drain()
        w = s.get_cell_water(*rc)
        s.set_total_drain(w if w > 0 else 0.0)
        assert np.float64(seeded).tobytes() == np.float64(s.get_total_drain()).tobytes()
    s.close()


@pytest.mark.parametrize("n_stripes,variant", [(3, 2), (3, 18)])
def test_in_process_stripes_with_a_rim_set(cuda_lib, n_stripes, variant):
    """A rim set crosses every stripe border: checksum and every per-outlet total equal the single solver's."""
    from wdpm_b200 import F64, Solver, ascgrid
    from wdpm_b200.stripes import StripeSolver, connect_in_process, plan_stripes
    rng = np.random.default_rng(503)
    rows, cols, n_it = 130, 300, 8
    D, W = random_case(rng, rows, cols, np.float64, nodata_fraction=0.02, wet_fraction=0.95)
    dem, w0 = D[1:-1, 1:-1], W[1:-1, 1:-1]
    outlets = ascgrid.rim_outlets(dem, NODATA) + [(r, c) for r in range(3, rows, 11) for c in (40, 41, 150) if dem[r - 1, c - 1] > NODATA]
    ref = Solver(rows, cols, NODATA, 2, dtype=F64, fused_variant=variant, fused_chunk_rows=21)
    ref.upload(dem, w0)
    ref.set_outlets(outlets)
    ref.seed_outlet_drains()
    ref.iterate(n_it)
    ref_sum, ref_td = ref.water_checksum(), ref.get_outlet_drains(len(outlets))
    ref.close()
    plan = plan_stripes(rows, n_stripes)
    ss = [StripeSolver(rows, cols, NODATA, 2, st, dtype=F64, fused_variant=variant, fused_chunk_rows=21) for st in plan]
    connect_in_process(ss)
    for s, st in zip(ss, plan):
        s.upload_band(dem[st.band_row0:st.band_row0 + st.band_rows], w0[st.band_row0:st.band_row0 + st.band_rows])
        s.set_outlets(outlets)
        s.seed_outlet_drains()
    for _ in range(n_it):  # lockstep
        for s in ss:
            s.phase(0)
        for s in ss:
            s.synchronize()
        for s in ss:
            s.phase(1)
        for s in ss:
            s.synchronize()
    chk = sum(s.water_checksum() for s in ss) % (1 << 64)
    td = sum(s.get_outlet_drains(len(outlets)) for s in ss)
    # free-running: the same solvers, each iteration's contacts folded by the next launch
    for s, st in zip(ss, plan):
        s.upload_band(dem[st.band_row0:st.band_row0 + st.band_rows], w0[st.band_row0:st.band_row0 + st.band_rows])
        s.seed_outlet_drains()
    for s in ss:
        s.block_begin()
    for s in ss:
        s.block_enqueue(n_it)
    for s in ss:
        s.block_end()
    chk2 = sum(s.water_checksum() for s in ss) % (1 << 64)
    td2 = sum(s.get_outlet_drains(len(outlets)) for s in ss)
    for s in ss:
        s.close()
    assert chk == ref_sum and np.array_equal(td, ref_td)
    assert chk2 == ref_sum and np.array_equal(td2, ref_td)


def _big_case():
    rng = np.random.default_rng(504)
    n = 1100
    d = (500 + 3 * rng.standard_normal((n, n))).round(4)
    w = rng.uniform(0, 0.2, (n, n))
    return rng, n, d, w


def test_limits_of_the_set(cuda_lib, oracle):
    from wdpm_b200 import F64, MAX_OUTLETS, Solver, SCHED_SERIAL, WdpmError, ascgrid
    rng, n, d, w = _big_case()
    rim = ascgrid.rim_outlets(d, NODATA)
    idx = np.arange(n * n)
    inner = idx[(idx // n > 0) & (idx // n < n - 1) & (idx % n > 0) & (idx % n < n - 1)]
    pick = rng.choice(inner, MAX_OUTLETS - len(rim), replace=False)
    full = rim + [(int(k // n) + 1, int(k % n) + 1) for k in pick]
    assert len(full) == MAX_OUTLETS == 1 << 20
    s = Solver(n, n, NODATA, 2, dtype=F64)
    s.upload(d, w)
    s.set_outlets(full)  # exactly 2^20: accepted, one block runs
    s.seed_outlet_drains()
    blk = s.run_block(3)
    tb = s.get_outlet_drains(len(full))
    b = s.download_water()
    D, W = ascgrid.pad_grid(d, NODATA), ascgrid.pad_grid(w, 0.0)
    ta = oracle.iterate_outlets(W, D, NODATA, 3, full, totals=_seeded(ascgrid.pad_grid(w, 0.0), full, np.float64))
    assert np.array_equal(W[1:-1, 1:-1], b) and np.array_equal(ta, tb)
    assert blk.total_drain == _ordered_sum(ta, np.float64)
    taken = np.zeros(n * n, dtype=bool)
    taken[pick] = True
    free = int(inner[~taken[inner]][0])
    extra = (free // n + 1, free % n + 1)
    with pytest.raises(WdpmError) as e:
        s.set_outlets(full + [extra])
    assert e.value.code == -1
    dup = full[:500000]
    dup[250000] = dup[7]
    t0 = time.perf_counter()
    with pytest.raises(WdpmError) as e:
        s.set_outlets(dup)
    assert e.value.code == -1 and time.perf_counter() - t0 < 1.0
    s.close()
    # an outlet on NODATA: refused at install, and by an upload that meets an earlier set
    d2 = d[:50, :60].copy()
    d2[10, 10] = NODATA
    s = Solver(50, 60, NODATA, 2, dtype=F64, kernel=2)
    s.upload(d2, None)
    with pytest.raises(WdpmError) as e:
        s.set_outlets([(5, 5), (11, 11)])
    assert e.value.code == -1
    s.set_outlets([(5, 5)])
    s.close()
    s = Solver(50, 60, NODATA, 2, dtype=F64, kernel=2)
    s.set_outlets([(5, 5), (11, 11)])
    with pytest.raises(WdpmError) as e:
        s.upload(d2, None)
    assert e.value.code == -1
    s.close()
    s = Solver(50, 60, NODATA, 2, dtype=F64, kernel=1, schedule=SCHED_SERIAL)
    s.upload(d[:50, :60], None)
    with pytest.raises(WdpmError) as e:
        s.set_outlets([(5, 5), (6, 9)])
    assert e.value.code == -5
    s.close()


def test_device_bytes_grow_linearly(cuda_lib):
    """wdpm_get_info().device_bytes: at most 560 bytes per outlet (fp64, one iteration per launch: three event
    buffers of 8 B mask + 4 B list + 10 slots x 16 B, plus total, saved elevation, (row, col) and position)."""
    from wdpm_b200 import F64, Solver
    rng, n, d, w = _big_case()
    s = Solver(n, n, NODATA, 2, dtype=F64)
    s.upload(d, w)
    base = s.info()["device_bytes"]
    sizes = {}
    for m in (1, 1000, 100000, 500000):
        k = rng.choice(n * n, m, replace=False)
        s.set_outlets([(int(q // n) + 1, int(q % n) + 1) for q in k])
        sizes[m] = s.info()["device_bytes"] - base
    s.close()
    per = (sizes[500000] - sizes[1]) / 499999
    print(f"device bytes per outlet: {per:.1f}", sizes)
    assert per <= 560 and sizes[1] == 0
    assert abs((sizes[100000] - sizes[1000]) / 99000 - per) < 1.0


# ---- the command-line host -------------------------------------------------------------------------------


@pytest.fixture(scope="module")
def host_bin(cuda_lib):
    from wdpm_b200 import build
    return build.build_host()


def _drain_argv(dem, water, out, thres="0.005"):
    return ["drain", str(dem), str(water), str(out), "NULL", "0.1", "1.0", "1", "1", thres, "0"]


def _run(host_bin, argv, **env):
    e = dict(os.environ)
    e.update(env)
    res = subprocess.run([str(host_bin)] + argv, capture_output=True, text=True, timeout=900, env=e)
    assert res.returncode == 0, res.stdout[-800:] + res.stderr
    return res.stdout


def _report(text):
    out = []
    for ln in text.split("\n"):
        if "Run Time" in ln or "Drain" in ln or "Min DEM" in ln or "file:" in ln:
            continue
        toks = ln.split()
        if toks and toks[0].isdigit() and len(toks) == 5:
            ln = " ".join(toks[:-1])
        out.append(ln.rstrip())
    return out


def _water_in(tmp_path, host_bin, dem):
    add = tmp_path / "add.asc"
    _run(host_bin, ["add", str(dem), "NULL", str(add), "NULL", "10", "1.0", "1.0", "1", "1", "0.005", "0"])
    return add


def test_cli_outlet_grid_with_the_reference_outlet(host_bin, tmp_path):
    """WDPM_B200_OUTLETS naming only the reference's outlet: the same output file, the same report apart from the
    outlet lines."""
    from wdpm_b200 import ascgrid
    dem = gunzip_to("basin5.asc.gz", tmp_path / "basin5.asc")
    add = _water_in(tmp_path, host_bin, dem)
    ref_out, set_out = tmp_path / "ref.asc", tmp_path / "set.asc"
    ref = _run(host_bin, _drain_argv(dem, add, ref_out))
    row = int(next(ln for ln in ref.split("\n") if "Drain row:" in ln).split()[-1])
    col = int(next(ln for ln in ref.split("\n") if "Drain column:" in ln).split()[-1])
    hdr, d = ascgrid.read_asc(dem)
    mark = np.zeros_like(d)
    mark[row - 1, col - 1] = 1.0
    grid = tmp_path / "outlet.asc"
    ascgrid.write_asc(grid, hdr, mark)
    got = _run(host_bin, _drain_argv(dem, add, set_out), WDPM_B200_OUTLETS=str(grid))
    assert set_out.read_bytes() == ref_out.read_bytes()
    assert _report(got) == _report(ref)
    assert "Drain outlets: 1" in " ".join(got.split())


def test_cli_rim_set_balances_and_is_partition_free(host_bin, tmp_path):
    import torch
    from wdpm_b200 import ascgrid
    dem = gunzip_to("basin5.asc.gz", tmp_path / "basin5.asc")
    add = _water_in(tmp_path, host_bin, dem)
    hdr, d = ascgrid.read_asc(dem)
    _, w = ascgrid.read_asc(add)
    gpus = ["1", "2"] if torch.cuda.device_count() >= 2 else ["1"]
    outs = {}
    for g in gpus:
        out, csv = tmp_path / f"rim{g}.asc", tmp_path / f"rim{g}.csv"
        text = _run(host_bin, _drain_argv(dem, add, out, thres="0"), WDPM_B200_OUTLETS="rim", WDPM_B200_GPUS=g, WDPM_B200_OUTLET_TOTALS=str(csv))
        outs[g] = (out.read_bytes(), csv.read_text(), text)
    rim = ascgrid.rim_outlets(d, hdr.nodata)
    lines = outs["1"][1].strip().split("\n")
    assert [tuple(map(int, ln.split(",")[:2])) for ln in lines] == rim
    assert f"Drain outlets: {len(rim)}" in " ".join(outs["1"][2].split())
    drained = 0.0
    for ln in lines:
        drained = drained + float(ln.split(",")[3])
    _, left = ascgrid.read_asc(tmp_path / "rim1.asc")
    valid = d > hdr.nodata
    cellarea = hdr.cellsize ** 2
    put_in = float(np.sum(w[valid])) * cellarea
    # each total starts with the water under its outlet, which stays in the grid until a centre empties the outlet
    # (WDPMCL.c:1029): that water is counted twice
    seeds = sum(max(float(w[r - 1, c - 1]), 0.0) for r, c in rim) * cellarea
    after = float(np.sum(left[valid])) * cellarea + drained - seeds
    assert abs(after - put_in) <= 1e-12 * put_in + 1e-6 * cellarea * valid.sum()  # the output file keeps 6 decimals
    for g in gpus[1:]:
        assert outs[g][0] == outs["1"][0] and outs[g][1] == outs["1"][1]
