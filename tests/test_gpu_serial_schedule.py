"""GPU (-m gpu): the serial schedule (WDPM_SCHEDULE_SERIAL, the reference's `cpu=0` branch) against the CPU oracle's
serial schedule and the unmodified reference's serial output files - bit for bit.

Serial Subtract relaxes with the Add step (runoffs); serial Drain empties the outlet's 3x3 neighbourhood into the
drained total after every iteration. Both are checked on every kernel: colour, a small k_fused test window, the
production warp-autonomous variant and the resident kernel, then on row stripes and through the command line."""
import os
import subprocess

import numpy as np
import pytest

from conftest import GOLDEN, golden_text, gunzip_to, random_case
from oracle import pyoracle as po
from wdpm_b200 import ascgrid

pytestmark = pytest.mark.gpu
NODATA = -99999.0


def _code(dt):
    from wdpm_b200 import F32, F64
    return F64 if dt == np.float64 else F32


def _kernels(dt):
    """(name, Solver keyword arguments): every kernel the serial schedule can run on."""
    from wdpm_b200 import KERNEL_COLOUR, KERNEL_FUSED, KERNEL_RESIDENT
    from wdpm_b200.solver import PRODUCTION_FUSED_VARIANT_F32, PRODUCTION_FUSED_VARIANT_F64
    prod = PRODUCTION_FUSED_VARIANT_F64 if dt == np.float64 else PRODUCTION_FUSED_VARIANT_F32
    return [("colour", dict(kernel=KERNEL_COLOUR)),
            ("fused_test_window", dict(kernel=KERNEL_FUSED, fused_variant=2, fused_chunk_rows=21)),
            ("fused_production", dict(kernel=KERNEL_FUSED, fused_variant=prod, fused_chunk_rows=21)),
            ("resident", dict(kernel=KERNEL_RESIDENT))]


def _outlets(D, strip_cols):
    """Interior, corners and edges (the 3x3 reaches the halo ring), next to NODATA, and on both sides of a fused
    CTA chunk boundary (fused_chunk_rows=21: padded rows 20 | 21) and a strip boundary."""
    R, C = D.shape[0] - 2, D.shape[1] - 2
    return [(R // 2, C // 2), (1, 1), (1, C), (R, 1), (R, C), (1, C // 3), (R // 3, C), ("nodata", None),
            (20, C // 2), (21, C // 2 + 1), (R // 2, strip_cols - 1), (R // 2 + 1, strip_cols)]


def _place_outlet(D, W, o):
    """Make cell o a valid, low cell; 'nodata' picks an interior cell and turns two of its neighbours into NODATA."""
    D = D.copy()
    R, C = D.shape[0] - 2, D.shape[1] - 2
    if o[0] == "nodata":
        o = (R // 3 + 1, 2 * C // 3 + 1)
        D[o[0] - 1, o[1]] = NODATA
        D[o[0], o[1] + 1] = NODATA
    o = (min(max(o[0], 1), R), min(max(o[1], 1), C))
    D[o] = D.dtype.type(480.0)
    W = np.where(D > NODATA, W, 0).astype(D.dtype)
    return D, W, o


def _strip_cols(dt, variant):
    from wdpm_b200 import solver
    return solver.fused_variant_info(variant, _code(dt))["strip_cols"]


def _run(D, W, module, dt, n, outlet=None, td=0.0, **kw):
    """wdpm_iterate on a serial-schedule solver, zero threshold 0, water uploaded as given."""
    from wdpm_b200 import SCHED_SERIAL, Solver
    with Solver(D.shape[0] - 2, D.shape[1] - 2, NODATA, module, dtype=_code(dt), schedule=SCHED_SERIAL, **kw) as s:
        s.upload(D[1:-1, 1:-1], W[1:-1, 1:-1])
        if module == 2:
            s.set_outlet(*outlet)
            s.set_total_drain(td)
        s.iterate(n)
        return ascgrid.pad_grid(s.download_water(), dt(0)), s.get_total_drain()


def _same(a, b):
    """Equal bit for bit, signed zeros included."""
    return np.array_equal(a.view(np.uint64 if a.dtype == np.float64 else np.uint32),
                          b.view(np.uint64 if b.dtype == np.float64 else np.uint32))


@pytest.mark.parametrize("dt", [np.float64, np.float32])
@pytest.mark.parametrize("module", [1, 2])
@pytest.mark.parametrize("kname", ["colour", "fused_test_window", "fused_production", "resident"])
def test_serial_iterate_matches_oracle(cuda_lib, oracle, dt, module, kname):
    kw = dict(_kernels(dt))[kname]
    rng = np.random.default_rng(31 + module)
    for rows, cols, n in ((33, 65, 9), (100, 131, 13), (130, 420, 7)):
        D0, W0 = random_case(rng, rows, cols, dt)
        sc = _strip_cols(dt, kw.get("fused_variant", 2))
        for o in (_outlets(D0, sc) if module == 2 else [(1, 1)]):
            D, W, outlet = _place_outlet(D0, W0, o)
            a = W.copy()
            ta = oracle.iterate(a, D, NODATA, module, n, schedule=po.SCHED_SERIAL, outlet=outlet, totaldrain=0.5)
            b, tb = _run(D, W, module, dt, n, outlet=outlet, td=0.5, **kw)
            assert _same(a, b), (kname, rows, cols, outlet, int((a != b).sum()))
            if module == 2:
                assert dt(ta) == dt(tb), (kname, rows, cols, outlet, ta, tb)


@pytest.mark.parametrize("dt", [np.float64, np.float32])
@pytest.mark.parametrize("module", [1, 2])
@pytest.mark.parametrize("kname", ["colour", "fused_test_window", "fused_production", "resident"])
def test_serial_run_block_matches_oracle(cuda_lib, oracle, dt, module, kname):
    """Two blocks with a zero threshold > 0 (the cheaper steps become selectable after the first prologue)."""
    kw = dict(_kernels(dt))[kname]
    rng = np.random.default_rng(41 + module)
    D0, W0 = random_case(rng, 100, 131, dt)
    for o in ((50, 60), (1, 1), (21, 70)):
        D, W, outlet = _place_outlet(D0, W0, o)
        a, td = W.copy(), 0.25
        from wdpm_b200 import SCHED_SERIAL, Solver
        s = Solver(100, 131, NODATA, module, dtype=_code(dt), schedule=SCHED_SERIAL, zero_threshold=5e-6, **kw)
        s.upload(D[1:-1, 1:-1], W[1:-1, 1:-1])
        if module == 2:
            s.set_outlet(*outlet)
            s.set_total_drain(td)
        for n in (11, 17):
            md, _, td = oracle.block(a, D, NODATA, module, 5e-6, n, schedule=po.SCHED_SERIAL, outlet=outlet, totaldrain=td)
            r = s.run_block(n)
            assert r.max_diff == md, (kname, outlet, n)
            if module == 2:
                assert dt(r.total_drain) == dt(td), (kname, outlet, n)
        b = ascgrid.pad_grid(s.download_water(), dt(0))
        s.close()
        assert _same(a, b), (kname, outlet, int((a != b).sum()))


@pytest.mark.parametrize("dt", [np.float64, np.float32])
@pytest.mark.parametrize("kname", ["colour", "fused_test_window", "fused_production", "resident"])
def test_add_does_not_depend_on_the_schedule(cuda_lib, dt, kname):
    from wdpm_b200 import SCHED_OPENCL, SCHED_SERIAL, Solver
    kw = dict(_kernels(dt))[kname]
    D, W = random_case(np.random.default_rng(5), 100, 131, dt)
    outs = []
    for sched in (SCHED_OPENCL, SCHED_SERIAL):
        with Solver(100, 131, NODATA, 0, dtype=_code(dt), schedule=sched, zero_threshold=1e-5, **kw) as s:
            s.upload(D[1:-1, 1:-1], W[1:-1, 1:-1])
            s.apply_add(0.01, 1.0)
            s.run_block(9)
            s.iterate(5)
            outs.append(s.download_water())
    assert _same(outs[0], outs[1])


def _negzero_case(rng, rows, cols, dt):
    """Integer elevations and water in halves, so that h == +0 is common; the water holds -0.0 on valid cells,
    negative values, and water on NODATA cells - as an uploaded water file may, with no apply_subtract after it."""
    d = np.round(500 + 2 * rng.standard_normal((rows, cols)))
    d[rng.uniform(size=d.shape) < 0.05] = NODATA
    D = ascgrid.pad_grid(d.astype(dt), dt(NODATA))
    choice = rng.choice(np.array([0.0, -0.0, 0.5, 1.0, 1.5, 2.0, -0.5]), size=D.shape)
    W = choice.astype(dt)
    W[0, :] = W[-1, :] = W[:, 0] = W[:, -1] = 0
    return D, W


def test_serial_subtract_with_negative_zero_water(cuda_lib, oracle):
    """Zero threshold 0, water uploaded as is: the fp64 sign-gated Add step would turn a -0.0 neighbour at h == +0
    into +0.0; the solver must run the reference form of the step on every kernel AUTO can pick."""
    from wdpm_b200 import KERNEL_AUTO, KERNEL_FUSED, KERNEL_RESIDENT
    from wdpm_b200.solver import PRODUCTION_FUSED_VARIANT_F32, PRODUCTION_FUSED_VARIANT_F64
    rng = np.random.default_rng(9)
    for dt in (np.float64, np.float32):
        prod = PRODUCTION_FUSED_VARIANT_F64 if dt == np.float64 else PRODUCTION_FUSED_VARIANT_F32
        D, W = _negzero_case(rng, 120, 150, dt)
        a = W.copy()
        oracle.iterate(a, D, NODATA, 1, 6, schedule=po.SCHED_SERIAL)
        assert np.any((a == 0) & np.signbit(a) & (D > NODATA)), "the case must keep some -0.0"
        for kw in (dict(kernel=KERNEL_AUTO), dict(kernel=KERNEL_RESIDENT), dict(kernel=KERNEL_FUSED, fused_variant=0),
                   dict(kernel=KERNEL_FUSED, fused_variant=prod), dict(kernel=KERNEL_FUSED, fused_variant=2)):
            b, _ = _run(D, W, 1, dt, 6, **kw)
            assert _same(a, b), (dt, kw, int((a != b).sum()))


def _lockstep(ss, n_it):
    for _ in range(n_it):
        for s in ss:
            s.phase(0)
        for s in ss:
            s.synchronize()
        for s in ss:
            s.phase(1)
        for s in ss:
            s.synchronize()


@pytest.mark.parametrize("dt", [np.float64, np.float32])
@pytest.mark.parametrize("module", [1, 2])
@pytest.mark.parametrize("n_stripes,variant", [(2, 2), (3, 2), (2, 18), (3, 18)])
def test_serial_in_process_stripes(cuda_lib, oracle, dt, module, n_stripes, variant):
    """Lockstep stripes; a Drain outlet on, directly above and directly below a stripe border, so that the 3x3
    it empties spans two stripes."""
    from wdpm_b200 import SCHED_SERIAL
    from wdpm_b200.stripes import StripeSolver, connect_in_process, plan_stripes
    if variant == 18 and dt == np.float32:
        variant = 15  # the fp32 test window of the warp-autonomous kernel
    rng = np.random.default_rng(83)
    rows, cols = 130, 300
    D0, W0 = random_case(rng, rows, cols, dt)
    plan = plan_stripes(rows, n_stripes)
    border = plan[1].row0
    n_it = 7
    for o in ((border, 100), (border - 1, 101), (border + 1, 150)) if module == 2 else ((1, 1),):
        D, W, outlet = _place_outlet(D0, W0, o)
        dem, w0 = D[1:-1, 1:-1], W[1:-1, 1:-1]
        ref = W.copy()
        td_ref = oracle.iterate(ref, D, NODATA, module, n_it, schedule=po.SCHED_SERIAL, outlet=outlet, totaldrain=0.5)
        ss = [StripeSolver(rows, cols, NODATA, module, st, dtype=_code(dt), fused_variant=variant, fused_chunk_rows=21,
                           schedule=SCHED_SERIAL) for st in plan]
        connect_in_process(ss)
        for s, st in zip(ss, plan):
            s.upload_band(dem[st.band_row0:st.band_row0 + st.band_rows], w0[st.band_row0:st.band_row0 + st.band_rows])
            if module == 2:
                s.set_outlet(*outlet)
                s.set_total_drain(0.5 if st.row0 <= outlet[0] < st.row0 + st.rows else 0.0)
        _lockstep(ss, n_it)
        full = np.concatenate([s.download_owned() for s in ss], axis=0)
        td = sum(s.get_total_drain() for s in ss)
        for s in ss:
            s.close()
        assert _same(full, np.ascontiguousarray(ref[1:-1, 1:-1])), (outlet, int((full != ref[1:-1, 1:-1]).sum()))
        if module == 2:
            assert dt(td) == dt(td_ref), (outlet, td, td_ref)


@pytest.mark.parametrize("module,n_stripes,dtype", [(2, 2, "f64"), (2, 3, "f32"), (1, 3, "f64")])
def test_serial_free_running_stripes(cuda_lib, module, n_stripes, dtype):
    import sys
    from pathlib import Path
    script = Path(__file__).resolve().parent / "stripes_freerun_serial_check.py"
    res = subprocess.run([sys.executable, str(script), str(n_stripes), str(module), "21", "23", dtype],
                         capture_output=True, text=True, timeout=600)
    assert "FREERUN_EQUAL" in res.stdout, res.stdout[-1000:] + res.stderr[-2000:]


def test_refusals(cuda_lib):
    from wdpm_b200 import SCHED_SERIAL, Solver, WdpmError
    with pytest.raises(WdpmError) as ei:
        Solver(20, 20, NODATA, 2, schedule=7)
    assert ei.value.code == -1
    D, W = random_case(np.random.default_rng(1), 20, 20, np.float64)
    with Solver(20, 20, NODATA, 2, schedule=SCHED_SERIAL) as s:
        s.upload(D[1:-1, 1:-1], W[1:-1, 1:-1])
        with pytest.raises(WdpmError) as ei:
            s.set_outlets([(3, 3), (10, 10)])
        assert ei.value.code == -5
        s.set_outlets([(3, 3)])
    with pytest.raises(WdpmError) as ei:  # two iterations per launch: the emptying cannot sit between them
        Solver(20, 20, NODATA, 2, schedule=SCHED_SERIAL, kernel=2, fused_variant=3)
    assert ei.value.code == -5


# ---- the command line against the unmodified reference's serial outputs ------------------------------------------

@pytest.fixture(scope="module")
def host_bin(cuda_lib):
    from wdpm_b200 import build
    return build.build_host()


def _normalise(report: str) -> list[str]:
    """test_cli's normalisation with this backend's lines: the serial reference prints one backend line, this
    host two."""
    import re
    out = []
    for ln in report.split("\n"):
        if re.search(r"(DEM|Water|Output|Scratch) file:", ln) or "for Computation" in ln or "serial-branch arithmetic" in ln \
                or "Run Time" in ln:
            continue
        toks = ln.split()
        if toks and toks[0].isdigit() and len(toks) in (3, 5):  # per-block line: drop the run-time column
            ln = " ".join(toks[:-1])
        out.append(ln.rstrip())
    return out


def _sequence(dem, tmp_path):
    add, drain, sub = tmp_path / "add.asc", tmp_path / "drain.asc", tmp_path / "sub.asc"
    return [("add10", f"add {dem} NULL {add} NULL 10 1.0 1.0 0 1 0.005 0", add),
            ("drain", f"drain {dem} {add} {drain} NULL 0.1 1.0 0 1 0.005 0", drain),
            ("sub10", f"subtract {dem} {drain} {sub} NULL 10 1.0 0 1 0.005 0", sub)]


def _check_outputs(runs, stdouts):
    from test_oracle import _check_goldens
    for (name, _, out), stdout in zip(runs, stdouts):
        text = out.read_text()
        assert text == golden_text(f"ref_serial_{name}.asc.gz"), name
        _check_goldens(name, text)
        assert "serial-branch arithmetic on CUDA" in stdout, name
        assert _normalise(stdout) == _normalise((GOLDEN / f"ref_serial_{name}.txt").read_text()), name


@pytest.mark.parametrize("kernel", ["0", "2"])
def test_cpu0_validation_sequence_matches_the_serial_reference(host_bin, tmp_path, kernel):
    dem = gunzip_to("basin5.asc.gz", tmp_path / "basin5.asc")
    runs = _sequence(dem, tmp_path)
    outs = []
    for name, argv, _ in runs:
        res = subprocess.run([str(host_bin)] + argv.split(), capture_output=True, text=True, timeout=900,
                             env=dict(os.environ, WDPM_B200_KERNEL=kernel))
        assert res.returncode == 0, res.stdout[-500:] + res.stderr
        outs.append(res.stdout)
    _check_outputs(runs, outs)


@pytest.mark.parametrize("gpus", ["1", "2"])
def test_cpu0_chain_matches_the_serial_reference(host_bin, tmp_path, gpus):
    import torch
    from test_oracle import _check_goldens
    if int(gpus) > torch.cuda.device_count():
        pytest.skip(f"needs {gpus} GPUs")
    dem = gunzip_to("basin5.asc.gz", tmp_path / "basin5.asc")
    runs = _sequence(dem, tmp_path)
    pfs = []
    for name, body, _ in runs:
        pf = tmp_path / f"{name}.txt"
        pf.write_text(body + "\n")
        pfs.append(str(pf))
    res = subprocess.run([str(host_bin), "chain"] + pfs, capture_output=True, text=True, timeout=900,
                         env=dict(os.environ, WDPM_B200_GPUS=gpus))
    assert res.returncode == 0, res.stdout[-800:] + res.stderr
    for name, _, out in runs:
        text = out.read_text()
        assert text == golden_text(f"ref_serial_{name}.asc.gz"), name
        _check_goldens(name, text)
    want = []
    for name, _, _ in runs:
        want += _normalise((GOLDEN / f"ref_serial_{name}.txt").read_text())
    assert [ln for ln in _normalise(res.stdout) if ln] == [ln for ln in want if ln]


def test_cpu0_on_two_gpus_matches_the_serial_reference(host_bin, tmp_path):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    dem = gunzip_to("basin5.asc.gz", tmp_path / "basin5.asc")
    runs = _sequence(dem, tmp_path)
    outs = []
    for name, argv, _ in runs:
        res = subprocess.run([str(host_bin)] + argv.split(), capture_output=True, text=True, timeout=900,
                             env=dict(os.environ, WDPM_B200_GPUS="2"))
        assert res.returncode == 0, res.stdout[-500:] + res.stderr
        outs.append(res.stdout)
    _check_outputs(runs, outs)
