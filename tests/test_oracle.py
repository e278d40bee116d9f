"""CPU: pin the oracle (oracle/wdpm_oracle_impl.h) against the reference.

1. raw-precision vectors produced by the VERBATIM runoff.cl (tests/golden/crop_vectors.npz);
2. the verbatim kernels live, when oracle/_ref was built (a reference checkout at pyoracle.reference_dir());
3. the unmodified WDPMCL.c's output files for validate_WDPM.sh's Add -> Drain -> Subtract sequence
   on basin5, both backends, byte for byte, through the host logic of wdpm_b200/wdpmcl.py;
4. the validation/ goldens (validate_WDPM.sh:48-70) via a restatement of the awk checks, and via the
   reference's own awk scripts when that checkout is there.
"""
import subprocess

import numpy as np
import pytest

from conftest import GOLDEN, golden_text, random_case
from oracle import pyoracle as po
from oracle_backend import factory
from wdpm_b200 import ascgrid
from wdpm_b200.wdpmcl import ModuleParams, run_module

MODS = [("add", po.ADD), ("subtract", po.SUBTRACT), ("drain", po.DRAIN)]


@pytest.mark.parametrize("dn,dt", [("f64", np.float64), ("f32", np.float32)])
@pytest.mark.parametrize("mn,mod", MODS)
def test_oracle_matches_verbatim_kernel_vectors(oracle, dn, dt, mn, mod):
    g = np.load(GOLDEN / "crop_vectors.npz")
    D = ascgrid.pad_grid(g["dem"].astype(dt), dt(g["nodata"]))
    w = g[f"w0_{dn}"].copy()
    td = oracle.iterate(w, D, float(g["nodata"]), mod, int(g["iters"]), outlet=tuple(int(x) for x in g["outlet"]))
    assert np.array_equal(w, g[f"w_{mn}_{dn}"])
    assert dt(td) == g[f"td_{mn}_{dn}"]


# edge shapes with NODATA holes, Drain's totaldrain starting non-zero: run live through the verbatim kernels when
# oracle/_ref is built, and stored from such a run in tests/golden/live_vectors.npz (make_golden.py writes it)
LIVE_SEED, LIVE_SHAPES, LIVE_ITERS, LIVE_TD0 = 11, ((1, 1), (2, 5), (31, 47), (64, 96), (97, 33)), 40, 0.5


def live_cases(oracle, dt):
    """(rows, cols, D, W, outlet) for each of LIVE_SHAPES, drawn from LIVE_SEED."""
    rng = np.random.default_rng(LIVE_SEED)
    for rows, cols in LIVE_SHAPES:
        D, W = random_case(rng, rows, cols, dt)
        yield rows, cols, D, W, oracle.find_outlet(D) or (1, 1)


@pytest.mark.parametrize("dt", [np.float64, np.float32])
@pytest.mark.parametrize("mn,mod", MODS)
def test_oracle_matches_verbatim_kernel_live(oracle, refcl, dt, mn, mod):
    for rows, cols, D, W, outlet in live_cases(oracle, dt):
        a, b = W.copy(), W.copy()
        ta = oracle.iterate(a, D, -99999.0, mod, LIVE_ITERS, outlet=outlet, totaldrain=LIVE_TD0)
        tb = refcl.iterate(b, D, -99999.0, mod, LIVE_ITERS, outlet=outlet, totaldrain=LIVE_TD0)
        assert np.array_equal(a, b), (rows, cols)
        assert ta == tb


@pytest.mark.parametrize("dn,dt", [("f64", np.float64), ("f32", np.float32)])
@pytest.mark.parametrize("mn,mod", MODS)
def test_oracle_matches_verbatim_kernel_stored(oracle, dn, dt, mn, mod):
    """The live test's cases, inputs and outputs as the verbatim kernels produced them (tests/golden/live_vectors.npz)."""
    if not (GOLDEN / "live_vectors.npz").exists():
        pytest.skip("tests/golden/live_vectors.npz not generated yet (make_golden.py --live-only, with the reference checkout)")
    g = np.load(GOLDEN / "live_vectors.npz")
    for k, (rows, cols) in enumerate(LIVE_SHAPES):
        D, w = g[f"{dn}_{k}_dem"], g[f"{dn}_{k}_w0"].copy()
        assert D.dtype == dt and D.shape == (rows + 2, cols + 2)
        td = oracle.iterate(w, D, -99999.0, mod, LIVE_ITERS, outlet=tuple(int(x) for x in g[f"{dn}_{k}_outlet"]), totaldrain=LIVE_TD0)
        assert np.array_equal(w, g[f"{mn}_{dn}_{k}_w"]), (rows, cols)
        assert dt(td) == g[f"{mn}_{dn}_{k}_td"], (rows, cols)


def test_serial_add_equals_opencl_add(oracle):
    """runoffs (serial Add) is bit-identical to runoffadd (SURVEY 8a, a8)."""
    rng = np.random.default_rng(3)
    D, W = random_case(rng, 60, 70, np.float64)
    a, b = W.copy(), W.copy()
    oracle.iterate(a, D, -99999.0, po.ADD, 60, schedule=po.SCHED_OPENCL)
    oracle.iterate(b, D, -99999.0, po.ADD, 60, schedule=po.SCHED_SERIAL)
    assert np.array_equal(a, b)


def test_find_outlet_rule(oracle):
    d = np.full((4, 5), 10.0)
    d[1, 2] = 3.0
    d[2, 1] = 3.0   # tie: the first in row-major order wins
    d[3, 3] = -5.0  # <= 0 is never an outlet, even though it is above nodata
    D = ascgrid.pad_grid(d, -99999.0)
    assert oracle.find_outlet(D) == (2, 3)
    assert oracle.find_outlet(ascgrid.pad_grid(np.full((3, 3), -1.0), -99999.0)) is None


def _awk_like(text: str):
    """Restatement of validation/{add,drain,subtract}_test.awk: volume over cells >= 0 and the
    patch sum over file lines 268-269, fields 59-61 (validate_WDPM.sh:46-49)."""
    lines = text.split("\n")
    cellsize = float(lines[4].split()[1])
    vol = 0.0
    count = 0
    patch = 0.0
    for nr, line in enumerate(lines[6:], start=7):
        for i, tok in enumerate(line.split(), start=1):
            v = float(tok)
            if v >= 0:
                vol += v * cellsize * cellsize
                count += 1
                if 59 <= i <= 61 and 268 <= nr <= 269:
                    patch += v
    return vol, count, patch, cellsize


def _check_goldens(step, text):
    vol, count, patch, cs = _awk_like(text)
    tol = 1e-4
    if step == "add10":
        spec = 10 / 1000 * count * cs * cs
        assert abs(vol - spec) / spec <= tol
        assert abs(patch - 0.420810) / 0.420810 <= tol
    elif step == "drain":
        assert abs(vol - 97577.54) / 97577.54 <= tol
        assert abs(patch - 0.420810) / 0.420810 <= tol
    else:
        assert abs(vol - 86762.40) / 86762.40 <= tol
        assert abs(patch - 0.360810) / 0.360810 <= tol


def _asc_text(hdr, water, tmp_path):
    p = tmp_path / "out.asc"
    ascgrid.write_asc(p, hdr, water)
    return p, p.read_text()


@pytest.mark.parametrize("backend_name,sched", [("opencl", po.SCHED_OPENCL), ("serial", po.SCHED_SERIAL)])
def test_validation_sequence_matches_reference_outputs(oracle, basin5, tmp_path, backend_name, sched):
    """Add 10 mm -> Drain -> Subtract 10 mm (validate_WDPM.sh:77,88,99) reproduces the reference's
    output files byte for byte and passes the validation goldens."""
    hdr, dem = basin5
    be = factory(np.float64, sched)
    steps = [
        ("add10", ModuleParams("add", depth_mm=10, runoff_fraction=1.0, elevation_tol_mm=1.0, zero_threshold_mm=0.005)),
        ("drain", ModuleParams("drain", elevation_tol_mm=0.1, drain_tol_m3=1.0, zero_threshold_mm=0.005)),
        # validate_WDPM.sh:99 - $subtract_elev_tol is undefined, so runoff_frac (1.0) lands in the tolerance slot
        ("sub10", ModuleParams("subtract", depth_mm=10, elevation_tol_mm=1.0, zero_threshold_mm=0.005)),
    ]
    water = None
    iters = {"add10": 30000, "drain": 11000, "sub10": 1000}
    for name, params in steps:
        rep = run_module(dem, hdr.nodata, hdr.cellsize, params, water=water, backend=be)
        assert rep.iterations == iters[name]
        path, text = _asc_text(hdr, rep.water, tmp_path)
        assert text == golden_text(f"ref_{backend_name}_{name}.asc.gz"), name
        _check_goldens(name, text)
        ref = po.reference_dir()
        if ref is not None and (ref / "validation").is_dir():
            awk_dir = ref / "validation"
            script = {"add10": "add_test.awk", "drain": "drain_test.awk", "sub10": "subtract_test.awk"}[name]
            extra = {"add10": ["-v", "add_depth=10", "-v", "specified_patch_depth=0.420810"],
                     "drain": ["-v", "specified_drain_vol=97577.54", "-v", "drain_row=333", "-v", "drain_col=468",
                               "-v", "specified_patch_depth=0.420810"],
                     "sub10": ["-v", "specified_subtract_vol=86762.40=", "-v", "specified_patch_depth=0.360810"]}[name]
            out = subprocess.run(["awk", "-f", str(awk_dir / script), "-v", "vol_tolerance=0.0001", "-v", "patch_top=268",
                                  "-v", "patch_bottom=269", "-v", "patch_left=59", "-v", "patch_right=61", *extra, str(path)],
                                 capture_output=True, text=True, check=True).stdout
            assert "failed" not in out and out.count("passed") >= 2, out
        # the next module reads this module's output FILE: values quantised by "%f", NODATA cells = -99999
        _, water = ascgrid.read_asc(path)


def test_drain_report_matches_reference_log(oracle, basin5):
    """Drain's outlet, totaldrain and per-block lines agree with the reference's stdout."""
    hdr, dem = basin5
    _, water = ascgrid.read_asc(GOLDEN / "ref_opencl_add10.asc.gz")
    rep = run_module(dem, hdr.nodata, hdr.cellsize, ModuleParams("drain", elevation_tol_mm=0.1, drain_tol_m3=1.0,
                                                                   zero_threshold_mm=0.005), water=water, backend=factory())
    log = (GOLDEN / "ref_opencl_drain.txt").read_text()
    assert f"Drain column: {rep.outlet[1]}" in log and f"Drain row: {rep.outlet[0]}" in log
    ref_lines = [ln.split() for ln in log.split("\n") if ln.strip() and ln.split()[0].isdigit() and len(ln.split()) == 5]
    assert len(ref_lines) == len(rep.blocks)
    for ref, blk in zip(ref_lines, rep.blocks):
        assert int(ref[0]) == blk.iterations
        assert ref[1] == "%8.3f" % blk.max_diff or ref[1] == ("%8.3f" % blk.max_diff).strip()
        assert ref[2] == ("%10.1f" % blk.vol_change).strip()
        assert ref[3] == ("%12.1f" % blk.water_left).strip()
    assert "%10.2f" % rep.drain_vol in log          # Volume drained
    assert "%10.2f" % rep.final_vol in log          # Final volume
    assert "%10.4f" % rep.water_frac in log         # Final water coverage
    assert "%10.2f" % (rep.mean_water * 1000.0) in log
    assert "%10.2f" % rep.max_depth_mm in log


def test_outlet_set_extension_reduces_to_the_reference_for_one_outlet(oracle):
    """oracle.iterate_outlets (the many-outlets extension) with ONE outlet is runoffdrain."""
    rng = np.random.default_rng(41)
    for dt in (np.float64, np.float32):
        D, W = random_case(rng, 37, 52, dt)
        outlet = oracle.find_outlet(D)
        a, b = W.copy(), W.copy()
        ta = oracle.iterate(a, D, -99999.0, po.DRAIN, 6, outlet=outlet, totaldrain=0.25)
        tb = oracle.iterate_outlets(b, D, -99999.0, 6, [outlet], totals=[0.25])
        assert np.array_equal(a, b) and dt(ta) == tb[0]
