"""Exact checkpoints: the capture of wdpm_checkpoint_arm / wdpm_checkpoint_wait is the state a block starts from, a
fresh solver fed with it continues the run bit for bit (other kernel, other partition), and the command line's
WDPM_B200_CHECKPOINT / WDPM_B200_RESUME reproduce the unmodified reference's outputs across a resume."""
import os
import re
import subprocess

import numpy as np
import pytest

from conftest import GOLDEN, golden_text, gunzip_to, random_case

pytestmark = pytest.mark.gpu

NODATA = -99999.0
THRES = 0.02  # clamps a few per cent of the cells at every prologue


def _code(dt):
    from wdpm_b200 import F32, F64
    return F64 if dt == np.float64 else F32


def _bits(a):
    return np.ascontiguousarray(a).view(np.uint64 if a.dtype == np.float64 else np.uint32)


def _same(a, b):
    return a.shape == b.shape and np.array_equal(_bits(a), _bits(b))


# ---- solver sets: one solver, or in-process row stripes on one GPU driven in lockstep or free-running -------------

class Run:
    def __init__(self, rows, cols, module, dt, n_stripes=0, driver="free", schedule=0, **kw):
        from wdpm_b200 import Solver
        from wdpm_b200.stripes import StripeSolver, connect_in_process, plan_stripes
        self.module, self.dt, self.driver, self.n_out = module, dt, driver, 1
        if n_stripes:
            self.plan = plan_stripes(rows, n_stripes)
            self.ss = [StripeSolver(rows, cols, NODATA, module, st, dtype=_code(dt), zero_threshold=THRES, fused_chunk_rows=21,
                                    schedule=schedule, **kw) for st in self.plan]
            connect_in_process(self.ss)
        else:
            self.plan = None
            self.ss = [Solver(rows, cols, NODATA, module, dtype=_code(dt), zero_threshold=THRES, schedule=schedule, **kw)]

    def upload(self, dem, w):
        if self.plan is None:
            self.ss[0].upload(dem, w)
        for s, st in zip(self.ss, self.plan or []):
            sl = slice(st.band_row0, st.band_row0 + st.band_rows)
            s.upload_band(dem[sl], w[sl])

    def outlets(self, outlets, totals=None):
        self.n_out = len(outlets)
        for s in self.ss:
            s.set_outlets(outlets)
            if totals is None:
                s.seed_outlet_drains()
            else:
                s.set_outlet_drains(totals)

    def block(self, n):
        from wdpm_b200.stripes import combine_block_results
        if self.plan is None:
            return self.ss[0].run_block(n)
        for s in self.ss:
            s.block_begin()
        if self.driver == "lockstep":
            for _ in range(n):
                for ph in (0, 1):
                    for s in self.ss:
                        s.phase(ph)
                    for s in self.ss:
                        s.synchronize()
        else:
            for done in range(0, n, 3):
                for s in self.ss:
                    s.block_enqueue(min(3, n - done))
        r = combine_block_results([s.block_end() for s in self.ss])
        if self.module == 2:  # the single-solver total: the outlets' totals added in outlet order, solver precision
            acc = self.dt(0)
            for v in self.totals().astype(self.dt):
                acc = self.dt(acc + v)
            r.total_drain = float(acc)
        return r

    def water(self):
        if self.plan is None:
            return self.ss[0].download_water()
        return np.concatenate([s.download_owned() for s in self.ss])

    def totals(self):
        return sum(s.get_outlet_drains(self.n_out) for s in self.ss)

    def arm(self):
        for s in self.ss:
            s.checkpoint_arm()

    def capture(self):
        caps = [s.checkpoint_wait() for s in self.ss]
        return np.concatenate([c[0] for c in caps]), sum(c[1] for c in caps)

    def close(self):
        for s in self.ss:
            s.close()


def _case(dt, rows=90, cols=400, seed=7):
    D, W = random_case(np.random.default_rng(seed), rows, cols, dt)
    return np.ascontiguousarray(D[1:-1, 1:-1]), np.ascontiguousarray(W[1:-1, 1:-1])


def _setup(run, case, dem, w, resume=False, totals=None, outlet=None):
    """Module initial conditions for `case` (a resumed run takes the water and totals as they are); returns the
    outlet list of a Drain case."""
    from wdpm_b200 import ascgrid
    run.upload(dem, w)
    if case == "add" and not resume:
        for s in run.ss:
            s.apply_add(0.01, 0.5)
    if case in ("sub", "sub-serial") and not resume:
        for s in run.ss:
            s.apply_subtract(0.01)
    if case in ("drain-ref", "drain-serial"):
        if outlet is None:
            with _single_like(run, dem, w) as probe:
                outlet = probe.find_outlet()[:2]
        run.outlets([outlet], totals)
        return [outlet]
    if case == "drain-rim":
        rim = ascgrid.rim_outlets(dem, NODATA)
        run.outlets(rim, totals)
        return rim
    return None


def _single_like(run, dem, w):
    from wdpm_b200 import Solver
    s = Solver(dem.shape[0], dem.shape[1], NODATA, run.module, dtype=_code(run.dt), zero_threshold=THRES)
    s.upload(dem, w)
    return s


CASES = {"add": (0, 0), "sub": (1, 0), "drain-ref": (2, 0), "drain-rim": (2, 0), "sub-serial": (1, 1), "drain-serial": (2, 1)}


def _kernels(dt):
    from wdpm_b200 import KERNEL_COLOUR, KERNEL_FUSED, KERNEL_RESIDENT
    from wdpm_b200.solver import PRODUCTION_FUSED_VARIANT_F32, PRODUCTION_FUSED_VARIANT_F64
    prod = PRODUCTION_FUSED_VARIANT_F64 if dt == np.float64 else PRODUCTION_FUSED_VARIANT_F32
    return {"colour": dict(kernel=KERNEL_COLOUR), "fused-small": dict(kernel=KERNEL_FUSED, fused_variant=2),
            "fused-production": dict(kernel=KERNEL_FUSED, fused_variant=prod), "resident": dict(kernel=KERNEL_RESIDENT)}


# ---- 1. the capture is the block-start state -----------------------------------------------------------------------

@pytest.mark.parametrize("dt", [np.float64, np.float32])
@pytest.mark.parametrize("kname", ["colour", "fused-small", "fused-production", "resident"])
@pytest.mark.parametrize("case", list(CASES))
def test_capture_is_the_block_start_state(cuda_lib, dt, kname, case):
    module, schedule = CASES[case]
    dem, w = _case(dt)
    run = Run(*dem.shape, module, dt, schedule=schedule, **_kernels(dt)[kname])
    try:
        _setup(run, case, dem, w)
        for _ in range(2):
            run.block(7)
        after, tot = run.water(), run.totals()
        run.arm()
        run.block(7)
        cw, ct = run.capture()
        assert _same(cw, np.where(after < dt(THRES), dt(0), after).astype(dt))
        assert _same(ct, tot)
    finally:
        run.close()


# ---- 2. a fresh solver fed with the capture continues bit for bit ----------------------------------------------------

RESUMES = [  # (case, dtype, first run, second run); a run = (stripes, driver, kernel name)
    ("add", np.float64, (0, None, "fused-production"), (0, None, "colour")),
    ("drain-rim", np.float64, (0, None, "fused-production"), (3, "free", "fused-small")),
    ("drain-ref", np.float32, (2, "lockstep", "fused-small"), (0, None, "resident")),
    ("sub-serial", np.float64, (0, None, "resident"), (2, "free", "fused-production")),
    ("drain-serial", np.float64, (3, "lockstep", "fused-small"), (0, None, "fused-production")),
    ("drain-rim", np.float32, (2, "free", "fused-production"), (3, "lockstep", "fused-small")),
    ("sub", np.float32, (0, None, "fused-production"), (2, "lockstep", "fused-production")),
]


@pytest.mark.parametrize("case,dt,first,second", RESUMES)
def test_resume_is_bit_for_bit(cuda_lib, case, dt, first, second):
    module, schedule = CASES[case]
    dem, w = _case(dt, rows=130, cols=300, seed=11)
    B, n = 3, 9
    a = Run(*dem.shape, module, dt, n_stripes=first[0], driver=first[1], schedule=schedule, **_kernels(dt)[first[2]])
    try:
        outlets = _setup(a, case, dem, w)
        ra = []
        for b in range(2 * B):
            if b == B:
                a.arm()  # arming changes nothing in the run itself
            ra.append(a.block(n))
        cw, ct = a.capture()
        wa, ta = a.water(), a.totals()
    finally:
        a.close()
    c = Run(*dem.shape, module, dt, n_stripes=second[0], driver=second[1], schedule=schedule, **_kernels(dt)[second[2]])
    try:
        _setup(c, case, dem, cw, resume=True, totals=ct if module == 2 else None, outlet=outlets[0] if outlets and case != "drain-rim" else None)
        rc = [c.block(n) for _ in range(B)]
        wc, tc = c.water(), c.totals()
    finally:
        c.close()
    same_partition = first[0] == second[0] == 0
    for x, y in zip(ra[B:], rc):
        assert (x.max_diff, x.total_drain, x.wet_cells) == (y.max_diff, y.total_drain, y.wet_cells)
        if same_partition:
            assert x.masked_sum == y.masked_sum
        else:
            assert abs(x.masked_sum - y.masked_sum) <= 1e-12 * abs(x.masked_sum)
    assert _same(wa, wc)
    if module == 2:
        assert _same(ta, tc)


# ---- 3. ordering is kept on the device ------------------------------------------------------------------------------

def test_capture_outlasting_blocks_is_still_the_boundary_state(cuda_lib):
    """8192^2 fp64 with 10-iteration blocks: the 0.5 GB copy outlasts a block. The next two blocks are enqueued
    before anyone waits; their prologues must wait for the copy on the device."""
    from wdpm_b200 import ADD, F64, Solver
    n = 8192
    rng = np.random.default_rng(3)
    dem = (500 + 3 * rng.standard_normal((n, n))).round(4)
    w = rng.uniform(0, 0.05, (n, n))
    with Solver(n, n, NODATA, ADD, dtype=F64, zero_threshold=THRES) as s:
        s.upload(dem, w)
        s.run_block(10)
        after = s.download_water()
        s.checkpoint_arm()
        for _ in range(3):
            s.block_begin()
            s.block_enqueue(10)
            s.block_end()
        cw, ct = s.checkpoint_wait()
    assert _same(cw, np.where(after < THRES, 0.0, after))
    assert ct.shape == (1,)


# ---- 4. set_outlet_drains ---------------------------------------------------------------------------------------------

def test_set_outlet_drains(cuda_lib):
    from wdpm_b200 import ADD, DRAIN, F64, Solver, WdpmError, ascgrid
    from wdpm_b200.stripes import StripeSolver, connect_in_process, plan_stripes
    dem, w = _case(np.float64, rows=60, cols=90)
    rim = ascgrid.rim_outlets(dem, NODATA)
    vals = np.random.default_rng(5).uniform(0, 1, len(rim))
    with Solver(60, 90, NODATA, DRAIN, dtype=F64) as s:
        s.upload(dem, w)
        s.set_outlets(rim)
        s.set_outlet_drains(vals)
        assert _same(s.get_outlet_drains(len(rim)), vals)
        with pytest.raises(WdpmError) as ei:
            s.set_outlet_drains(vals[:-1])
        assert ei.value.code == -1
    with Solver(60, 90, NODATA, ADD, dtype=F64) as s:
        s.upload(dem, w)
        with pytest.raises(WdpmError) as ei:
            s.set_outlet_drains([0.0])
        assert ei.value.code == -4
    plan = plan_stripes(60, 2)
    ss = [StripeSolver(60, 90, NODATA, DRAIN, st, dtype=F64, fused_variant=2) for st in plan]
    connect_in_process(ss)
    for s, st in zip(ss, plan):
        sl = slice(st.band_row0, st.band_row0 + st.band_rows)
        s.upload_band(dem[sl], w[sl])
        s.set_outlets(rim)
        s.set_outlet_drains(vals)
    parts = [s.get_outlet_drains(len(rim)) for s in ss]
    for s in ss:
        s.close()
    rows = np.array([r for r, _ in rim])
    for p, st in zip(parts, plan):
        own = (rows >= st.row0) & (rows < st.row0 + st.rows)
        assert _same(p[own], vals[own]) and not p[~own].any()
    assert _same(parts[0] + parts[1], vals)


def test_outlet_set_installed_after_the_arm(cuda_lib):
    """The capture is sized by the set installed when the block begins, not by the one at the arm: arm with the
    reference's single outlet, install the rim, run a block; the capture holds every rim total."""
    from wdpm_b200 import DRAIN, F64, Solver, ascgrid
    dem, w = _case(np.float64, rows=120, cols=300)
    rim = ascgrid.rim_outlets(dem, NODATA)
    assert len(rim) > 500
    vals = np.random.default_rng(6).uniform(0, 1, len(rim))
    with Solver(120, 300, NODATA, DRAIN, dtype=F64, zero_threshold=THRES) as s:
        s.upload(dem, w)
        s.find_outlet()
        s.checkpoint_arm()
        s.run_block(3)
        assert s.checkpoint_wait()[1].shape == (1,)
        s.checkpoint_arm()
        s.set_outlets(rim)
        s.set_outlet_drains(vals)
        s.run_block(3)
        cw, ct = s.checkpoint_wait()
    assert _same(ct, vals)


# ---- 5-7. the command line ---------------------------------------------------------------------------------------------

@pytest.fixture(scope="module")
def host_bin(cuda_lib):
    from wdpm_b200 import build
    return build.build_host()


def _normalise(report: str) -> list[str]:
    out = []
    for ln in report.split("\n"):
        if re.search(r"(DEM|Water|Output|Scratch) file:", ln) or "for Computation" in ln or "backend flags" in ln \
                or "serial-branch arithmetic" in ln or "Run Time" in ln:
            continue
        toks = ln.split()
        if toks and toks[0].isdigit() and len(toks) in (3, 5):  # per-block line: drop the run-time column
            ln = " ".join(toks[:-1])
        out.append(ln.rstrip())
    return out


def _from(report: str, k: int) -> list[str]:
    """Block lines from iteration k on, and the summary."""
    lines = _normalise(report)
    first = next(i for i, ln in enumerate(lines) if ln.split()[:1] == [str(k)])
    return lines[first:]


def _run(host_bin, argv, **env):
    res = subprocess.run([str(host_bin)] + [str(x) for x in argv], capture_output=True, text=True, timeout=900,
                         env=dict(os.environ, **{k: str(v) for k, v in env.items()}))
    return res


def _ok(res):
    assert res.returncode == 0, res.stdout[-800:] + res.stderr
    return res.stdout


def _add(dem, out, tol="1.0", cpu="1", limit="0"):
    return ["add", dem, "NULL", out, "NULL", "10", "1.0", tol, cpu, "1", "0.005", limit]


def _drain(dem, water, out, cpu="1"):
    return ["drain", dem, water, out, "NULL", "0.1", "1.0", cpu, "1", "0.005", "0"]


@pytest.fixture(scope="module")
def basin(tmp_path_factory):
    d = tmp_path_factory.mktemp("basin5")
    return d, gunzip_to("basin5.asc.gz", d / "basin5.asc")


def _checkpointed_then_resumed(host_bin, tmp, argv_of, golden_asc, golden_txt, resume_at, **env):
    """Run with checkpoints every block, then resume from the one at `resume_at`; both outputs must equal the golden
    file and the resumed report the golden's lines from resume_at + 1000 on."""
    full = tmp / "full.asc"
    out = _ok(_run(host_bin, argv_of(full), WDPM_B200_CHECKPOINT=tmp / "ck_%d.bin", **env))
    assert full.read_text() == golden_asc
    last = max(int(m.group(1)) for p in tmp.glob("ck_*.bin") if (m := re.match(r"ck_(\d+)\.bin$", p.name)))
    assert all((tmp / f"ck_{k}.bin").exists() for k in range(1000, last + 1, 1000))
    resume_at = resume_at or max(1000, last // 2000 * 1000)
    assert resume_at < last
    assert not list(tmp.glob("*.tmp"))
    res = tmp / "resumed.asc"
    env.pop("WDPM_B200_GPUS", None)
    rout = _ok(_run(host_bin, argv_of(res), WDPM_B200_RESUME=tmp / f"ck_{resume_at}.bin", **env))
    assert "Checkpoint found" in rout and f"Resuming at iteration: {resume_at}" in rout
    assert res.read_text() == golden_asc
    assert _from(rout, resume_at + 1000) == _from(golden_txt, resume_at + 1000)
    return out, rout


def test_cli_add_resume_matches_the_reference(host_bin, basin, tmp_path):
    _, dem = basin
    _checkpointed_then_resumed(host_bin, tmp_path, lambda o: _add(dem, o), golden_text("ref_opencl_add10.asc.gz"),
                               (GOLDEN / "ref_opencl_add10.txt").read_text(), 10000)


@pytest.mark.parametrize("cpu,ref", [("1", "opencl"), ("0", "serial")])
def test_cli_drain_resume_matches_the_reference(host_bin, basin, tmp_path, cpu, ref):
    _, dem = basin
    water = gunzip_to(f"ref_{ref}_add10.asc.gz", tmp_path / "add.asc")
    _checkpointed_then_resumed(host_bin, tmp_path, lambda o: _drain(dem, water, o, cpu), golden_text(f"ref_{ref}_drain.asc.gz"),
                               (GOLDEN / f"ref_{ref}_drain.txt").read_text(), 10000)


def test_cli_drain_rim_resume(host_bin, basin, tmp_path):
    _, dem = basin
    water = gunzip_to("ref_opencl_add10.asc.gz", tmp_path / "add.asc")
    ref, ref_csv = tmp_path / "ref.asc", tmp_path / "ref.csv"
    ref_out = _ok(_run(host_bin, _drain(dem, water, ref), WDPM_B200_OUTLETS="rim", WDPM_B200_OUTLET_TOTALS=ref_csv))
    csv = tmp_path / "resumed.csv"
    _checkpointed_then_resumed(host_bin, tmp_path, lambda o: _drain(dem, water, o), ref.read_text(), ref_out, None,
                                         WDPM_B200_OUTLETS="rim", WDPM_B200_OUTLET_TOTALS=csv)
    assert csv.read_bytes() == ref_csv.read_bytes()


def test_cli_checkpoint_on_two_gpus_resumes_on_one(host_bin, basin, tmp_path):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    _, dem = basin
    _checkpointed_then_resumed(host_bin, tmp_path, lambda o: _add(dem, o), golden_text("ref_opencl_add10.asc.gz"),
                               (GOLDEN / "ref_opencl_add10.txt").read_text(), 10000, WDPM_B200_GPUS=2)


@pytest.mark.parametrize("first", [dict(limit="10000"), dict(tol="10.0")])
def test_cli_extends_a_finished_run(host_bin, basin, tmp_path, first):
    """A run stopped by its iteration limit, or converged at 10 mm, continues to 1 mm from its end-of-run checkpoint
    and writes what one uninterrupted 1 mm run writes."""
    _, dem = basin
    ck = tmp_path / "ck.bin"
    _ok(_run(host_bin, _add(dem, tmp_path / "first.asc", **first), WDPM_B200_CHECKPOINT=ck))
    out = tmp_path / "out.asc"
    _ok(_run(host_bin, _add(dem, out), WDPM_B200_RESUME=ck))
    assert out.read_text() == golden_text("ref_opencl_add10.asc.gz")


def test_cli_refuses_another_identity(host_bin, basin, tmp_path):
    d, dem = basin
    add_ck, drain_ck = tmp_path / "add.bin", tmp_path / "drain.bin"
    _ok(_run(host_bin, _add(dem, tmp_path / "a.asc", limit="2000"), WDPM_B200_CHECKPOINT=add_ck))
    water = gunzip_to("ref_opencl_add10.asc.gz", tmp_path / "add.asc")
    _ok(_run(host_bin, _drain(dem, water, tmp_path / "d.asc"), WDPM_B200_CHECKPOINT=drain_ck, WDPM_B200_CHECKPOINT_EVERY=100))
    toks = dem.read_text().split()
    k = 12 + 100 * int(toks[1]) + 200  # one cell after the six header pairs
    toks[k] = f"{float(toks[k]) + 0.001:.4f}"
    dem2 = tmp_path / "dem2.asc"
    dem2.write_text(" ".join(toks[:12]) + "\n" + " ".join(toks[12:]) + "\n")
    short = tmp_path / "short.bin"
    short.write_bytes(add_ck.read_bytes()[:-9])
    cases = [
        (_add(dem2, None), add_ck, {}, "another DEM"),
        (_add(dem, None)[:10] + ["0.006", "0"], add_ck, {}, "zero depth threshold"),
        (["subtract", dem, water, None, "NULL", "10", "1.0", "1", "1", "0.005", "0"], add_ck, {}, "another module"),
        (_drain(dem, water, None), drain_ck, {"WDPM_B200_OUTLETS": "rim"}, "other drain outlets"),
        (_add(dem, None, cpu="0"), add_ck, {}, "cpu flag"),
        (_add(dem, None), short, {}, "truncated"),
    ]
    for i, (argv, ck, env, why) in enumerate(cases):
        out = tmp_path / f"refused{i}.asc"
        argv = [out if a is None else a for a in argv]
        res = _run(host_bin, argv, WDPM_B200_RESUME=ck, **env)
        assert res.returncode == 1 and why in res.stderr, (why, res.stdout[-300:], res.stderr)
        assert not out.exists()
