#!/usr/bin/env python
"""Benchmark of the WDPM redistribution path (BASELINE.json: cell-updates/s, 32768^2 DEM).

    python bench.py [--gpus N] [--steps K] [--warmup W]            our CUDA path
    python bench.py --impl reference [...]                         the reference's CPU path, bounded sample
    python bench.py [...] --dump-outputs DIR                       also write what the last timed step computed

`--dump-outputs DIR`: after the K timed steps, DIR/<name>.npy holds what a caller of the timed path receives
from the last of them: `water` (the whole water grid in the run's precision) or, above DUMP_CELLS cells,
`water_sample` (the cells at sample_cells(rows, cols): a fixed, seeded, sorted set of flat row-major indices),
and the block's reductions `max_diff`, `masked_sum`, `total_drain`, `wet_cells` (float64). The DEM is
generated from a fixed seed, so two builds given the same arguments can be compared file by file.

One STEP = one convergence block of the reference's solver loop
(/root/reference/src/WDPMCL.c:1054-1268): zero-threshold + snapshot, 1000 iterations of the nine
colour sub-passes, masked max-difference / water-balance reductions - over the whole DEM.
1 cell-update = one interior cell carried through one iteration, so a step is rows*cols*1000
cell-updates. Workload at every N: BASELINE.json configs[3], the synthetic 32768 x 32768 fractal DEM
(wdpm_b200/synth.py), Add 300 mm, runoff fraction 1.0, zero threshold 0.005 mm, fp64 (the
reference's precision); N > 1 partitions the same DEM into row stripes (strong scaling).

`value`  : device-timed (CUDA events on the solver's stream, max over ranks), grids resident in HBM.
`e2e`    : the same block through the public C-ABI call sequence a host makes per block when it
           round-trips like the reference does (WDPMCL.c:1129-1153, :1217-1233): upload DEM + water
           from pinned host memory, run the block, download the water grid - all inside the timed region.
`roofline`: dominant kernel = the fused iteration kernel; algorithmic bytes per launch =
           cells * 3 * sizeof(T) * iterations_per_launch (read dem, read water, write water once per
           iteration; SURVEY.md 8d) over its mean launch time, measured with CUDA events around the
           launch sequence inside the library.
`cpu_baseline`: the verbatim reference kernels (oracle/_ref/librunoffcl_ref.so, built from
           /root/reference/src/runoff.cl; kind "reference") or, if that binary is absent, the C oracle
           (kind "port"), all host threads, on a window of the SAME DEM in the SAME state the timed GPU
           steps start from.
`cpu_baseline_serial`: the UNMODIFIED reference program (oracle/_ref/WDPMCL_ref = /root/reference/src/WDPMCL.c
           compiled where it lies) with cpu=0 - its serial backend, one core - one 1000-iteration block on a
           512 x 512 window of the same DEM, timed by its own "run time" column (SURVEY.md 8d(i)).
`--impl reference`: the same unmodified program with cpu=1 - its OpenCL branch, carried by the CPU stand-in
           runtime of oracle/ref_shim (every NDRange under OpenMP on all host cores) - one run = one step =
           one 1000-iteration block (the reference's minimum, WDPMCL.c:1285-1287) of Add on a 1024 x 1024
           window of the workload's DEM written as an .asc file; value = cells x 1000 / the program's own
           "run time" of the block (file parsing excluded). `sample` says so; `config` stays the workload's.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

BLOCK_ITERS = 1000
THRES_MM = 0.005
NODATA = -99999.0
MODULES = {"add": 0, "subtract": 1, "drain": 2}
DUMP_CELLS = 1 << 22  # sampled water cells of --dump-outputs: 32 MiB in fp64
DUMP_SEED = 20261020


def sample_cells(rows: int, cols: int) -> np.ndarray:
    """Flat row-major indices of the water cells --dump-outputs writes: all of them up to DUMP_CELLS, else a
    fixed sample drawn from DUMP_SEED (sorted, without repeats)."""
    n = rows * cols
    if n <= DUMP_CELLS:
        return np.arange(n, dtype=np.int64)
    return np.unique(np.random.default_rng(DUMP_SEED).integers(0, n, DUMP_CELLS, dtype=np.int64))


def sampled_rows(idx: np.ndarray, cols: int, row0: int, block: np.ndarray) -> np.ndarray:
    """Values of the sampled cells `idx` (sorted flat indices of the whole grid) that lie in `block`, the grid's rows
    row0 .. row0 + len(block) - 1 (a stripe's owned rows), in index order."""
    lo, hi = np.searchsorted(idx, [row0 * cols, (row0 + block.shape[0]) * cols])
    return block.ravel()[idx[lo:hi] - row0 * cols]


def dump_outputs(out_dir: Path, rows: int, cols: int, water: np.ndarray, r) -> None:
    """Write the water grid (or its sample) and the block reductions `r` of the last timed step."""
    out_dir.mkdir(parents=True, exist_ok=True)
    if rows * cols <= DUMP_CELLS:
        np.save(out_dir / "water.npy", water.reshape(rows, cols))
    else:
        np.save(out_dir / "water_sample.npy", water)
    for name in ("max_diff", "masked_sum", "total_drain", "wet_cells"):
        np.save(out_dir / f"{name}.npy", np.array([getattr(r, name)], dtype=np.float64))


def host_threads() -> int:
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


def use_all_host_threads() -> int:
    """torch.distributed.run exports OMP_NUM_THREADS=1; the CPU legs must use every core they can get. Sets the
    OpenMP runtime's thread count directly (the environment variable is only read when libgomp initialises)."""
    n = host_threads()
    os.environ["OMP_NUM_THREADS"] = str(n)
    try:
        import ctypes
        ctypes.CDLL("libgomp.so.1").omp_set_num_threads(n)
    except Exception:
        pass
    return n


def measured_peak_gbs():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        try:
            return float(json.loads(p.read_text())["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """Samples SM clocks and throttle reasons with NVML while the timed region runs."""

    REASONS = {0x2: "applications_clocks_setting", 0x4: "sw_power_cap", 0x8: "hw_slowdown", 0x20: "sw_thermal_slowdown",
               0x40: "hw_thermal_slowdown", 0x80: "hw_power_brake_slowdown", 0x100: "display_clock_setting"}

    def __init__(self, index: int):
        self.index = index
        self.samples = []
        self.reasons = set()
        self.max_mhz = None
        self._stop = threading.Event()
        self._thread = None

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            self._nv = pynvml
            self._h = pynvml.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = int(pynvml.nvmlDeviceGetMaxClockInfo(self._h, pynvml.NVML_CLOCK_SM))
        except Exception:
            self._nv = None
            return self
        self._thread = threading.Thread(target=self._run, daemon=True)
        self._thread.start()
        return self

    def _run(self):
        nv = self._nv
        while not self._stop.is_set():
            try:
                self.samples.append(int(nv.nvmlDeviceGetClockInfo(self._h, nv.NVML_CLOCK_SM)))
                mask = int(nv.nvmlDeviceGetCurrentClocksEventReasons(self._h))
                for bit, name in self.REASONS.items():
                    if mask & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            self._stop.wait(0.2)

    def stop(self) -> dict:
        self._stop.set()
        if self._thread:
            self._thread.join(timeout=2)
        med = int(np.median(self.samples)) if self.samples else None
        return {"sm_mhz": med, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(self.samples)}


def physical_gpu_index(local_rank: int) -> int:
    vis = os.environ.get("CUDA_VISIBLE_DEVICES")
    if vis:
        try:
            return int(vis.split(",")[local_rank])
        except Exception:
            return local_rank
    return local_rank


# --------------------------------------------------------------------------- reference arm


def warn_no_reference(what: str) -> None:
    print(f"bench.py: WARNING: the reference-derived binaries under oracle/_ref are not built (no reference checkout at "
          f"build time, see oracle/pyoracle.py reference_dir()): {what}", file=sys.stderr)


def cpu_kernel():
    """(callable iterate(w, d, n_iters), kind, threads) - the reference kernels if built, else the port."""
    from oracle import pyoracle as po
    po_o = po.Oracle()
    if po.RefCL.available():
        ref = po.RefCL()
        # keep the column-major layout across calls (the reference flattens once per block)
        import ctypes as C

        class Runner:
            kind = "reference"
            threads = po_o.threads

            def __init__(self, w, d):
                self.wf = np.ascontiguousarray(w.T)
                self.df = np.ascontiguousarray(d.T)
                self.R, self.Cc = w.shape[0] - 2, w.shape[1] - 2
                self.td = np.zeros(1)

            def iterate(self, n):
                ref.lib.refcl_iterate_f64(C.c_int(0), self.wf.ctypes.data_as(C.c_void_p), self.df.ctypes.data_as(C.c_void_p),
                                          C.c_double(NODATA), C.c_int(self.R), C.c_int(self.Cc), C.c_int(n),
                                          self.td.ctypes.data_as(C.c_void_p), C.c_int(0), C.c_int(0))
        return Runner

    warn_no_reference("the CPU baseline times this repository's C port of the kernels (kind 'port')")

    class Runner:  # noqa: F811
        kind = "port"
        threads = po_o.threads

        def __init__(self, w, d):
            self.w, self.d = w, d

        def iterate(self, n):
            po_o.iterate(self.w, self.d, NODATA, po.ADD, n)
    return Runner


def time_cpu_sample(D: np.ndarray, W: np.ndarray, budget_s: float = 12.0):
    """Cell-updates/s of the CPU path on padded window (D, W); iterations chosen to fill ~budget_s."""
    use_all_host_threads()
    Runner = cpu_kernel()
    r = Runner(W.copy(), D)
    cells = (D.shape[0] - 2) * (D.shape[1] - 2)
    t = time.perf_counter()
    r.iterate(4)
    per_it = (time.perf_counter() - t) / 4
    n = int(max(8, min(2000, budget_s / max(per_it, 1e-6))))
    t = time.perf_counter()
    r.iterate(n)
    dt = time.perf_counter() - t
    return cells * n / dt, Runner.kind, Runner.threads, n, dt


def write_sample_asc(path: Path, dem: np.ndarray):
    with open(path, "w") as f:
        f.write("NCOLS %d\nNROWS %d\nXLLCORNER 0\nYLLCORNER 0\nCELLSIZE 10\nNODATA_VALUE %d\n" % (dem.shape[1], dem.shape[0], int(NODATA)))
        np.savetxt(f, dem, fmt="%.4f")


def run_reference_binary(workdir: Path, module: str, add_mm: float, cpu_flag: int, threads: int, iter_limit: int = 1000):
    """One run of the unmodified reference program (oracle/_ref/WDPMCL_ref) on workdir/dem.asc. Returns
    (iterations, its own 'run time' of the last block line in seconds, wall seconds)."""
    import re
    import subprocess
    from oracle import pyoracle as po
    exe = po.ref_binary()
    # WDPMCL.c fopen()s "runoff.cl" in the working directory before building its program (WDPMCL.c:1, :610); the CPU
    # stand-in runtime binds the kernels compiled into the binary and never parses the file, so a placeholder will do
    stub = workdir / "runoff.cl"
    if not stub.exists():
        stub.write_text("/* placeholder: oracle/ref_shim/minicl.c binds the kernels compiled into WDPMCL_ref */\n")
    if module == "add":
        argv = ["add", "dem.asc", "NULL", "out.asc", "NULL", f"{add_mm:g}", "1.0", "1.0", str(cpu_flag), "0", f"{THRES_MM}", str(iter_limit)]
    else:
        raise SystemExit("the reference arm times the Add module")
    env = dict(os.environ, OMP_NUM_THREADS=str(threads))
    t = time.perf_counter()
    res = subprocess.run([str(exe), *argv], cwd=workdir, capture_output=True, text=True, env=env)
    wall = time.perf_counter() - t
    if res.returncode != 0:
        raise RuntimeError(f"reference program failed ({res.returncode}): {res.stdout[-400:]} {res.stderr[-400:]}")
    rows = re.findall(r"^\s+(\d+)\s+([0-9.]+)\s+([0-9.]+)\s*$", res.stdout, flags=re.M)
    if not rows:
        raise RuntimeError("no block line in the reference program's output: " + res.stdout[-400:])
    return int(rows[-1][0]), float(rows[-1][2]), wall


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if rank != 0:
        return
    import tempfile
    from oracle import pyoracle as po
    from wdpm_b200 import ascgrid, synth
    threads = use_all_host_threads()
    size = min(args.sample_size, args.size)
    dem = synth.fractal_dem(size, size, seed=args.size, device="cpu").numpy()
    cells = size * size
    if po.ref_binary() is not None and args.module == "add":
        work = Path(tempfile.mkdtemp(prefix="wdpm_ref_"))
        write_sample_asc(work / "dem.asc", dem)
        for _ in range(args.warmup):
            run_reference_binary(work, args.module, args.add_mm, 1, threads)
        secs, iters = 0.0, 0
        for _ in range(args.steps):
            it, rt, _ = run_reference_binary(work, args.module, args.add_mm, 1, threads)
            secs += rt
            iters += it
        value = cells * iters / secs
        kind = "reference"
        sample = (f"{size}x{size} window of the synthetic DEM (seed {args.size}) as an .asc file, Add {args.add_mm:g} mm from the dry start; one step = one run of the "
                  f"UNMODIFIED reference program (oracle/_ref/WDPMCL_ref, cpu=1: its OpenCL branch on the OpenMP stand-in runtime, {threads} threads) "
                  f"with iter_limit {iters // args.steps}; timed by the program's own 'run time' column")
        ms_per_step = secs / args.steps * 1e3
        import shutil
        shutil.rmtree(work, ignore_errors=True)
    else:  # the reference-derived binaries are absent: verbatim kernel library if there, else this repo's port
        D = ascgrid.pad_grid(dem, NODATA)
        W = np.where(D > NODATA, args.add_mm / 1000.0, 0.0)
        Runner = cpu_kernel()
        r = Runner(W, D)
        iters = args.ref_iters_per_step
        for _ in range(args.warmup):
            r.iterate(iters)
        t = time.perf_counter()
        for _ in range(args.steps):
            r.iterate(iters)
        dt = time.perf_counter() - t
        value = cells * iters * args.steps / dt
        kind = Runner.kind
        sample = f"{size}x{size} window of the synthetic DEM (seed {args.size}), Add {args.add_mm:g} mm from the dry start, {iters} iterations per step, {threads} threads"
        ms_per_step = dt / args.steps * 1e3
    line = {
        "impl": "reference", "metric": "cell_updates_per_s", "value": value, "unit": "cell-updates/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": workload_config(args, world),
        "sample": sample,
        "cpu_baseline": {"value": value, "unit": "cell-updates/s", "cores": threads, "kind": kind, "sample": sample},
        "e2e": {"value": value, "unit": "cell-updates/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


# --------------------------------------------------------------------------- our arm


def workload_config(args, world):
    what = (f"Add {args.add_mm:g} mm, rof 1.0" if args.module == "add" else
            f"{args.module.capitalize()} on a uniform {args.add_mm:g} mm water layer" + (" (Subtract 0 mm: redistribution only)" if args.module == "subtract" else ", outlet = lowest cell"))
    return {"workload": f"synthetic {args.size}x{args.size} fractal DEM (H=0.7, sigma 3.34 m), {what}, "
                        f"zero-threshold {THRES_MM} mm, one step = one {BLOCK_ITERS}-iteration convergence block",
            "rows": args.size, "cols": args.size, "block_iters": args.block_iters,
            "partition": "single GPU" if world == 1 else f"{world} row stripes, halo exchange over NVLink",
            "l2_policy": "inputs larger than L2 (3 grids x rows x cols x 8 B per iteration)"}


def run_ours(args):
    import torch
    import torch.distributed as dist

    from wdpm_b200 import ADD, F32, F64, KERNEL_AUTO, Solver, ascgrid, synth
    from wdpm_b200.stripes import DistributedSolver
    module = MODULES[args.module]

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world == 1 and args.gpus > 1:
        raise SystemExit("launch N>1 with torch.distributed.run (one process per GPU)")
    if world > 1 and module != ADD:
        raise SystemExit("--module subtract|drain is a single-GPU bench line (scripts/large_drain.py drives Drain on several GPUs)")
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product has no CPU path")
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    def max_over_ranks(x: float) -> float:
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    dtype_code, np_dt, torch_dt, esize = (F64, np.float64, torch.float64, 8) if args.dtype == "f64" else (F32, np.float32, torch.float32, 4)
    size = args.size
    cells = size * size
    dem_dev = synth.fractal_dem(size, size, seed=size, device=f"cuda:{local_rank}", dtype=torch.float64)
    if args.dtype == "f32":
        dem_dev = dem_dev - dem_dev.min()  # fp32 mode: base elevation removed before rounding (DESIGN.md)

    common = dict(dtype=dtype_code, zero_threshold=THRES_MM / 1000, kernel=KERNEL_AUTO, fused_variant=args.variant)
    if world == 1:
        s = Solver(size, size, NODATA, module, device=local_rank, iters_per_launch=args.iters_per_launch, **common)
        r0, nrows, o0, orows = 0, size, 0, size
    else:
        ds = DistributedSolver(size, size, NODATA, ADD, device=local_rank, **common)
        s = ds.solver
        st = ds.stripe
        r0, nrows, o0, orows = st.band_row0, st.band_rows, st.owned_row0, st.owned_rows
    # this rank's rows (owned + halos) in pinned host memory: what a host application would hand over
    dem_host = torch.empty((nrows, size), dtype=torch_dt, pin_memory=True)
    dem_host.copy_(dem_dev[r0:r0 + nrows].to(torch_dt))
    del dem_dev
    torch.cuda.empty_cache()
    water_host = torch.zeros((nrows, size), dtype=torch_dt, pin_memory=True)
    owned_host = water_host[o0 - r0:o0 - r0 + orows]  # contiguous view: the owned rows inside the band

    def upload(with_water: bool):
        if world == 1:
            s.upload_ptr(dem_host.data_ptr(), water_host.data_ptr() if with_water else None)
        else:
            ds.upload_band_ptr(dem_host.data_ptr(), water_host.data_ptr() if with_water else None)

    def run_block():
        return s.run_block(args.block_iters) if world == 1 else ds.run_block(args.block_iters)

    stream = torch.cuda.Stream()
    s.set_stream(stream.cuda_stream)
    if module == ADD:
        upload(False)
        s.apply_add(args.add_mm / 1000.0, 1.0)
    else:  # Subtract / Drain start from a uniform layer (every cell wet: the full chain everywhere, like Add's first blocks)
        water_host.fill_(args.add_mm / 1000.0)
        upload(True)
        if module == 2:
            s.find_outlet()
            s.set_total_drain(0.0)

    for _ in range(args.warmup):
        run_block()

    # state the timed steps start from, for the CPU baseline sample (N=1, rank 0)
    do_cpu = args.cpu_baseline and rank == 0 and world == 1
    if do_cpu:
        s.download_water_ptr(water_host.data_ptr())
        n = min(args.sample_size, size)
        c0 = (size - n) // 2
        Dw = ascgrid.pad_grid(dem_host.numpy()[c0:c0 + n, c0:c0 + n].astype(np.float64), NODATA)
        Ww = ascgrid.pad_grid(water_host.numpy()[c0:c0 + n, c0:c0 + n].astype(np.float64), 0.0)
        wet = float(np.count_nonzero(Ww > 0)) / (n * n)

    # ---- timed region: K steps, device time on the solver's stream, max over ranks
    sampler = ClockSampler(physical_gpu_index(local_rank)).start()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    iter_ms, klaunch, last = [], 0, None
    barrier()
    ev0.record(stream)
    for _ in range(args.steps):
        r = run_block()
        iter_ms.append(r.iterate_ms)
        klaunch += r.launches
        last = r
    ev1.record(stream)
    barrier()
    clocks = sampler.stop()
    total_ms = max_over_ranks(ev0.elapsed_time(ev1))
    value = cells * args.block_iters * args.steps / (total_ms / 1e3)
    # order-free checksum of the assembled water grid after the timed steps: equal at every N iff the grids are
    checksum = s.water_checksum()
    if world > 1:
        parts = [None] * world
        dist.all_gather_object(parts, checksum)
        checksum = sum(parts) % (1 << 64)

    # ---- end to end: host buffers in, host buffers out, every step (max over ranks, wall clock
    # bracketed by barriers since the host<->device copies are synchronous calls)
    if world == 1:
        s.download_water_ptr(water_host.data_ptr())
    else:
        # refresh the whole band (halos too) so the re-upload resumes the same state
        s.download_water_ptr(owned_host.data_ptr())
        parts = [None] * world
        dist.all_gather_object(parts, (o0, owned_host.numpy()[[0, 1, 2, 3, 4, 5, -3, -2, -1]].copy()))
        if rank > 0:
            water_host[0:o0 - r0] = torch.from_numpy(parts[rank - 1][1][-(o0 - r0):])
        if rank + 1 < world:
            nb = nrows - (o0 - r0) - orows
            water_host[o0 - r0 + orows:] = torch.from_numpy(parts[rank + 1][1][:nb])
    if args.dump_outputs:  # the owned rows hold the state after the last timed step; stripes send their sampled cells to rank 0
        water = sampled_rows(sample_cells(size, size), size, o0, owned_host.numpy())
        if world > 1:
            parts = [None] * world
            dist.all_gather_object(parts, (o0, water))
            water = np.concatenate([p[1] for p in sorted(parts, key=lambda p: p[0])])
        if rank == 0:
            dump_outputs(args.dump_outputs, size, size, water, last)
    e2e_steps = max(1, min(args.steps, args.e2e_steps))
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        upload(True)
        if module == 2:
            s.set_total_drain(0.0)
        r2 = run_block()
        s.download_water_ptr(owned_host.data_ptr() if world > 1 else water_host.data_ptr())
        klaunch += r2.launches
        if world > 1 and e2e_steps > 1:
            parts = [None] * world
            dist.all_gather_object(parts, owned_host.numpy()[[0, 1, 2, 3, 4, 5, -3, -2, -1]].copy())
            if rank > 0:
                water_host[0:o0 - r0] = torch.from_numpy(parts[rank - 1][-(o0 - r0):])
            if rank + 1 < world:
                nb = nrows - (o0 - r0) - orows
                water_host[o0 - r0 + orows:] = torch.from_numpy(parts[rank + 1][:nb])
    barrier()
    t_e2e = max_over_ranks(time.perf_counter() - t0)
    e2e_value = cells * args.block_iters * e2e_steps / t_e2e

    info2 = s.info()
    K = info2["iters_per_launch"]
    iter_launches = args.block_iters // K
    my_cells = orows * size
    peak, peak_src = measured_peak_gbs()
    launch_ms = float(np.mean(iter_ms)) / iter_launches
    achieved = my_cells * 3 * esize * K / (launch_ms / 1e3) / 1e9
    kernel_name = {1: "k_colour", 2: "k_fused_wa" if info2.get("warp_autonomous") else "k_fused", 3: "k_resident"}[info2["kernel"]]
    traffic = None
    try:  # DRAM bytes per launch from the committed ncu capture of this very configuration, if there is one
        tj = json.loads((ROOT / "profiles" / "ncu_traffic.json").read_text())
        traffic = tj[f"{kernel_name}:{args.module}:{args.dtype}:{size}x{size}:{world}gpu"]["traffic_bytes"]
    except Exception:
        traffic = None
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": traffic, "kernel": kernel_name, "launch_ms": launch_ms,
                "algorithmic_bytes_per_launch": my_cells * 3 * esize * K, "peak_source": peak_src, "per": "GPU (slowest rank's launch time)"}

    line = {
        "metric": "cell_updates_per_s", "value": value, "unit": "cell-updates/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": total_ms / args.steps, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": args.dtype, "data": "synthetic", "config": workload_config(args, world),
        "e2e": {"value": e2e_value, "unit": "cell-updates/s", "h2d_bytes_per_step": 2 * nrows * size * esize * world if world > 1 else 2 * cells * esize,
                "d2h_bytes_per_step": cells * esize + 64 * world, "steps": e2e_steps},
        "gpu_launches": int(klaunch), "clocks": clocks, "roofline": roofline,
        "state": {"max_diff": last.max_diff, "wet_fraction": last.wet_cells / cells, "checksum": f"{checksum:016x}",
                  "checksum_after_iterations": (args.warmup + args.steps) * args.block_iters,
                  "iterations_done": (args.warmup + args.steps + e2e_steps) * args.block_iters},
        "tiling": {k: info2[k] for k in ("kernel", "strip_cols", "window_cols", "chunk_rows", "grid_ctas", "cta_threads", "smem_bytes", "iters_per_launch", "sm_count", "warp_autonomous")},
    }
    if do_cpu:
        v, kind, threads, n_it, dt = time_cpu_sample(Dw, Ww, args.cpu_budget)
        line["cpu_baseline"] = {"value": v, "unit": "cell-updates/s", "cores": threads, "kind": kind,
                                "sample": f"{Dw.shape[0]-2}x{Dw.shape[1]-2} centre window of the same DEM in the state after warm-up "
                                          f"(wet fraction {wet:.3f}), {n_it} iterations in {dt:.1f} s"}
        from oracle import pyoracle as po
        if args.serial_baseline and module == ADD and po.ref_binary() is None:
            warn_no_reference("no cpu_baseline_serial (it runs the unmodified reference program)")
        if args.serial_baseline and module == ADD and po.ref_binary() is not None:
            import shutil
            import tempfile
            n = min(args.serial_sample_size, size)
            c0 = (size - n) // 2
            work = Path(tempfile.mkdtemp(prefix="wdpm_serial_"))
            write_sample_asc(work / "dem.asc", dem_host.numpy()[c0:c0 + n, c0:c0 + n].astype(np.float64))
            it, rt, wall = run_reference_binary(work, "add", args.add_mm, 0, 1)
            shutil.rmtree(work, ignore_errors=True)
            line["cpu_baseline_serial"] = {"value": n * n * it / rt, "unit": "cell-updates/s", "cores": 1, "kind": "reference",
                                           "sample": f"unmodified reference program (oracle/_ref/WDPMCL_ref, cpu=0: serial backend), Add {args.add_mm:g} mm on the "
                                                     f"{n}x{n} centre window of the same DEM as an .asc file, iter_limit {it}: {rt:.2f} s by its own 'run time' column"}
        # the reference arm's sample (bench.py --impl reference) through the CUDA path, for a like-for-like ratio
        n = min(args.sample_size_ref, size)
        demw = np.ascontiguousarray(synth.fractal_dem(n, n, seed=size, device="cpu").numpy().astype(np_dt))
        with Solver(n, n, NODATA, ADD, device=local_rank, dtype=dtype_code, zero_threshold=THRES_MM / 1000, kernel=KERNEL_AUTO) as s2:
            s2.upload(demw, None)
            s2.apply_add(args.add_mm / 1000.0, 1.0)
            s2.run_block(args.block_iters)
            s2.upload(demw, None)
            s2.apply_add(args.add_mm / 1000.0, 1.0)
            rr = s2.run_block(args.block_iters)
            line["gpu_on_reference_sample"] = {"value": n * n * args.block_iters / (rr.block_ms / 1e3), "unit": "cell-updates/s",
                                               "sample": f"{n}x{n} window, Add {args.add_mm:g} mm from the dry start, one {args.block_iters}-iteration block (device time), "
                                                         f"kernel {s2.info()['kernel']}"}
    if world == 1:
        s.close()
    else:
        ds.close()
        dist.destroy_process_group()
    if rank == 0:
        print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--size", type=int, default=32768)
    ap.add_argument("--dtype", default="f64", choices=["f64", "f32"])
    ap.add_argument("--block-iters", type=int, default=BLOCK_ITERS)
    ap.add_argument("--iters-per-launch", type=int, default=0)
    ap.add_argument("--variant", type=int, default=0)
    ap.add_argument("--e2e-steps", type=int, default=5)
    ap.add_argument("--module", default="add", choices=["add", "subtract", "drain"])
    ap.add_argument("--add-mm", type=float, default=300.0, help="water depth of the workload (BASELINE configs[2]: 100)")
    ap.add_argument("--no-serial-baseline", dest="serial_baseline", action="store_false")
    ap.add_argument("--serial-sample-size", type=int, default=512)
    ap.add_argument("--sample-size-ref", type=int, default=1024, help="window of the reference arm (unmodified program)")
    ap.add_argument("--no-cpu-baseline", dest="cpu_baseline", action="store_false")
    ap.add_argument("--cpu-budget", type=float, default=12.0)
    ap.add_argument("--sample-size", type=int, default=2048)
    ap.add_argument("--ref-iters-per-step", type=int, default=100)
    ap.add_argument("--dump-outputs", metavar="DIR", type=Path, default=None,
                    help="write the water grid (a fixed sample above 4 Mi cells) and reductions of the last timed step as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes what the CUDA path computed; the reference arm has no such output")
    if args.impl == "reference":
        args.sample_size = args.sample_size_ref
        run_reference_arm(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
