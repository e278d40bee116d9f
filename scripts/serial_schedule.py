#!/usr/bin/env python
"""What the serial schedule (WDPM_SCHEDULE_SERIAL, the reference's `cpu=0`) costs against the OpenCL schedule, one GPU.

1. basin5 (the reference's sample DEM), the validate_WDPM.sh sequence Add 10 mm -> Drain -> Subtract 10 mm, each
   module run to its stop test through wdpm_b200.wdpmcl with the water handed on through "%f" files: device time
   (sum of the blocks' CUDA-event time) and iterations per module under both schedules.
2. 8192 x 8192 fp64, the fractal DEM of bench.py, every cell wet under a uniform 300 mm layer (as `bench.py
   --module` sets Subtract and Drain up), zero threshold 0.005 mm: ms per iteration of Subtract and Drain under
   both schedules - one warm-up block, then timed blocks - and wdpm_water_checksum of the grid afterwards.

Prints one JSON object; the card's name and power limit (read-only nvidia-smi query) are part of it.

    python scripts/serial_schedule.py [--size 8192] [--blocks 3] [--block-iters 200] [--out FILE]
"""
from __future__ import annotations

import argparse
import json
import subprocess
import sys
import tempfile
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))

from wdpm_b200 import DRAIN, F64, KERNEL_AUTO, SCHED_OPENCL, SCHED_SERIAL, SUBTRACT, Solver, ascgrid, synth, wdpmcl  # noqa: E402

NODATA = -99999.0
THRES_MM = 0.005
SCHEDS = {"opencl": SCHED_OPENCL, "serial": SCHED_SERIAL}


def card() -> dict:
    res = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                         capture_output=True, text=True)
    name, power = (x.strip() for x in res.stdout.strip().split("\n")[0].split(",", 1))
    return {"gpu": name, "power_limit": power}


def basin5_sequence(sched: int, work: Path) -> dict:
    hdr, dem = ascgrid.read_asc(ROOT / "tests" / "golden" / "basin5.asc.gz")
    backend = wdpmcl.default_backend(schedule=sched)
    steps = [("add10", wdpmcl.ModuleParams("add", depth_mm=10, runoff_fraction=1.0, elevation_tol_mm=1.0, zero_threshold_mm=THRES_MM)),
             ("drain", wdpmcl.ModuleParams("drain", elevation_tol_mm=0.1, drain_tol_m3=1.0, zero_threshold_mm=THRES_MM)),
             ("sub10", wdpmcl.ModuleParams("subtract", depth_mm=10, elevation_tol_mm=1.0, zero_threshold_mm=THRES_MM))]
    water, out = None, {}
    for name, params in steps:
        rep = wdpmcl.run_module(dem, hdr.nodata, hdr.cellsize, params, water=water, backend=backend)
        path = work / f"{name}.asc"
        ascgrid.write_asc(path, hdr, rep.water)
        water = ascgrid.read_asc(path)[1]
        out[name] = {"device_ms": round(rep.solver_ms, 3), "iterations": rep.iterations,
                     "us_per_iteration": round(1000.0 * rep.solver_ms / rep.iterations, 3)}
    return out


def large(module: int, sched: int, dem: np.ndarray, blocks: int, block_iters: int) -> dict:
    size = dem.shape[0]
    with Solver(size, size, NODATA, module, dtype=F64, zero_threshold=THRES_MM / 1000, kernel=KERNEL_AUTO, schedule=sched) as s:
        s.upload(dem, np.full_like(dem, 0.3))
        if module == DRAIN:
            s.find_outlet()
            s.set_total_drain(0.0)
        s.run_block(block_iters)  # warm-up
        ms = [s.run_block(block_iters).iterate_ms for _ in range(blocks)]
        info = s.info()
        return {"ms_per_iteration": round(sum(ms) / (blocks * block_iters), 5), "kernel": info["kernel"],
                "warp_autonomous": info["warp_autonomous"],
                "total_drain": s.get_total_drain() if module == DRAIN else None, "water_checksum": f"{s.water_checksum():016x}"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--size", type=int, default=8192)
    ap.add_argument("--blocks", type=int, default=3)
    ap.add_argument("--block-iters", type=int, default=200)
    ap.add_argument("--out", type=Path)
    args = ap.parse_args()
    result = {"card": card(), "basin5_sequence": {}, f"grid_{args.size}_f64": {}}
    with tempfile.TemporaryDirectory() as tmp:
        for k, sched in SCHEDS.items():
            result["basin5_sequence"][k] = basin5_sequence(sched, Path(tmp))
    import torch
    dem = synth.fractal_dem(args.size, args.size, seed=args.size, device="cuda:0", dtype=torch.float64).cpu().numpy()
    for mname, module in (("subtract", SUBTRACT), ("drain", DRAIN)):
        for k, sched in SCHEDS.items():
            r = large(module, sched, dem, args.blocks, args.block_iters)
            result[f"grid_{args.size}_f64"][f"{mname}_{k}"] = r
    text = json.dumps(result, indent=1)
    print(text)
    if args.out:
        args.out.parent.mkdir(parents=True, exist_ok=True)
        args.out.write_text(text + "\n")


if __name__ == "__main__":
    main()
