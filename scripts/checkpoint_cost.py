#!/usr/bin/env python
"""What an exact checkpoint capture (wdpm_checkpoint_arm / wdpm_checkpoint_wait) costs, one GPU, fp64 Add.

For each size: the fractal DEM of bench.py, every cell wet (wdpm_apply_add of 300 mm on a dry grid), zero
threshold 0.005 mm. After a warm-up block, blocks with a capture and blocks without alternate; each block's device
time is the library's own CUDA-event time on the solver's stream (wdpm_block_result.block_ms), so a capture that
slows the iteration kernels shows up there. Reported beside it:
  - capture_landed_ms: for each captured block, host time from wdpm_block_begin until wdpm_checkpoint_wait
    returns, the whole block's iterations having been enqueued in between. The wait ends on the capture's
    completion event, so this is the capture itself under a running block: the prologue, the totals' gather and
    the side stream's pitched copy of the grid into pinned memory (wdpm_checkpoint_wait called through ctypes, so
    no copy into numpy is timed);
  - writer_gb_per_s: the host writer's system calls (pwrite, fsync, rename) from Python on the first GiB of the
    captured grid (or all of it, if smaller), to a file in the system's temporary directory; best of three.

Prints one JSON object; the card's name and power limit (read-only nvidia-smi query) are part of it.

    python scripts/checkpoint_cost.py [--sizes 8192 32768] [--pairs 8] [--block-iters 100 200] [--out FILE]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))

from wdpm_b200 import ADD, F64, Solver, synth  # noqa: E402

NODATA = -99999.0


def card() -> dict:
    res = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                         capture_output=True, text=True)
    name, power = (x.strip() for x in res.stdout.strip().split("\n")[0].split(",", 1))
    return {"gpu": name, "power_limit": power}


def captured_block(s: Solver, block_iters: int) -> tuple[float, float]:
    """(block device ms, ms from the block's begin until its capture has landed)"""
    s.checkpoint_arm()
    t = time.perf_counter()
    s.block_begin()
    s.block_enqueue(block_iters)
    rc = s._lib.wdpm_checkpoint_wait(s._h, None, None, None)
    landed = 1000 * (time.perf_counter() - t)
    assert rc == 0
    return s.block_end().block_ms, landed


def writer_gb_per_s(grid: np.ndarray, reps: int = 3) -> float:
    best = 0.0
    with tempfile.TemporaryDirectory() as tmp:
        path = os.path.join(tmp, "ck.bin")
        for _ in range(reps):
            t = time.perf_counter()
            fd = os.open(path + ".tmp", os.O_WRONLY | os.O_CREAT | os.O_TRUNC, 0o644)
            view, off = memoryview(np.ascontiguousarray(grid).view(np.uint8)), 0
            while off < len(view):
                off += os.pwrite(fd, view[off:off + (1 << 30)], off)
            os.fsync(fd)
            os.close(fd)
            os.rename(path + ".tmp", path)
            best = max(best, grid.nbytes / (time.perf_counter() - t) / 1e9)
    return best


def measure(n: int, pairs: int, block_iters: int) -> dict:
    import torch  # the DEM is generated on the GPU
    dem = synth.fractal_dem(n, n, seed=n, device="cuda:0", dtype=torch.float64).cpu().numpy()
    out = {"block_iters": block_iters, "grid_bytes": n * n * 8}
    with Solver(n, n, NODATA, ADD, dtype=F64, zero_threshold=0.005 / 1000) as s:
        s.upload(dem, None)
        del dem
        s.apply_add(0.3, 1.0)
        s.run_block(block_iters)  # warm-up
        s.checkpoint_arm()  # the first arm allocates the staging
        s.run_block(block_iters)
        s.checkpoint_wait()
        plain, captured, landed = [], [], []
        for _ in range(pairs):
            ms, ms_landed = captured_block(s, block_iters)
            captured.append(ms)
            landed.append(ms_landed)
            plain.append(s.run_block(block_iters).block_ms)
        out["block_ms_plain"] = [round(x, 3) for x in plain]
        out["block_ms_captured"] = [round(x, 3) for x in captured]
        out["capture_overhead_pct"] = round(100 * (np.median(captured) / np.median(plain) - 1), 2)
        out["capture_landed_ms"] = [round(x, 3) for x in landed]
        out["capture_gb_per_s"] = round(n * n * 8 / np.median(landed) / 1e6, 2)
        water, _ = s.checkpoint_wait()
    out["writer_gb_per_s"] = round(writer_gb_per_s(water.reshape(-1)[: 1 << 27]), 2)  # the first GiB of the capture
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", type=int, nargs="+", default=[8192, 32768])
    ap.add_argument("--block-iters", type=int, nargs="+", default=[100, 200])
    ap.add_argument("--pairs", type=int, default=8)
    ap.add_argument("--out", type=Path)
    args = ap.parse_args()
    result = {"card": card()}
    for n, it in zip(args.sizes, args.block_iters):
        result[f"add_{n}_f64"] = measure(n, args.pairs, it)
    text = json.dumps(result, indent=1)
    print(text)
    if args.out:
        args.out.parent.mkdir(parents=True, exist_ok=True)
        args.out.write_text(text + "\n")


if __name__ == "__main__":
    main()
