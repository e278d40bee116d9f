"""Cost of a Drain outlet set: 8192^2 fp64 Drain, every cell wet, the warp-autonomous fused kernel (k_fused_wa),
with 1 outlet, 64 outlets, the rim (32 764) and 2^20 outlets. Per case: ms per iteration, the block-end time (the
reductions and the outlet-order sum of the totals), and the solver's device bytes.

    python scripts/outlet_sets.py [--size 8192] [--iters 500] [--out profiles/outlet_sets_b200.json]
"""
import argparse
import json
import subprocess
import sys
from pathlib import Path

import numpy as np

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
from wdpm_b200 import F64, MAX_OUTLETS, Solver, ascgrid, synth  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--size", type=int, default=8192)
ap.add_argument("--iters", type=int, default=500)
ap.add_argument("--out", default="profiles/outlet_sets_b200.json")
a = ap.parse_args()
n = a.size
d = synth.fractal_dem(n, n, seed=1, device="cuda").cpu().numpy()
w = np.full((n, n), 0.05)
rng = np.random.default_rng(3)
rim = ascgrid.rim_outlets(d, -99999.0)
inner = rng.choice(n * n, MAX_OUTLETS, replace=False)
full = sorted(set(rim) | {(int(k // n) + 1, int(k % n) + 1) for k in inner})[:MAX_OUTLETS]
cases = {"1": None, "64": [(int(k // n) + 1, int(k % n) + 1) for k in inner[:64]], "rim": rim, "2^20": full}
smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
rows = []
for name, outlets in cases.items():
    s = Solver(n, n, -99999.0, 2, dtype=F64, fused_variant=17)
    s.upload(d, w)
    if outlets is None:
        s.find_outlet()
        outlets = [None]
    else:
        s.set_outlets(outlets)
    s.seed_outlet_drains()
    s.run_block(50)  # warm-up
    r = s.run_block(a.iters)
    rows.append({"case": name, "n_outlets": len(outlets), "ms_per_iter": r.iterate_ms / a.iters,
                 "block_end_ms": r.block_ms - r.iterate_ms, "block_ms": r.block_ms, "iters": a.iters,
                 "device_bytes": s.info()["device_bytes"], "total_drain": r.total_drain})
    print(rows[-1], flush=True)
    s.close()
res = {"gpu": smi, "size": n, "dtype": "f64", "kernel": "k_fused_wa (variant 17)", "water": "0.05 m on every cell", "cases": rows}
Path(a.out).parent.mkdir(parents=True, exist_ok=True)
Path(a.out).write_text(json.dumps(res, indent=1) + "\n")
