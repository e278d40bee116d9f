#!/usr/bin/env python
"""Regenerate tests/golden/ from the UNMODIFIED reference (needs a checkout of
CentreForHydrology/WDPM at pyoracle.reference_dir(); the tests only read the fixtures).

What it runs (oracle/_ref/WDPMCL_ref = <reference>/src/WDPMCL.c compiled as is
and linked to the minicl stand-in runtime that executes the verbatim runoff.cl):

  validate_WDPM.sh's sequence on dem/basin5.asc, once per backend
      add 10 mm (rof 1.0, tol 1 mm, thr 0.005 mm) -> drain (0.1 mm, 1.0 m3) -> subtract 10 mm
      backend "serial" = cpu 0, backend "opencl" = cpu 1 gpu 0
  -> ref_<backend>_<step>.asc.gz (the output water file) and .txt (stdout)

  raw-precision vectors on a 96x90 window of basin5 from the verbatim kernel file
  (oracle/_ref/librunoffcl_ref.so), per module and precision
  -> crop_vectors.npz

  tests/test_oracle.py's live cases (edge shapes, NODATA holes, LIVE_ITERS iterations from
  totaldrain LIVE_TD0) through the verbatim kernel file, per module and precision: inputs,
  outputs and totaldrain -> live_vectors.npz   [--live-only: this file alone]

  BASELINE.json configs[0] (basin5 Add 300 mm, rof 1.0, tol 1 mm, thr 0.005 mm; 320 000
  iterations, ~6 min on 8 threads through the OpenCL branch; its output file is
  byte-identical to the serial backend's) -> ref_opencl_add300.asc.gz / .txt   [--cfg1]

Usage: [WDPM_REFERENCE=<checkout>] python tests/golden/make_golden.py [--reuse DIR] [--cfg1] [--live-only]
       (DIR/rt{0,1}/{add,drain,sub}.{asc,txt}, DIR/cfg1/add300.{asc,txt})
"""
import argparse
import gzip
import shutil
import subprocess
import sys
import tempfile
from pathlib import Path

import numpy as np

HERE = Path(__file__).resolve().parent
ROOT = HERE.parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(HERE.parent))

from oracle import pyoracle as po  # noqa: E402
from wdpm_b200 import ascgrid  # noqa: E402

REF = po.reference_dir()
if REF is None:
    raise SystemExit("no reference checkout: put it beside this repository as `reference` or set WDPM_REFERENCE (it must hold src/runoff.cl)")


def gz(src: Path, dst: Path):
    with open(src, "rb") as f, gzip.GzipFile(dst, "wb", mtime=0) as g:
        shutil.copyfileobj(f, g)


def run_sequence(outdir: Path, rt: int):
    exe = po.ref_binary()
    dem = REF / "dem" / "basin5.asc"
    outdir.mkdir(parents=True, exist_ok=True)
    steps = [
        ("add", ["add", dem, "NULL", outdir / "add.asc", "NULL", "10", "1.0", "1.0", rt, 0, "0.005", 0]),
        ("drain", ["drain", dem, outdir / "add.asc", outdir / "drain.asc", "NULL", "0.1", "1.0", rt, 0, "0.005", 0]),
        ("sub", ["subtract", dem, outdir / "drain.asc", outdir / "sub.asc", "NULL", "10", "1.0", rt, 0, "0.005", 0]),
    ]
    for name, argv in steps:
        # cwd = reference src/: WDPMCL.c fopen()s "runoff.cl" by relative path (WDPMCL.c:1,132)
        res = subprocess.run([str(exe)] + [str(a) for a in argv], cwd=REF / "src", capture_output=True, text=True, check=True)
        (outdir / f"{name}.txt").write_text(res.stdout)


def live_vectors():
    """test_oracle_matches_verbatim_kernel_live's cases through the verbatim kernels -> live_vectors.npz."""
    from test_oracle import LIVE_ITERS, LIVE_TD0, MODS, live_cases
    oracle, ref = po.Oracle(), po.RefCL()
    out = {}
    for dt, dn in ((np.float64, "f64"), (np.float32, "f32")):
        for k, (_, _, D, W, outlet) in enumerate(live_cases(oracle, dt)):
            out[f"{dn}_{k}_dem"], out[f"{dn}_{k}_w0"], out[f"{dn}_{k}_outlet"] = D, W, np.array(outlet, dtype=np.int32)
            for mn, mod in MODS:
                w = W.copy()
                td = ref.iterate(w, D, -99999.0, mod, LIVE_ITERS, outlet=outlet, totaldrain=LIVE_TD0)
                out[f"{mn}_{dn}_{k}_w"], out[f"{mn}_{dn}_{k}_td"] = w, np.array(td, dtype=dt)
    np.savez_compressed(HERE / "live_vectors.npz", **out)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reuse", type=Path)
    ap.add_argument("--cfg1", action="store_true")
    ap.add_argument("--live-only", action="store_true")
    args = ap.parse_args()
    po.build()
    live_vectors()
    if args.live_only:
        return
    gz(REF / "dem" / "basin5.asc", HERE / "basin5.asc.gz")
    work = args.reuse or Path(tempfile.mkdtemp())
    for rt, backend in ((0, "serial"), (1, "opencl")):
        d = work / f"rt{rt}"
        if not args.reuse:
            run_sequence(d, rt)
        for step, tag in (("add", "add10"), ("drain", "drain"), ("sub", "sub10")):
            gz(d / f"{step}.asc", HERE / f"ref_{backend}_{tag}.asc.gz")
            shutil.copyfile(d / f"{step}.txt", HERE / f"ref_{backend}_{tag}.txt")

    if args.cfg1:
        d = work / "cfg1"
        if not args.reuse:
            d.mkdir(parents=True, exist_ok=True)
            res = subprocess.run([str(po.ref_binary()), "add", str(REF / "dem" / "basin5.asc"), "NULL",
                                  str(d / "add300.asc"), "NULL", "300", "1.0", "1.0", "1", "0", "0.005", "0"],
                                 cwd=REF / "src", capture_output=True, text=True, check=True)
            (d / "add300.txt").write_text(res.stdout)
        gz(d / "add300.asc", HERE / "ref_opencl_add300.asc.gz")
        shutil.copyfile(d / "add300.txt", HERE / "ref_opencl_add300.txt")

    # usage texts and exit codes of the unmodified binary (WDPMCL.c:308-355)
    exe = str(po.ref_binary())
    for name, argv in (("usage_all", []), ("usage_add", ["add"]), ("usage_subtract", ["subtract"]), ("usage_drain", ["drain"]),
                       ("usage_badcount", ["add", "a", "b", "c"])):
        res = subprocess.run([exe] + argv, capture_output=True, text=True)
        (HERE / f"{name}.txt").write_text(f"exit={res.returncode}\n" + res.stdout)

    # raw-precision crop vectors from the verbatim kernels
    hdr, dem = ascgrid.read_asc(REF / "dem" / "basin5.asc")
    win = dem[180:276, 200:290].copy()  # mixed valid / NODATA window with relief
    ref = po.RefCL()
    out = {"dem": win, "nodata": np.float64(hdr.nodata), "iters": np.int32(150)}
    rng = np.random.default_rng(5)
    for dt, dn in ((np.float64, "f64"), (np.float32, "f32")):
        D = ascgrid.pad_grid(win.astype(dt), dt(hdr.nodata))
        W0 = np.where(D > hdr.nodata, rng.uniform(0.0, 0.08, D.shape), 0.0).astype(dt)
        W0[rng.uniform(size=D.shape) < 0.35] = 0
        out[f"w0_{dn}"] = W0
        outlet = po.Oracle().find_outlet(D)
        out["outlet"] = np.array(outlet, dtype=np.int32)
        for mod, mn in ((po.ADD, "add"), (po.SUBTRACT, "subtract"), (po.DRAIN, "drain")):
            w = W0.copy()
            td = ref.iterate(w, D, hdr.nodata, mod, 150, outlet=outlet, totaldrain=0.0)
            out[f"w_{mn}_{dn}"] = w
            out[f"td_{mn}_{dn}"] = np.array(td, dtype=dt)
    np.savez_compressed(HERE / "crop_vectors.npz", **out)
    print("golden fixtures written to", HERE)


if __name__ == "__main__":
    main()
