"""Measurement aid: shear maps (slicer_shear, SLICER_b200 --shear).
usage: python tools/shear_e2e.py [--sizes 2048,8192] [--reps 20] [--ng 512] [--numfiles 16] [--k 8] [--zs 1.0,0.75,0.5,0.25] [--runs 3]
                                 [--gpus 0] [--work /tmp/e2e_real] [--out FILE] [--no-driver]
1. Device time of one slicer_shear (CUDA events through slicer_timer_*), median of --reps after warm-up, for npix in --sizes at the
   driver's FFT size (the smallest power of two >= 2 npix), with the bytes its passes move (pass_bytes below) and the resulting
   rate.  Both sizes' working sets (2 x 16 B x P^2) exceed the 126 MB L2.
2. The C3-shaped run of tools/kappa_e2e.py (K inis, S source redshifts, --no-planes) without and with --shear, the modes
   alternating, --runs times: medians of total - set-up and of the shear phase of SLICER_B200_TIMING, and one JSON line per run.
The GPU's name, power limit and SM clock are read in the same process and printed with the numbers."""
import argparse
import json
import math
import os
import re
import shutil
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from slicer_b200 import capi, host, synth  # noqa: E402
from test_gpu_driver import INI  # noqa: E402

S_ = dict(box=256000.0, npix=2048, fov=5.0, zs=1.0, nsnap=12)  # "c3" of tools/realisations_e2e.py
ap = argparse.ArgumentParser()
ap.add_argument("--sizes", default="2048,8192")
ap.add_argument("--reps", type=int, default=20)
ap.add_argument("--ng", type=int, default=512)
ap.add_argument("--numfiles", type=int, default=16)
ap.add_argument("--k", type=int, default=8)
ap.add_argument("--zs", default="1.0,0.75,0.5,0.25")
ap.add_argument("--runs", type=int, default=3, help="runs of each mode, the modes alternating")
ap.add_argument("--gpus", default="0")
ap.add_argument("--work", default="/tmp/e2e_real")
ap.add_argument("--out", default=None, help="also append the JSON lines to this file")
ap.add_argument("--no-driver", action="store_true", help="part 1 only")
a = ap.parse_args()


def emit(d):
    line = json.dumps(d)
    print(line, flush=True)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "a") as f:
            f.write(line + "\n")


def pass_bytes(npix, P):
    """HBM bytes the launches of one slicer_shear read and write (16 B per complex element, 8 B per κ or γ value; the twiddle
    table, P x 16 B, is left out).  Two radix stages per launch: ceil(stages / 2) launches per axis."""
    stages, n = 0, 1
    while n < P:
        n *= 4 if P // n >= 4 else 2
        stages += 1
    L = (stages + 1) // 2
    rows, full = npix * P, P * P
    fwd_rows = (8 * npix * npix + 16 * rows) + (L - 1) * 32 * rows  # the first launch reads κ
    fwd_cols = (16 * rows + 16 * full) + (L - 1) * 32 * full  # the first launch reads the npix rows the row passes wrote
    inv_cols = L * 32 * full
    inv_rows = (L - 1) * 32 * rows + (16 * rows + 16 * npix * npix)  # the last launch writes γ1, γ2 of the window
    return fwd_rows + fwd_cols + inv_cols + inv_rows, 4 * L


gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm,clocks.sm", "--format=csv,noheader"], capture_output=True,
                     text=True).stdout.strip().splitlines()
emit(dict(gpu=gpu))

# ---- 1. device time of slicer_shear ---------------------------------------------------------------------------------------------
for npix in [int(v) for v in a.sizes.split(",")]:
    P = 1 << math.ceil(math.log2(2 * npix))
    k = np.random.default_rng(1).standard_normal((npix, npix)) * 0.01
    with capi.Slicer(npix_max=npix, max_planes=1) as s:
        s.kappa_maps(1, npix)
        s.kappa_load(0, k)
        for _ in range(3):
            s.shear(0, P)
        s.synchronize()
        times = []
        for _ in range(a.reps):
            s.timer_begin()
            s.shear(0, P)
            times.append(s.timer_end())
        s.shear_fetch()
    times.sort()
    ms = times[len(times) // 2]
    nbytes, launches = pass_bytes(npix, P)
    emit(dict(kernel="shear_fft_pass", npix=npix, fft=P, launches=launches, median_ms=round(ms, 4), min_ms=round(times[0], 4), bytes=nbytes,
              GBs=round(nbytes / ms / 1e6, 1), share_of_datasheet_7700GBs=round(nbytes / ms / 1e6 / 7700, 3), gpu=gpu))

if a.no_driver:
    sys.exit(0)

# ---- 2. the C3-shaped run with and without --shear -------------------------------------------------------------------------------
os.makedirs(a.work + "/snaps", exist_ok=True)
names = []
for i in range(S_["nsnap"]):
    base = f"{a.work}/snaps/snap_{i:03d}"
    if not os.path.exists(base + ".0"):
        synth.write_snapshot(base, {1: synth.hash_positions(a.ng ** 3, S_["box"], 1000 + i)}, [0, 1.0375, 0, 0, 0, 0], 0.1 * i, S_["box"],
                             numfiles=a.numfiles, with_vel_id=False)
    names.append(f"snap_{i:03d}")
open(a.work + "/snapshot_list.txt", "w").write("\n".join(names))


def ini(tag, k):
    out = f"{a.work}/{tag}"
    os.makedirs(out, exist_ok=True)
    t = INI.format(npix=S_["npix"], zs=S_["zs"], fov=S_["fov"], list=a.work + "/snapshot_list.txt", snapdir=a.work + "/snaps/", outdir=out + "/lc_",
                   pip=0, snopt=0)
    for old, new in zip((-229, -230, -231), (-229 - 17 * k, -230 + 5 * k, -231 - 3 * k)):
        t = t.replace(f"\n{old}\n", f"\n{new}\n")
    t = t.replace("PLC Suffix ###########\n0\n", f"PLC Suffix ###########\nr{k}\n")
    path = f"{a.work}/{tag}_{k}.ini"
    open(path, "w").write(t)
    return path


def phase(line, pat):
    m = re.search(pat + r" ([0-9.e+-]+)", line)
    return float(m.group(1)) if m else None


MODES = (("kappa", ["--kappa-zs", a.zs, "--no-planes"]), ("kappa+shear", ["--kappa-zs", a.zs, "--no-planes", "--shear"]))
res = {m: [] for m, _ in MODES}
for run_i, (mode, extra) in [(i, m) for i in range(a.runs) for m in MODES]:
    shutil.rmtree(f"{a.work}/shear_out", ignore_errors=True)
    inis = [ini("shear_out", k) for k in range(a.k)]
    t0 = time.time()
    r = subprocess.run([host.EXE_PATH, "--quiet", "--gpus", a.gpus, *extra, *inis], cwd=a.work, capture_output=True, text=True,
                       env=dict(os.environ, SLICER_B200_TIMING="1"))
    wall = time.time() - t0
    assert r.returncode == 0, r.stderr[-2000:]
    line = next(l for l in r.stderr.splitlines() if l.startswith("[timing] total"))
    files = os.listdir(f"{a.work}/shear_out")
    d = dict(mode=mode, run=run_i, K=a.k, S=len(a.zs.split(",")), ng=a.ng, npix=S_["npix"], wall_s=round(wall, 2), total_s=phase(line, "total"),
             setup_s=phase(line, "engine/CUDA set-up"), kappa_s=phase(line, "convergence maps"), shear_s=phase(line, "shear maps"),
             kappa_files=sum(".kappa_" in f for f in files), gamma_files=sum(".gamma" in f for f in files))
    res[mode].append(d)
    emit(d)
shutil.rmtree(f"{a.work}/shear_out", ignore_errors=True)
for mode, runs in res.items():
    emit(dict(mode=mode, median_total_minus_setup_s=round(float(np.median([r["total_s"] - r["setup_s"] for r in runs])), 3),
              median_shear_s=(round(float(np.median([r["shear_s"] for r in runs])), 3) if runs[0]["shear_s"] is not None else None), gpu=gpu))
