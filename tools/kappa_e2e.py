"""Measurement aid: convergence maps on the C3-shaped files of tools/realisations_e2e.py (K realisations, S source redshifts).
usage: python tools/kappa_e2e.py [--ng 512] [--numfiles 16] [--k 8] [--zs 1.0,0.75,0.5,0.25] [--gpus 0] [--work /tmp/e2e_real] [--out FILE]
1. One `SLICER_b200` run of K inis each for: planes only (no convergence maps), planes + maps (--kappa-zs), maps only
   (--no-planes), the modes alternating, --runs times: wall time and the driver's SLICER_B200_TIMING phases, one JSON line per run.
2. Device time of slicer_kappa_add over one light cone's planes at the shape's map size (CUDA events through slicer_timer_*),
   after warm-up, the planes in calls of up to 16 slots as the driver makes them; bytes by the kernel's traffic formula
   (8 B x npix^2 per plane read, 2 x 8 B x npix^2 per map per call) and their share of MEASURED_PEAKS.json:hbm_gbs when that
   file exists.
The GPU's name and power limit are read in the same process and printed with the numbers."""
import argparse
import json
import os
import re
import shutil
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from slicer_b200 import capi, host, synth  # noqa: E402
from test_gpu_driver import INI  # noqa: E402

S_ = dict(box=256000.0, npix=2048, fov=5.0, zs=1.0, nsnap=12)  # "c3" of tools/realisations_e2e.py
ap = argparse.ArgumentParser()
ap.add_argument("--ng", type=int, default=512)
ap.add_argument("--numfiles", type=int, default=16)
ap.add_argument("--k", type=int, default=8)
ap.add_argument("--zs", default="1.0,0.75,0.5,0.25")
ap.add_argument("--gpus", default="0")
ap.add_argument("--work", default="/tmp/e2e_real")
ap.add_argument("--out", default=None, help="also append the JSON lines to this file")
ap.add_argument("--reps", type=int, default=20, help="timed light cones of slicer_kappa_add")
ap.add_argument("--runs", type=int, default=3, help="runs of each mode, the modes alternating")
a = ap.parse_args()


def emit(d):
    line = json.dumps(d)
    print(line, flush=True)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "a") as f:
            f.write(line + "\n")


gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                     text=True).stdout.strip().splitlines()
emit(dict(gpu=gpu))

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


PHASES = [("total", "total"), ("setup", "engine/CUDA set-up"), ("reads", "sub-file reads"), ("gpu_waits", r"fetch \(waits for the GPU\)"),
          ("fits_writes", r"FITS writes \(background thread\)"), ("device", "device passes"), ("kappa", "convergence maps"),
          ("kappa_adds", r"\(adds"), ("kappa_out", "read-out and writes")]

zs_list = [float(v) for v in a.zs.split(",")]
MODES = (("planes", []), ("planes+kappa", ["--kappa-zs", a.zs]), ("kappa", ["--kappa-zs", a.zs, "--no-planes"]))
for run_i, (mode, extra) in [(i, m) for i in range(a.runs) for m in MODES]:
    shutil.rmtree(f"{a.work}/kappa_out", ignore_errors=True)
    inis = [ini("kappa_out", k) for k in range(a.k)]
    t0 = time.time()
    r = subprocess.run([host.EXE_PATH, "--quiet", "--gpus", a.gpus, *extra, *inis], cwd=a.work, capture_output=True, text=True,
                       env=dict(os.environ, SLICER_B200_TIMING="1"))
    wall = time.time() - t0
    assert r.returncode == 0, r.stderr[-2000:]
    line = next(l for l in r.stderr.splitlines() if l.startswith("[timing] total"))
    files = os.listdir(f"{a.work}/kappa_out")
    emit(dict(mode=mode, run=run_i, K=a.k, S=len(zs_list) if mode != "planes" else 0, ng=a.ng, numfiles=a.numfiles, npix=S_["npix"], wall_s=round(wall, 2),
              phases_s={k: float(re.search(pat + r" ([0-9.e+-]+)", line).group(1)) for k, pat in PHASES},
              plane_files=sum(".plane_" in f for f in files), kappa_files=sum(".kappa_" in f for f in files),
              fits_GB=round(sum(os.path.getsize(f"{a.work}/kappa_out/{f}") for f in files if f.endswith(".fits")) / 1e9, 2)))
shutil.rmtree(f"{a.work}/kappa_out", ignore_errors=True)

# ---- device time of slicer_kappa_add over one light cone ------------------------------------------------------------------------
plan = host.plan(0.3, 0.7, -1.0, S_["zs"], [0.1 * i for i in range(S_["nsnap"])], [S_["box"]] * S_["nsnap"], a.work + "/", "kappa_e2e")
nplanes, npix, S = plan["nplanes"], S_["npix"], len(zs_list)
w = host.kappa_weights(0.3, 0.7, -1.0, S_["zs"], [0.1 * i for i in range(S_["nsnap"])], [S_["box"]] * S_["nsnap"], S_["fov"], npix, zs_list)
calls = [(q, min(16, nplanes - q)) for q in range(0, nplanes, 16)]
n = 1 << 24
with capi.Slicer(npix_max=npix, max_planes=16, particle_capacity=n + 64) as s:
    s.begin_snapshot(S_["box"], [0, 1.0375, 0, 0, 0, 0], False)
    s.stage_synthetic(1, n, 5)
    fov = S_["fov"] / 180 * 3.141592653589793
    s.deposit([capi.plane_desc([1, 1, 1], 1, [0.5, 0.5, 0.5], 0.0, 16.0 * j, 16.0 * (j + 1), fov, npix) for j in range(16)])
    s.kappa_maps(S, npix)

    def light_cone():
        for q, m in calls:  # the planes q .. q+m-1 of the light cone, in slots 0 .. m-1
            s.kappa_add(0, [0] * m, w["scale"][q:q + m], w["offset"][q:q + m])

    for _ in range(3):
        light_cone()
    s.synchronize()
    times = []
    for _ in range(a.reps):
        s.timer_begin()
        light_cone()
        times.append(s.timer_end())
    s.kappa_fetch(0)
times.sort()
ms = times[len(times) // 2]
touched = [int(((w["scale"][q:q + m] != 0) | (w["offset"][q:q + m] != 0)).any(axis=0).sum()) for q, m in calls]
nbytes = 8 * npix * npix * (nplanes + 2 * sum(touched))
peak = None
pk = os.path.join(ROOT, "MEASURED_PEAKS.json")
if os.path.exists(pk):
    peak = json.load(open(pk)).get("hbm_gbs")
emit(dict(kernel="kappa_add_kernel", npix=npix, planes=nplanes, sources=S, calls=len(calls), median_ms=round(ms, 4), min_ms=round(times[0], 4),
          ms_per_plane=round(ms / nplanes, 4), bytes=nbytes, GBs=round(nbytes / ms / 1e6, 1), hbm_gbs=peak,
          share_of_hbm=round(nbytes / ms / 1e6 / peak, 3) if peak else None, gpu=gpu))
