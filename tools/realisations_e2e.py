"""Measurement aid: K light-cone realisations (inis that differ only in their seeds and output suffix) on configuration-shaped
synthetic snapshots, as K separate `SLICER_b200 X.ini` runs and as one `SLICER_b200 A.ini B.ini ...` run.
usage: python tools/realisations_e2e.py [--ng 512] [--numfiles 16] [--shape c3] [--ks 1,4,8] [--gpus 0] [--work /tmp/e2e_real]
Prints one JSON line per K: wall time of both, the driver's SLICER_B200_TIMING phases (set-up, sub-file reads, waits for the
GPU, FITS writes, device time of the passes), device time per light cone, and whether the two output sets are byte-identical.
Snapshot files are written before timing (page cache warm); each K's outputs are removed after its comparison."""
import argparse
import filecmp
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
from slicer_b200 import host, synth  # noqa: E402
from test_gpu_driver import INI  # noqa: E402

SHAPES = {"c1": dict(box=128000.0, npix=256, fov=2.0, zs=0.5, nsnap=7), "c3": dict(box=256000.0, npix=2048, fov=5.0, zs=1.0, nsnap=12)}
ap = argparse.ArgumentParser()
ap.add_argument("--ng", type=int, default=512)
ap.add_argument("--numfiles", type=int, default=16)
ap.add_argument("--gpus", default="0")
ap.add_argument("--shape", default="c3", choices=sorted(SHAPES))
ap.add_argument("--ks", default="1,4,8")
ap.add_argument("--work", default="/tmp/e2e_real")
a = ap.parse_args()
S = SHAPES[a.shape]
os.makedirs(a.work + "/snaps", exist_ok=True)
names = []
for i in range(S["nsnap"]):
    base = f"{a.work}/snaps/snap_{i:03d}"
    if not os.path.exists(base + ".0"):
        synth.write_snapshot(base, {1: synth.hash_positions(a.ng ** 3, S["box"], 1000 + i)}, [0, 1.0375, 0, 0, 0, 0], 0.1 * i, S["box"],
                             numfiles=a.numfiles, with_vel_id=False)
    names.append(f"snap_{i:03d}")
open(a.work + "/snapshot_list.txt", "w").write("\n".join(names))


def ini(tag, k):
    """realisation k: its own seed triple (entries 7-9) and suffix (entry 12), output directory `tag`"""
    out = f"{a.work}/{tag}"
    os.makedirs(out, exist_ok=True)
    t = INI.format(npix=S["npix"], zs=S["zs"], fov=S["fov"], list=a.work + "/snapshot_list.txt", snapdir=a.work + "/snaps/", outdir=out + "/lc_",
                   pip=0, snopt=0)
    for old, new in zip((-229, -230, -231), (-229 - 17 * k, -230 + 5 * k, -231 - 3 * k)):
        t = t.replace(f"\n{old}\n", f"\n{new}\n")
    t = t.replace("PLC Suffix ###########\n0\n", f"PLC Suffix ###########\nr{k}\n")
    path = f"{a.work}/{tag}_{k}.ini"
    open(path, "w").write(t)
    return path


PHASES = [("total", "total"), ("setup", "engine/CUDA set-up"), ("reads", "sub-file reads"), ("gpu_waits", r"fetch \(waits for the GPU\)"),
          ("fits_writes", r"FITS writes \(background thread\)"), ("device", "device passes")]


def run(inis):
    t0 = time.time()
    r = subprocess.run([host.EXE_PATH, "--quiet", "--gpus", a.gpus, *inis], cwd=a.work, capture_output=True, text=True,
                       env=dict(os.environ, SLICER_B200_TIMING="1"))
    wall = time.time() - t0
    assert r.returncode == 0, r.stderr[-2000:]
    line = next(l for l in r.stderr.splitlines() if l.startswith("[timing] total"))
    return wall, {k: float(re.search(pat + r" ([0-9.e+-]+)", line).group(1)) for k, pat in PHASES}


for K in [int(v) for v in a.ks.split(",")]:
    for tag in ("alone", "together"):
        shutil.rmtree(f"{a.work}/{tag}", ignore_errors=True)
    sep_wall, sep = 0.0, {k: 0.0 for k, _ in PHASES}
    for k in range(K):
        w, ph = run([ini("alone", k)])
        sep_wall += w
        sep = {key: sep[key] + ph[key] for key in sep}
    one_wall, one = run([ini("together", k) for k in range(K)])
    files = sorted(os.listdir(f"{a.work}/alone"))
    same = files == sorted(os.listdir(f"{a.work}/together")) and all(
        filecmp.cmp(f"{a.work}/alone/{f}", f"{a.work}/together/{f}", shallow=False) for f in files)
    fits = [f for f in files if f.endswith(".fits")]
    print(json.dumps(dict(shape=a.shape, ng=a.ng, numfiles=a.numfiles, snapshots=S["nsnap"], npix=S["npix"], gpus=a.gpus, K=K, planes=len(fits),
                          fits_GB=round(sum(os.path.getsize(f"{a.work}/together/{f}") for f in fits) / 1e9, 2),
                          separate_wall_s=round(sep_wall, 2), together_wall_s=round(one_wall, 2), speedup=round(sep_wall / one_wall, 2),
                          separate_phases_s={k: round(v, 3) for k, v in sep.items()}, together_phases_s={k: round(v, 3) for k, v in one.items()},
                          device_s_per_light_cone=dict(separate=round(sep["device"] / K, 3), together=round(one["device"] / K, 3)),
                          byte_identical=same)), flush=True)
    for tag in ("alone", "together"):
        shutil.rmtree(f"{a.work}/{tag}", ignore_errors=True)
