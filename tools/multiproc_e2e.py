"""Measurement aid: one light cone on configuration-shaped synthetic snapshots as ONE SLICER_b200 process driving N GPUs
(--gpus 0,..,N-1) and as a job of N processes with one GPU each (torchrun's variables on 127.0.0.1), N from --ns.
usage: python tools/multiproc_e2e.py [--ng 512] [--numfiles 16] [--shape c3] [--ns 2,8] [--repeats 2] [--work /tmp/e2e_mp]
Prints one JSON line per N: wall time of both (each repeated, alternating, best and all), rank 0's SLICER_B200_TIMING phases,
whether the two output sets are byte-identical, and the GPU's name and power limit.  N larger than the visible GPUs is skipped.
Snapshot files are written before timing (page cache warm).  One node cannot show the gain of more nodes' read and copy
bandwidth; what this measures is what the processes cost against one process on the same GPUs."""
import argparse
import filecmp
import json
import os
import re
import shutil
import socket
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from slicer_b200 import capi, host, synth  # noqa: E402
from test_gpu_driver import INI  # noqa: E402

SHAPES = {"c1": dict(box=128000.0, npix=256, fov=2.0, zs=0.5, nsnap=7), "c3": dict(box=256000.0, npix=2048, fov=5.0, zs=1.0, nsnap=12)}
ap = argparse.ArgumentParser()
ap.add_argument("--ng", type=int, default=512)
ap.add_argument("--numfiles", type=int, default=16)
ap.add_argument("--shape", default="c3", choices=sorted(SHAPES))
ap.add_argument("--ns", default="2,8")
ap.add_argument("--repeats", type=int, default=2)
ap.add_argument("--work", default="/tmp/e2e_mp")
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
LAUNCHER = ("OMPI_COMM_WORLD_RANK", "OMPI_COMM_WORLD_SIZE", "PMI_RANK", "PMI_SIZE", "SLURM_PROCID", "SLURM_STEP_NUM_TASKS", "RANK", "WORLD_SIZE",
            "TORCHELASTIC_RUN_ID")
BASE_ENV = {k: v for k, v in os.environ.items() if k not in LAUNCHER}
BASE_ENV["SLICER_B200_TIMING"] = "1"


def ini(tag):
    out = f"{a.work}/{tag}"
    shutil.rmtree(out, ignore_errors=True)
    os.makedirs(out)
    path = f"{a.work}/{tag}.ini"
    open(path, "w").write(INI.format(npix=S["npix"], zs=S["zs"], fov=S["fov"], list=a.work + "/snapshot_list.txt", snapdir=a.work + "/snaps/",
                                     outdir=out + "/lc_", pip=0, snopt=0))
    return path


def timing(stderr):
    line = next(l for l in stderr.splitlines() if l.startswith("[timing]"))
    return {k: float(re.search(k + r" ([0-9.e+-]+)", line).group(1)) for k in ("total", "set-up", "reads", "device passes")}


def one_process(n):
    path = ini("one")
    t0 = time.time()
    r = subprocess.run([host.EXE_PATH, "--quiet", "--gpus", ",".join(map(str, range(n))), path], cwd=a.work, capture_output=True, text=True,
                       env=BASE_ENV)
    wall = time.time() - t0
    assert r.returncode == 0, r.stderr[-2000:]
    return wall, timing(r.stderr)


def job(n):
    path = ini("job")
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    t0 = time.time()
    procs = [subprocess.Popen([host.EXE_PATH, "--quiet", "--gpus", str(r), path], cwd=a.work, stdout=subprocess.PIPE, stderr=subprocess.PIPE,
                              text=True, env=dict(BASE_ENV, RANK=str(r), WORLD_SIZE=str(n), LOCAL_RANK=str(r), MASTER_ADDR="127.0.0.1",
                                                  MASTER_PORT=str(port))) for r in range(n)]
    try:
        outs = [p.communicate(timeout=3600) for p in procs]
    finally:
        for p in procs:
            if p.poll() is None:
                p.kill()
                p.communicate()
    wall = time.time() - t0
    assert all(p.returncode == 0 for p in procs), [e[-2000:] for _, e in outs]
    return wall, timing(outs[0][1])


gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout.splitlines()
for n in [int(v) for v in a.ns.split(",")]:
    if capi.device_count() < n:
        print(json.dumps(dict(N=n, skipped=f"{capi.device_count()} GPUs visible")), flush=True)
        continue
    walls = {"one_process": [], "n_processes": []}
    phases = {}
    for _ in range(a.repeats):  # alternating, so that both see the same state of the shared host
        for tag, fn in (("one_process", one_process), ("n_processes", job)):
            w, ph = fn(n)
            walls[tag].append(round(w, 2))
            phases[tag] = ph
    files = sorted(os.listdir(f"{a.work}/one"))
    same = files == sorted(os.listdir(f"{a.work}/job")) and all(filecmp.cmp(f"{a.work}/one/{f}", f"{a.work}/job/{f}", shallow=False) for f in files)
    print(json.dumps(dict(shape=a.shape, ng=a.ng, numfiles=a.numfiles, snapshots=S["nsnap"], npix=S["npix"], N=n,
                          planes=sum(f.endswith(".fits") for f in files), wall_s=walls,
                          best_s={k: min(v) for k, v in walls.items()}, rank0_phases_s=phases, byte_identical=same, gpu=gpu[:n])), flush=True)
