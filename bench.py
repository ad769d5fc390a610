#!/usr/bin/env python
"""bench.py — throughput of the light-cone mass-map hot path on B200 (and of the reference's CPU path beside it).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload c3|c4|c5] [--scaling strong|weak]
                    [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Workloads (BASELINE.json configs; synthetic uniform particles from a counter hash, resident in HBM before the timed region):
  c3  configs[2]  1024^3 DM particles, box 256 Mpc/h, 2048^2 map, 5 deg, zs = 1.0, TSC; light cone = 9 randomisation groups
  c5  configs[4]  2048^3 DM particles, box 1000 Mpc/h, 8192^2 map, 5 deg, TSC; light cone = 6 groups (piled boxes to zs ~ 4)
  c4  configs[3]  gas + DM + stars, 512^3 each, per-particle masses for gas and stars (1 % above MAX_M), per-type 1024^2 maps
                  (Part. in Planes = 1), geometry of c3
One STEP = one whole light cone: one pass of the hot path per randomisation group; a pass streams every resident particle
through box transform -> shell selection -> projection -> FoV cut -> TSC deposit into the 4 lens planes of the group
(numberOfLensPerSnap = 4, densitymaps.h:23) and leaves the finished int64 planes in HBM (on rank 0 after the reduce).
The reference needs 4 passes over the snapshot for the same 4 planes (slicer-v2.cpp:138-207); both arms report
`particles / second` = snapshot particles turned into their 4 planes per second.

Multi-GPU: particles shard over the ranks (the reference: sub-files over MPI ranks, slicer-v2.cpp:162-175), every rank
deposits into private planes and the planes are summed onto rank 0 with ncclReduce(int64) inside the step (replaces
slicer-v2.cpp:214-217), on its own stream and into alternating accumulator slots so that it overlaps the next pass.
  --scaling strong (default): the workload's particle count is split over the N GPUs (configs[2]: "sharded over 8 GPUs")
  --scaling weak            : every rank holds the whole count
"""
from __future__ import annotations

import argparse
import ctypes
import hashlib
import json
import math
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "tsc_deposited_particles_per_sec"
UNIT = "particles/s"
SEEDS = (-229, -230, -231)   # examples/InputParams.ini
LENS_PER_SNAP = 4
MASS = 5.2                   # 1e10 Msun/h, massarr[1]

WORKLOADS = {
    "c3": dict(label="C3", ng=1024, species=1, box=256000.0, npix=2048, fov_deg=5.0, zs=1.0, ngroups=9, per_type=False,
               text="synthetic 1024^3 DM particles (uniform, counter-hash), box 256 Mpc/h, 2048^2 map, 5 deg, zs=1.0, TSC"),
    "c5": dict(label="C5", ng=2048, species=1, box=1000000.0, npix=8192, fov_deg=5.0, zs=4.0, ngroups=6, per_type=False,
               text="synthetic 2048^3 DM particles, box 1000 Mpc/h, 8192^2 map, 5 deg, 6 piled boxes (zs ~ 4), TSC"),
    "c4": dict(label="C4", ng=512, species=3, box=256000.0, npix=1024, fov_deg=5.0, zs=1.0, ngroups=9, per_type=True,
               text="synthetic hydro snapshot: gas + DM + stars, 512^3 each, per-particle masses for gas and stars (1 % above "
                    "MAX_M), Part. in Planes=1 (per-type maps), box 256 Mpc/h, 1024^2 map, 5 deg, zs=1.0, TSC"),
}
# aliases kept for tools/
NG, BOX, NPIX, FOV_DEG, ZS, NGROUPS = 1024, 256000.0, 2048, 5.0, 1.0, 9


def c3_planes(BOX=BOX, NPIX=NPIX, FOV_DEG=FOV_DEG, NGROUPS=NGROUPS):
    """Plane descriptors of a light cone, group by group: the plan arithmetic of buildPlanes / randomizeBox, taken from the
    product's C++ plan stage (slicer_b200/host/plan.cpp through slicer_b200/host.py)."""
    from slicer_b200 import capi, host

    nplanes = NGROUPS * LENS_PER_SNAP
    randomize = [1 if i % LENS_PER_SNAP == 0 else 0 for i in range(nplanes)]
    rnd = host.randomize_box(*SEEDS, randomize)
    fov = float(np.float32(FOV_DEG))  # data.cpp:29 parses fov with stof
    fovrad = fov / 180.0 * math.pi
    thick = BOX / 1e3 / LENS_PER_SNAP
    groups, raw = [], []
    ld2 = 0.0
    for i in range(nplanes):
        ld = ld2
        ld2 = ld + thick  # ldbut += box/1e3/numOfLensPerSnap (densitymaps.cpp:93-100): a running sum
        g = i // LENS_PER_SNAP
        # rcase = floor(ld/box*1e3) (slicer-v2.cpp:137,184-185)
        d = dict(sgn=[int(rnd["sgnX"][i]), int(rnd["sgnY"][i]), int(rnd["sgnZ"][i])], face=int(rnd["face"][i]),
                 centre=[float(rnd["x0"][i]), float(rnd["y0"][i]), float(rnd["z0"][i])], rcase=float(g), ld=ld, ld2=ld2,
                 nrepperp=0, fovradiants=fovrad, boxsize=BOX)
        raw.append(d)
        if i % LENS_PER_SNAP == 0:
            groups.append([])
        groups[-1].append(capi.plane_desc(d["sgn"], d["face"], d["centre"], d["rcase"], d["ld"], d["ld2"], fovrad, NPIX))
    return groups, raw


def shard_range(total: int, world: int, rank: int):
    """Contiguous particle range of `rank` under strong scaling (multiples of 4 so that every shard stays 16-byte aligned)."""
    q = (total // world) & ~3
    lo = rank * q
    hi = total if rank == world - 1 else lo + q
    return lo, hi


def linear_checksums(a: np.ndarray):
    """Two linear functionals of an int64 plane modulo 2^64: sum(a) and sum(a * (i + 1)).  Linear, so the checksums of a
    reduced plane equal the sums of the per-rank checksums — the bench uses this to verify ncclReduce(int64) on hardware."""
    u = np.ascontiguousarray(a).reshape(-1).view(np.uint64)
    with np.errstate(over="ignore"):
        s0 = int(u.sum(dtype=np.uint64))
        s1 = int((u * np.arange(1, u.size + 1, dtype=np.uint64)).sum(dtype=np.uint64))
    return s0, s1


def exact_sum(a: np.ndarray) -> int:
    """Sum of an int64 plane as a Python integer (a 2048^2 plane of 2^40-scaled masses overflows int64)."""
    a = np.ascontiguousarray(a).reshape(-1)
    return (int((a >> 24).sum()) << 24) + int((a & ((1 << 24) - 1)).sum())


def csrc_sha() -> str:
    """Hash of the CUDA sources: ncu-derived numbers under profiles/ are stamped with it and only quoted when it matches."""
    h = hashlib.sha256()
    d = os.path.join(ROOT, "slicer_b200", "csrc")
    for f in sorted(os.listdir(d)):
        if f.endswith((".cu", ".cuh", ".h")):
            h.update(open(os.path.join(d, f), "rb").read())
    return h.hexdigest()[:16]


# ---- clocks --------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.rows = []
        self.proc = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "50",
                                          "-i", str(index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), line.strip()))

    def stop(self):
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()

    def summary(self, t0, t1):
        sm, mx, reasons = [], [], set()
        for t, line in self.rows:
            if t < t0 or t > t1 + 0.15:
                continue
            p = [v.strip() for v in line.split(",")]
            try:
                sm.append(float(p[0]))
                mx.append(float(p[1]))
            except Exception:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), p[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons), "samples": len(sm)}


# ---- the reference on the host cores -------------------------------------------------------------------------
def _write_sample_file(path_base, n, seed, box, start=0):
    from slicer_b200 import synth

    pos = synth.hash_positions(n, box, seed, start=start)
    synth.write_snapshot(path_base, {1: pos}, [0, MASS, 0, 0, 0, 0], 0.0, box, numfiles=1, with_vel_id=False)
    return path_base


def _ref_worker(args):
    """One 'MPI rank' of the reference: createDensityMaps (densitymaps.cpp:419) on its own sub-file, for each of the
    4 planes of each group in `groups` (a full snapshot pass per plane, exactly as slicer-v2.cpp:138-207 drives it)."""
    path_base, raw_planes, groups, npix = args
    from oracle.ref_bindings import RefLib

    devnull = os.open(os.devnull, os.O_WRONLY)
    os.dup2(devnull, 1)  # the reference prints per-type min/max for rank 0; keep the bench's stdout clean
    ref = RefLib(ngp=False)
    t0 = time.perf_counter()
    checksum = 0.0
    for g in groups:
        for p in raw_planes[g * LENS_PER_SNAP:(g + 1) * LENS_PER_SNAP]:
            m = ref.create_density_maps(path_base, 0, 1, npix, p["fovradiants"], p["sgn"], p["face"], p["centre"], p["rcase"],
                                        p["ld"], p["ld2"], p["nrepperp"])
            checksum += float(m.sum(dtype=np.float64))
    return time.perf_counter() - t0, checksum


def run_reference_sample(ncores, n_per_core, groups, raw_planes, tmpdir, W, seed=1234):
    """-> (particles/s for the 4-planes-per-snapshot job, wall seconds).  Files are written before timing."""
    import multiprocessing as mp

    bases = []
    for r in range(ncores):
        bases.append(_write_sample_file(os.path.join(tmpdir, f"sample_{r}"), n_per_core, seed, W["box"], start=r * n_per_core))
    jobs = [(b, raw_planes, groups, W["npix"]) for b in bases]
    if ncores == 1:
        saved = os.dup(1)
        try:
            res = [_ref_worker(jobs[0])]
        finally:
            os.dup2(saved, 1)
            os.close(saved)
    else:
        with mp.get_context("fork").Pool(ncores) as pool:
            res = pool.map(_ref_worker, jobs)
    wall = max(r[0] for r in res)  # slowest rank, as an MPI job would finish; excludes process start-up
    # every group = one snapshot turned into its 4 planes; all ranks work on disjoint sub-files of that snapshot
    particles = ncores * n_per_core * len(groups)
    return particles / wall, wall, res


def reference_arm(args, rank, world):
    if rank != 0:
        return
    from oracle import ref_bindings

    if not ref_bindings.available():
        print(json.dumps({"impl": "reference", "unavailable": "oracle/_ref/libslicer_ref.so not built"}))
        return
    W = WORKLOADS[args.workload]
    _, raw = c3_planes(W["box"], W["npix"], W["fov_deg"], W["ngroups"])
    ncores = os.cpu_count() or 1
    # a step = a bounded sample of the workload's step: each core streams a `n_per_core`-particle sub-file of the snapshot into the
    # 4 planes of ONE group of the light cone (step i: group i mod ngroups), ~0.12 us per particle and plane -> ~2 s per step.
    # (Sub-files much smaller than this would charge the reference its per-call set-up — 7 maps of npix^2 floats — over and over.)
    n_per_core = 1 << 22
    ngr = W["ngroups"]
    with tempfile.TemporaryDirectory() as td:
        for i in range(args.warmup):
            run_reference_sample(ncores, n_per_core, [i % ngr], raw, td, W)
        wall = 0.0  # the sample files are written outside the timed part of run_reference_sample
        particles = 0
        for i in range(args.steps):
            _, w, _ = run_reference_sample(ncores, n_per_core, [i % ngr], raw, td, W)
            wall += w
            particles += ncores * n_per_core
    value = particles / wall
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": wall / args.steps * 1e3, "higher_is_better": True, "scaling": args.scaling,
        "vs_baseline": None, "dtype": "f32+f64", "data": "synthetic",
        "config": workload_config(args.workload, args.scaling, args.gpus),  # identical to our arm's; the sample is described in cpu_baseline
        "sample": f"{ncores} sub-files x {n_per_core} particles into the 4 planes of one group per step",
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": ncores, "kind": "reference",
                         "sample": f"{ncores} processes (one per host core, as MPI ranks over sub-files), each createDensityMaps on a "
                                   f"{n_per_core}-particle sub-file for the {LENS_PER_SNAP} planes of one group of the light cone per step "
                                   f"(step i: group i mod {ngr})"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


def workload_config(name, scaling, n_gpus):
    W = WORKLOADS[name]
    total = W["species"] * W["ng"] ** 3
    per_gpu = total if scaling == "weak" else total // n_gpus
    return {
        "workload": f"{W['label']}: {W['text']}; step = one light cone = {W['ngroups']} snapshot passes, each into the "
                    f"{LENS_PER_SNAP} lens planes of one randomisation group",
        "particles_total": total * (n_gpus if scaling == "weak" else 1), "particles_per_gpu": per_gpu, "npix": W["npix"],
        "fov_deg": W["fov_deg"], "zs": W["zs"], "planes_per_pass": LENS_PER_SNAP, "passes_per_step": W["ngroups"], "mas": "TSC",
        "l2": "inputs per pass larger than L2 (126 MB) at every N; no flush needed" if per_gpu * 12 > 4e8 else
              "inputs per pass comparable to L2; every pass reads a different projection and writes fresh accumulators",
        "parallelism": (f"particle shards x{n_gpus} ({scaling} scaling), ncclReduce(int64) of the 4 planes per pass on its own "
                        "stream, alternating accumulator slots") if n_gpus > 1 else "1 GPU",
    }


# ---- our arm -------------------------------------------------------------------------------------------------
class Workload:
    """Resident particles of one rank + the light cone's plane groups."""

    def __init__(self, name, scaling, rank, world, local_rank, deposit_mode=0, guard_eta=0.0):
        from slicer_b200 import capi

        self.name, self.W = name, WORKLOADS[name]
        W = self.W
        self.world, self.rank = world, rank
        self.groups, self.raw = c3_planes(W["box"], W["npix"], W["fov_deg"], W["ngroups"])
        per_species = W["ng"] ** 3
        if scaling == "weak":
            lo, hi = 0, per_species
            self.seed_off = rank  # every rank its own realisation
        else:
            lo, hi = shard_range(per_species, world, rank)
            self.seed_off = 0     # one realisation, sharded
        self.lo, self.hi = lo, hi
        self.n_species = hi - lo
        self.n = self.n_species * W["species"]
        self.total = per_species * W["species"] * (world if scaling == "weak" else 1)
        self.bytes_per_pass = self.n_species * (12 if W["species"] == 1 else 16 + 12 + 16)
        self.hydro = W["species"] == 3
        self.massarr = [0, MASS, 0, 0, 0, 0]
        self._torch_keep = []
        self.s = capi.Slicer(npix_max=W["npix"], max_planes=2 * LENS_PER_SNAP, mas=capi.MAS_TSC,
                             particle_capacity=0 if self.hydro else self.n + 64, device=local_rank, deposit_mode=deposit_mode,
                             record_capacity=min(self.n, 1 << 30), per_type_maps=W["per_type"], guard_eta=guard_eta)
        self.s.begin_snapshot(W["box"], self.massarr, self.hydro)
        if self.hydro:
            self._stage_hydro(local_rank)
        else:
            self._stage_dm()
        self.s.synchronize()

    def _stage_dm(self, s=None):
        # the counter hash is keyed by the global particle index, so a shard is a window of the one realisation; segments of at
        # most 2^31 particles (the library streams a segment with 32-bit particle indices)
        s = s or self.s
        self.segments = []
        done = 0
        while done < self.n_species:
            m = min(self.n_species - done, 1 << 31)
            s.stage_synthetic(1, m, 1000 + self.seed_off, start=self.lo + done)
            self.segments.append(m)
            done += m

    def _stage_hydro(self, local_rank):
        import torch

        dev = torch.device("cuda", local_rank)
        n = self.n_species
        for k, ptype in enumerate((0, 1, 4)):
            g = torch.Generator(device=dev)
            g.manual_seed(4242 + 17 * k + 1000 * self.seed_off)
            pos = torch.rand((self.hi, 3), generator=g, device=dev, dtype=torch.float32)[self.lo:].contiguous() * float(np.float32(self.W["box"]))
            mass = None
            if ptype != 1:
                mass = (torch.rand(self.hi, generator=g, device=dev, dtype=torch.float32)[self.lo:] * 2.0 + 0.05).contiguous()
                mass[::100] = 2000.0  # above MAX_M = 1e3 (densitymaps.h:21): counted, deposited as 0
            self._torch_keep += [pos, mass]
            torch.cuda.synchronize()
            self.s.stage_device(ptype, pos.data_ptr(), n, mass.data_ptr() if mass is not None else 0)

    def close(self):
        self.s.close()
        self._torch_keep = []


def run_light_cones(wl: Workload, steps, warmup, world, barrier, max_over_ranks):
    """Timed region: `steps` light cones.  Returns (ms total, stats, per-pass bookkeeping)."""
    s = wl.s
    ngr = wl.W["ngroups"]

    def finish(slot):
        # the planes of a pass are finished once the pairs it left to the host's libm are settled (and, at N > 1, summed onto
        # rank 0 on the communication stream); both wait for that pass only
        if world > 1:
            s.reduce_slots(slot, LENS_PER_SNAP, 0)
        else:
            s.settle_slots(slot, LENS_PER_SNAP)

    def light_cone():
        # two ranges of accumulator slots: the next pass is submitted before the previous one is finished off, so the device
        # does not wait for the host in between; every plane is final (in HBM, on rank 0) when the light cone returns
        prev = None
        for g in range(ngr):
            slot = (g & 1) * LENS_PER_SNAP
            s.deposit_slots(wl.groups[g], slot)
            if prev is not None:
                finish(prev)
            prev = slot
        finish(prev)

    for _ in range(warmup):
        light_cone()
    s.synchronize()
    s.reset_stats()
    f0 = s.stats().flagged_pairs
    barrier()
    s.synchronize()
    t0 = time.time()
    s.timer_begin()
    for _ in range(steps):
        light_cone()
    s.synchronize()
    ms = s.timer_end()
    barrier()
    t1 = time.time()
    ms = max_over_ranks(ms)
    st = s.stats()
    return ms, st, (t0, t1), int(st.flagged_pairs - f0)


DUMP_MAP_BYTES = 40 << 20  # the maps; with the sample's float64 pixel indices and the small arrays < 64e6 bytes in all
DUMP_SEED = 20240229


def dump_outputs(wl: Workload, out_dir, rank=0, world=1):
    """The planes of every group of the last timed light cone, as slicer_fetch hands them to a caller: per plane (and map type)
    the float32 map, accepted and in-grid counts, plus the map's float64 sum over all pixels.  The last two groups are read from
    the accumulator slots the timed step left them in.  The two slot ranges alternate, so the earlier groups were overwritten
    within the step: they are deposited again here, after the timed region, with the calls the step makes (integer accumulators:
    the same planes).  Maps larger than the budget are cut to one fixed, seeded sample of pixels, the same for every map
    (pixel_index.npy).  Every rank takes part (the reduces); rank 0 writes DIR/group<g>_*.npy."""
    W = wl.W
    npix, ngr = W["npix"], W["ngroups"]
    types = [0, 1, 4] if W["per_type"] else [-1]  # per-type maps: the types _stage_hydro stages
    nmaps = ngr * LENS_PER_SNAP * len(types)
    size = npix * npix
    sample = None
    if nmaps * size * 4 > DUMP_MAP_BYTES:
        sample = np.sort(np.random.default_rng(DUMP_SEED).choice(size, DUMP_MAP_BYTES // (4 * nmaps), replace=False))
    sfx = {t: "" if t < 0 else f"_type{t}" for t in types}
    if rank == 0:
        os.makedirs(out_dir, exist_ok=True)
    # the groups still in their slots first, then the earlier ones through slot 0
    for g in [g for g in (ngr - 1, ngr - 2) if g >= 0] + list(range(ngr - 2)):
        slot = (g & 1) * LENS_PER_SNAP if g >= ngr - 2 else 0
        if g < ngr - 2:
            wl.s.deposit_slots(wl.groups[g], slot)
            if world > 1:
                wl.s.reduce_slots(slot, LENS_PER_SNAP, 0)
            else:
                wl.s.settle_slots(slot, LENS_PER_SNAP)
        if rank != 0:
            continue
        out = {"counts": [], "ingrid": []}
        for t in types:
            out["maps" + sfx[t]], out["map_sums" + sfx[t]] = [], []
        for k in range(LENS_PER_SNAP):
            for t in types:
                m, c, i = wl.s.fetch(slot + k, t, npix)
                m = m.reshape(-1)
                out["map_sums" + sfx[t]].append(m.sum(dtype=np.float64))
                out["maps" + sfx[t]].append(m if sample is None else m[sample])
            out["counts"].append(c.astype(np.float64))  # accepted pairs per type, whichever map was fetched
            out["ingrid"].append(i.astype(np.float64))
        for key, v in out.items():
            np.save(os.path.join(out_dir, f"group{g}_{key}.npy"), np.stack(v))
    if sample is not None and rank == 0:
        np.save(os.path.join(out_dir, "pixel_index.npy"), sample.astype(np.float64))


def per_group_times(wl: Workload):
    out = []
    for g in range(wl.W["ngroups"]):
        wl.s.deposit_slots(wl.groups[g], 0)
        wl.s.synchronize()
        out.append(wl.s.stats().last_deposit_ms)
    return out


def verify_single(wl: Workload, local_rank, groups=(1, -1)):
    """N = 1 self-check, outside the timed region: the planes the production path leaves in HBM against the one-thread-per-particle
    baseline kernel (SLICER_KERNEL_SIMPLE: no screen, no queues, no sort, map atomics straight from the general chain) on the same
    particles: counts, total mass and pixels.  Both paths hand the pairs inside their rounding guard to the host's libm, so the
    planes are expected to be identical."""
    from slicer_b200 import capi

    if wl.hydro:
        return None
    W = wl.W
    ref = capi.Slicer(npix_max=W["npix"], max_planes=LENS_PER_SNAP, mas=capi.MAS_TSC, particle_capacity=wl.n + 64, device=local_rank,
                      kernel=capi.KERNEL_SIMPLE)
    ref.begin_snapshot(W["box"], wl.massarr, False)
    wl._stage_dm(ref)
    out = {"against": "SLICER_KERNEL_SIMPLE on the same particles", "groups": [], "counts_equal": True, "mass_rel_diff_max": 0.0,
           "pixels_differing": 0, "pixels_compared": 0}
    for g in groups:
        g = g % W["ngroups"]
        wl.s.deposit_slots(wl.groups[g], 0)
        ref.deposit(wl.groups[g])
        for k in range(LENS_PER_SNAP):
            a = wl.s.fetch_fixed(k, -1, W["npix"])
            b = ref.fetch_fixed(k, -1, W["npix"])
            ca, cb = wl.s.fetch(k, -1, W["npix"], want_map=False)[1:], ref.fetch(k, -1, W["npix"], want_map=False)[1:]
            out["counts_equal"] = out["counts_equal"] and ca[0].tolist() == cb[0].tolist() and ca[1].tolist() == cb[1].tolist()
            sa, sb = exact_sum(a), exact_sum(b)
            if sb:
                out["mass_rel_diff_max"] = max(out["mass_rel_diff_max"], abs(sa - sb) / abs(sb))
            out["pixels_differing"] += int(np.count_nonzero(a != b))
            out["pixels_compared"] += int(a.size)
            if k == LENS_PER_SNAP - 1:
                out["groups"].append({"group": g, "accepted_pairs_plane3": int(ca[0][1]), "mass_plane3": sa * 2.0 ** -wl.s.frac_bits})
    ref.close()
    # a pair whose float map coordinate differs by one ulp between the two evaluations moves 9 stencil pixels by ~1e-4 of its mass
    out["ok"] = bool(out["counts_equal"] and out["mass_rel_diff_max"] <= 1e-12 and out["pixels_differing"] <= 9 * 8)
    return out


def verify_reduce(wl: Workload, world, rank, dist, group=-1):
    """N > 1: the reduced planes on rank 0 against the per-rank planes, through two linear checksums modulo 2^64."""
    import torch

    W = wl.W
    g = group % W["ngroups"]
    s = wl.s
    s.deposit_slots(wl.groups[g], 0)
    mine = []
    for k in range(LENS_PER_SNAP):
        a = s.fetch_fixed(k, -1, W["npix"])
        c = s.fetch(k, -1, W["npix"], want_map=False)[1]
        mine.append(list(linear_checksums(a)) + [int(c.sum())])
    # signed 64-bit transport of the unsigned checksums
    t = torch.tensor([[v - (1 << 64) if v >= (1 << 63) else v for v in row] for row in mine], dtype=torch.int64)
    allt = [torch.zeros_like(t) for _ in range(world)]
    dist.all_gather(allt, t)
    s.deposit_slots(wl.groups[g], 0)
    s.reduce_slots(0, LENS_PER_SNAP, 0)
    ok = True
    if rank == 0:
        for k in range(LENS_PER_SNAP):
            a = s.fetch_fixed(k, -1, W["npix"])
            c = s.fetch(k, -1, W["npix"], want_map=False)[1]
            s0, s1 = linear_checksums(a)
            e0 = sum(int(x[k][0]) for x in allt) & ((1 << 64) - 1)
            e1 = sum(int(x[k][1]) for x in allt) & ((1 << 64) - 1)
            ec = sum(int(x[k][2]) for x in allt)
            ok = ok and s0 == e0 and s1 == e1 and int(c.sum()) == ec
    else:
        s.synchronize()
    flag = torch.tensor([1 if ok else 0], dtype=torch.int64)
    dist.broadcast(flag, src=0)
    return bool(flag[0])


def measure(args, name, scaling, steps, warmup, rank, world, local_rank, dist, sample_clocks, verify=True, dump_dir=None):
    """One workload at the current world size -> dict of results (rank 0 holds the aggregated numbers).  With `dump_dir`, rank 0
    writes the planes of the last timed step there (dump_outputs)."""
    import torch

    def barrier():
        if world > 1:
            dist.barrier()

    def max_over_ranks(v):
        if world == 1:
            return v
        t = torch.tensor([v], dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t[0])

    from slicer_b200 import capi

    wl = Workload(name, scaling, rank, world, local_rank, args.deposit_mode)
    if world > 1:
        uid = [capi.Slicer.comm_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(uid, src=0)
        wl.s.comm_init_rank(uid[0], world, rank)
    sampler = ClockSampler(local_rank) if (rank == 0 and sample_clocks) else None
    ms, st, (t0, t1), flagged = run_light_cones(wl, steps, warmup, world, barrier, max_over_ranks)
    clocks = None
    if sampler:
        time.sleep(0.25)
        sampler.stop()
        clocks = sampler.summary(t0, t1)
    if dump_dir:
        dump_outputs(wl, dump_dir, rank, world)  # before per_group_times and the self-checks reuse the accumulator slots
    ngr = wl.W["ngroups"]
    passes = steps * ngr
    value = wl.total * passes / (ms * 1e-3)
    kernel_ms = st.deposit_ms_sum / max(1, st.deposit_passes)  # device time of the pass kernels only (events around each pass)
    res = dict(workload=name, scaling=scaling, value=value, ms=ms, ms_per_step=ms / steps, ms_per_pass=ms / passes, kernel_ms=kernel_ms,
               launches=int(st.launches), flagged_pairs=flagged, bytes_per_pass=wl.bytes_per_pass, n_per_gpu=wl.n, total=wl.total, clocks=clocks)
    res["per_group_ms"] = [round(v, 3) for v in per_group_times(wl)]
    if world == 1 and verify and not args.no_verify:
        res["verify"] = verify_single(wl, local_rank)
    if world > 1 and verify and not args.no_verify:
        res["reduce_ok"] = verify_reduce(wl, world, rank, dist)
    return res, wl


def roofline_of(res, peaks):
    peak = float(peaks.get("hbm_gbs", 6650.0))
    achieved = res["bytes_per_pass"] / (res["kernel_ms"] * 1e-3) / 1e9
    per_group = [round(res["bytes_per_pass"] / (t * 1e-3) / 1e9 / peak, 4) for t in res["per_group_ms"]]
    out = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": None,
           "kernel": "one pass = pipe::deposit_pipelined_kernel<TSC,AOS,SINGLE,*> (TMA-staged stream + float screen + lean exact projection) "
                     "[+ binned::bin_* counting sort + binned::tile_deposit_kernel when > 3 % of the snapshot is inside the field]; "
                     "averaged over the passes of the timed light cones (CUDA events around every pass on the library's compute stream)",
           "kernel_ms": res["kernel_ms"], "algorithmic_bytes_per_launch": res["bytes_per_pass"], "frac_per_group": per_group,
           "peak_source": "MEASURED_PEAKS.json hbm_gbs (measured)" if peaks else "fallback 6650 GB/s"}
    prof = os.path.join(ROOT, "profiles", f"r02_traffic_{res['workload']}.json")
    if os.path.exists(prof):
        try:
            t = json.load(open(prof))
            if t.get("csrc_sha") == csrc_sha():
                out["traffic"] = t.get("dram_bytes_per_launch")
                out["traffic_source"] = f"profiles/r02_traffic_{res['workload']}.json (ncu, same CUDA sources: {t.get('csrc_sha')})"
            else:
                out["traffic_source"] = "profiles/ holds an ncu capture of OTHER CUDA sources: not quoted"
        except Exception:
            pass
    return out


def ours(args, rank, world, local_rank):
    import torch
    import torch.distributed as dist

    from slicer_b200 import capi

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; this framework has no CPU path (use --impl reference for the CPU reference)")
    bad = [k for k in ("SLICER_B200_DEBUG", "SLICER_B200_NO_SERIES", "SLICER_B200_NO_LEAN") if os.environ.get(k)]
    if bad:
        raise SystemExit(f"bench.py: refusing to measure with {', '.join(bad)} set (they switch kernel stages off)")
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("cpu:gloo,cuda:nccl", rank=rank, world_size=world)
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass

    res, wl = measure(args, args.workload, args.scaling, args.steps, args.warmup, rank, world, local_rank, dist, True,
                      dump_dir=args.dump_outputs)
    W = wl.W
    roofline = roofline_of(res, peaks)

    # ------------------------------------------------------------------ e2e phase: host buffers through the C ABI
    e2e = None
    if not args.no_e2e and not wl.hydro:
        # the same particles in pinned host memory; one light cone = 9 snapshots staged sub-file by sub-file (8 batches, two staging
        # pools: the copy of batch k+1 overlaps the pass over batch k), planes reduced and fetched as float maps on rank 0
        nb = 8
        n = wl.n
        per = (n // nb) & ~3
        sizes = [per] * (nb - 1) + [n - per * (nb - 1)]
        pin = capi.PinnedBuffer(n * 12)
        _download_all(wl, pin)
        wl.close()
        e = capi.Slicer(npix_max=W["npix"], max_planes=2 * LENS_PER_SNAP, mas=capi.MAS_TSC, particle_capacity=max(sizes) + 64, staging_buffers=2,
                        device=local_rank, deposit_mode=args.deposit_mode)
        if world > 1:
            uid = [capi.Slicer.comm_unique_id() if rank == 0 else None]
            dist.broadcast_object_list(uid, src=0)
            e.comm_init_rank(uid[0], world, rank)
        maps = [np.empty((W["npix"], W["npix"]), np.float32) for _ in range(LENS_PER_SNAP)]
        cnt = np.zeros(6, np.int64)

        def fetch(slot):
            for k in range(LENS_PER_SNAP):
                capi._check(capi.lib().slicer_fetch(e.h, slot + k, -1, maps[k].ctypes.data, cnt.ctypes.data, None))

        def e2e_light_cone():
            prev = None
            for g in range(W["ngroups"]):
                slot = (g & 1) * LENS_PER_SNAP
                e.begin_snapshot(W["box"], wl.massarr, False)
                o = 0
                for b in range(nb):
                    if b:
                        e.next_batch()
                    e.stage_ptr(1, pin.ptr + o * 12, sizes[b])
                    e.deposit_slots(wl.groups[g], slot, accumulate=b > 0)
                    o += sizes[b]
                if world > 1:
                    e.reduce_slots(slot, LENS_PER_SNAP, 0)
                if rank == 0 and prev is not None:
                    fetch(prev)  # the previous group's maps: their read-out overlaps this group's copies and passes
                prev = slot
            if rank == 0:
                fetch(prev)

        esteps = max(1, min(args.steps, 2))
        e2e_light_cone()  # warm-up
        e.synchronize()
        barrier = (lambda: dist.barrier()) if world > 1 else (lambda: None)
        barrier()
        e.synchronize()
        w0 = time.perf_counter()
        e.timer_begin()
        for _ in range(esteps):
            e2e_light_cone()
        e.synchronize()
        ems = e.timer_end()
        wall_ms = (time.perf_counter() - w0) * 1e3
        ems = max(ems, wall_ms)  # the host wall clock includes the synchronous fetches
        if world > 1:
            t = torch.tensor([ems], dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ems = float(t[0])
        npass = esteps * W["ngroups"]
        e2e = {"value": wl.total * npass / (ems * 1e-3), "unit": UNIT, "h2d_bytes_per_step": 12 * wl.total * W["ngroups"],
               "d2h_bytes_per_step": (LENS_PER_SNAP * W["npix"] * W["npix"] * 4 + 48) * W["ngroups"], "ms_per_step": ems / esteps,
               "steps": esteps,
               "api": "slicer_begin_snapshot/next_batch/stage_particles(pinned)/deposit_slots/reduce_slots/fetch, "
                      f"{nb} sub-file batches per snapshot, 2 staging pools, {W['ngroups']} snapshots per step"}
        launches_e2e = int(e.stats().launches)
        e.close()
        pin.free()
    else:
        launches_e2e = None
        wl.close()

    # ------------------------------------------------------------------ the other stated configurations, a few steps each
    also = {}
    for spec in [a for a in args.also.split(",") if a]:
        name, _, sc = spec.partition(":")
        sc = sc or "strong"
        if name == args.workload and sc == args.scaling:
            continue
        try:
            r2, w2 = measure(args, name, sc, max(1, min(args.steps, 3)), min(args.warmup, 1), rank, world, local_rank, dist, False,
                             verify=(world > 1))  # (N > 1: every configuration's reduced planes are checked, the 2 GiB of C5 included)
            w2.close()
            r2["roofline"] = roofline_of(r2, peaks)
            for k in ("clocks", "ms"):
                r2.pop(k, None)
            also[f"{name}:{sc}"] = r2
        except Exception as ex:  # e.g. not enough device memory for that configuration at this N
            also[f"{name}:{sc}"] = {"error": str(ex)[:300]}

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        from oracle import ref_bindings

        if ref_bindings.available():
            with tempfile.TemporaryDirectory() as td:
                n = 1 << 21
                v, wall, _ = run_reference_sample(1, n, list(range(W["ngroups"])), wl.raw, td, W)
            cpu = {"value": v, "unit": UNIT, "cores": 1, "kind": "reference",
                   "sample": f"reference createDensityMaps (oracle/_ref) on a {n}-particle sub-file of the same synthetic snapshot, "
                             f"all {LENS_PER_SNAP * W['ngroups']} planes of the {W['ngroups']} groups ({wall:.1f} s)"}
    if rank == 0:
        line = {
            "metric": METRIC, "value": res["value"], "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": res["ms_per_step"], "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
            "dtype": "f32+f64->int64", "data": "synthetic", "config": workload_config(args.workload, args.scaling, world),
            "roofline": roofline, "cpu_baseline": cpu, "e2e": e2e, "gpu_launches": res["launches"], "clocks": res["clocks"],
            "extra": {"per_group_kernel_ms": res["per_group_ms"], "ms_per_pass": res["ms_per_pass"], "kernel_ms_avg": res["kernel_ms"],
                      "stream_rate_particles_per_s": res["value"], "ref_equiv_particle_passes_per_s": res["value"] * LENS_PER_SNAP,
                      "flagged_pairs_settled_with_libm": res["flagged_pairs"], "verify": res.get("verify"), "reduce_ok": res.get("reduce_ok"),
                      "gpu_launches_e2e": launches_e2e, "csrc_sha": csrc_sha(), "also": also},
        }
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def _download_all(wl, pin):
    """Copy the resident segments of `wl` into the pinned buffer, in staging order."""
    from slicer_b200 import capi

    off = 0
    for seg, m in enumerate(wl.segments):
        capi._check(capi.lib().slicer_download_segment(wl.s.h, seg, ctypes.c_void_p(pin.ptr + off * 12), None))
        off += m


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c3", choices=sorted(WORKLOADS))
    ap.add_argument("--scaling", default="strong", choices=["strong", "weak"])
    ap.add_argument("--also", default=None, help="other configurations measured for a few steps in the same run and reported under "
                    "extra.also, e.g. 'c5,c4,c3:weak'; default: c5,c4 (plus c3:weak at N > 1); '' for none")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-verify", action="store_true")
    ap.add_argument("--deposit-mode", type=int, default=0, help="0 auto, 1 direct map atomics, 2 binned shared-memory tiles")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the planes of every group of the last step (maps, map sums, counts, in-grid "
                         "counts) as DIR/*.npy, < 64 MB in all: maps as one fixed, seeded sample of pixels where they are larger; "
                         "the groups the step overwrote are deposited again, outside the timed region")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the planes of the GPU path (--impl ours)")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
    os.environ.setdefault("MASTER_PORT", "29511")
    if world != args.gpus and world == 1 and args.gpus > 1:
        # convenience: re-launch under torchrun
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}", "--master-addr", "127.0.0.1",
               "--master-port", os.environ["MASTER_PORT"], os.path.abspath(__file__)] + sys.argv[1:]
        raise SystemExit(subprocess.call(cmd))
    if args.also is None:
        args.also = "c5,c4" + (",c3:weak" if world > 1 else "")
        if args.workload != "c3":
            args.also = ""
    if args.impl == "reference":
        reference_arm(args, rank, world)
    else:
        ours(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
