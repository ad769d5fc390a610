"""Every variant of the pipelined record kernel, and the simple kernel, against the oracle at its decision boundaries, in every box
orientation.

`deposit_pipelined_kernel` is compiled once per entry of `pipelined_table` (csrc/deposit_pipelined.cuh): mass assignment (TSC,
NGP) x layout (AoS, SoA) x one randomisation or several x exact phase (GENERIC, FAST, EMIT, FAST_LEAN, EMIT_LEAN), 32 kernels
in 40 slots (NGP has no record kernels: a binned NGP pass runs the TSC record kernel and the tile kernel applies NGP).  Which one a pass runs
follows from `build_pass` (`fast`, `lean`), `use_binned` and `pipelined_path` in csrc/slicer_capi.cu; `plan` below restates those
rules.  Every row of the matrix (a) is put by `plan` in the cell it is meant for, for the reason it names, (b) runs exactly that
kernel (`Slicer.kernels_run`, include/slicer_b200.h: slicer_kernels_run) and (c) equals the oracle on every plane: accepted and
in-grid counts and int64 maps bit for bit, float maps within the bars of test_gpu_parity, every particle type.

The particles of a pass are about 100k uniform ones plus
  * sweeps of consecutive float32 raw coordinates across each decision of each plane, placed by inverting the plane's
    randomisation (face permutation, signs, centre, pile offset): the slab edges (the first slab of every randomisation starts
    exactly at rcase, so its lower edge is also the wrap of z at the centre), the field edges in ra and dec at mid-depth, the
    pixel edge at the map centre and the outer map border;
  * raw coordinates on and around the box faces: 0, the smallest denormal, 2^-40 (the lean transform's lower bound), raw_hi,
    the box size and just above it, with the other two coordinates inside the field and the slab;
  * for the planes at the observer (rcase 0, ld 0): particles exactly at the observer and on the plane z = 0.
Type 1 carries a constant mass, type 4 per-particle masses (a run of consecutive floats around MAX_M among them).
"""
import functools
import math
import os
import subprocess
import sys

import numpy as np
import pytest

from oracle.oracle_bindings import MAX_M
from slicer_b200 import capi, synth
from test_gpu_parity import check_against_oracle

# ---- the selection rules, restated (csrc/slicer_capi.cu: build_pass, use_binned, run_pass; csrc/lean_math.h: lean_setup;
# csrc/deposit_pipelined.cuh: pipelined_path, pipelined_index) --------------------------------------------------------------
PATHS = ("GENERIC", "FAST", "EMIT", "FAST_LEAN", "EMIT_LEAN")
NPATHS = len(PATHS)
VARIANTS = 2 * 2 * 2 * NPATHS                                 # PIPELINED_VARIANTS; bit VARIANTS + mas: deposit_simple_kernel
PERM = {1: (0, 1, 2), 2: (0, 2, 1), 3: (1, 2, 0), 4: (1, 0, 2), 5: (2, 0, 1), 6: (2, 1, 0)}  # raw axis feeding output axis k
LEAN_UMIN = 2.0 ** -40                                        # LeanDev::umin
MAS_OF = {"tsc": capi.MAS_TSC, "ngp": capi.MAS_NGP}
LAYOUT_OF = {"aos": capi.LAYOUT_AOS, "soa": capi.LAYOUT_SOA}


def f32(v):
    return float(np.float32(v))


def float_ceil(d):
    f = np.float32(d)
    return float(np.nextafter(f, np.float32(np.inf)) if float(f) < d else f)


def float_floor(d):
    f = np.float32(d)
    return float(np.nextafter(f, np.float32(-np.inf)) if float(f) > d else f)


def variant_index(mas, layout, single, path):
    return ((mas * 2 + layout) * 2 + (1 if single else 0)) * NPATHS + PATHS.index(path)


def nonempty_variants():
    return {i for i in range(VARIANTS) if not (i // (4 * NPATHS) == capi.MAS_NGP and PATHS[i % NPATHS] in ("EMIT", "EMIT_LEAN"))}


def plane_consts(p, box):
    """build_pass: slab edges (float), half field T and the terms of the general chain's small-angle series (0: libdevice)."""
    zlo, zhi = float_ceil(p["ld"] / box * 1.e+3 / 1.0), float_ceil(p["ld2"] / box * 1.e+3 / 1.0)
    T = p["fovradiants"] * (1. + 2. / p["npix"]) * 0.5
    nt = 0
    if T < 1.5:
        pre_tx = float_ceil(math.tan(T) * (1.0 + 1e-5) / math.cos(T))
        if pre_tx * 1.01 <= 0.385:
            nt = max(2, math.ceil(55.0 * math.log(2.0) / (2.0 * math.log(1.0 / (pre_tx * 1.01)))))
            nt = 0 if nt > 20 else nt
    return dict(zlo=zlo, zhi=zhi, T=T, nt=nt)


def lean_terms(fov, T):
    """lean_setup: K, the series terms of the lean projection (0: the field is too wide for it)."""
    if not (T < 1.5 and fov > 0):
        return 0
    arg_lim = math.tan(T) * (1.0 + 1e-5) / math.cos(T) * 1.01
    if not arg_lim <= 0.385:
        return 0
    a = [1.0]
    for k in range(1, 22):
        a.append(a[-1] * (2 * k - 1) ** 2 / (2 * k * (2 * k + 1)))
    z = arg_lim * arg_lim
    for k in range(2, 21):
        if a[k + 1] * z ** (k + 1) / (1.0 - z) <= 2.0 ** -53 and z ** (k + 1) / (2.0 * k + 3.0) <= 2.0 ** -53:
            return k
    return 0


def xform_key(p):
    return (tuple(p["sgn"]), p["face"], tuple(p["centre"]), f32(p["rcase"]))


def plan(box, planes, kernel, mode, mas, layout):
    """-> the kernel a pass runs: path, mask bit, and the quantities the choice depends on."""
    keys = list(dict.fromkeys(xform_key(p) for p in planes))
    C = [plane_consts(p, box) for p in planes]
    if kernel == capi.KERNEL_SIMPLE:
        return dict(path="SIMPLE", bit=VARIANTS + mas, nx=len(keys), fast=None, lean=None, K=0, nt=C[0]["nt"])
    assert mode in (capi.DEPOSIT_DIRECT, capi.DEPOSIT_BINNED)  # (DEPOSIT_AUTO's estimate is not restated)
    fast = True
    for key in keys:
        grp = [i for i, p in enumerate(planes) if xform_key(p) == key]
        for a in grp:
            n = planes[a]["npix"]
            fast &= n & (n - 1) == 0 and planes[a]["nrepperp"] == 0
            for b in grp:
                if b > a and C[a]["zlo"] < C[b]["zhi"] and C[b]["zlo"] < C[a]["zhi"]:
                    fast = False  # overlapping slabs
    exact = f32(box) == box and all(f32(c) == c for p in planes for c in p["centre"])
    same = all((C[q]["T"], p["fovradiants"], p["npix"]) == (C[0]["T"], planes[0]["fovradiants"], planes[0]["npix"])
               for q, p in enumerate(planes))
    lean = fast and C[0]["nt"] > 0 and 2.0 ** -40 <= box <= 2.0 ** 40 and exact and same
    K = lean_terms(planes[0]["fovradiants"], C[0]["T"]) if lean else 0
    lean = lean and K > 0 and float_floor(box * (1.0 - 1e-6)) > LEAN_UMIN and \
        all(0.0 <= f32(c) <= 1.0 for p in planes for c in p["centre"])
    # use_binned under DEPOSIT_BINNED: a fast pass, one map size (maps of <= 256^2 stay far below the 16-bit record keys)
    binned = mode == capi.DEPOSIT_BINNED and fast and len({p["npix"] for p in planes}) == 1
    path = ("EMIT_LEAN" if lean else "EMIT") if binned else "GENERIC" if not fast else ("FAST_LEAN" if lean else "FAST")
    bit = variant_index(capi.MAS_TSC if binned else mas, layout, len(keys) == 1, path)
    return dict(path=path, bit=bit, nx=len(keys), fast=fast, lean=lean, K=K, nt=C[0]["nt"])


# ---- the rows ---------------------------------------------------------------------------------------------------------
# What sends a row to its path (the reason), and the field it uses:
#   fov5 / fov0.6   lean: 5 degrees (series of K <= 6 terms, the unrolled Horner scheme) / 0.6 rad (K > 6, the loop)
#   box             the box size is not a float (123456.789)                      -> not lean
#   centre          a centre coordinate is not a float (0.1)                      -> not lean
#   fov0.9          the general chain's series does not reach (nt = 0)            -> not lean
#   mixed           planes of 256^2 and 128^2 (direct passes only: not binned)    -> not lean
#   npix333 / nrep1 / overlap, each -narrow (series, nt > 0) or -wide (libdevice, nt = 0)   -> not fast: GENERIC
FIELDS = {"fov5": (float(np.float32(5.0)) / 180.0 * np.pi, (2, 3)), "fov0.6": (0.6, (0, 1)), "box": (0.3, (1, 2)),
          "centre": (0.3, (1, 2)), "fov0.9": (0.9, (0,)), "mixed": (0.3, (1,)), "narrow": (0.2, (2, 3)), "wide": (1.2, (0,))}
LEAN_WIDE_FOV = 0.65  # the widest lean field of the listed ones at 256^2 (0.7 rad is not lean)

# (mas, layout, randomisations, planes per randomisation, path, reason)
ROWS = [
    ("tsc", "aos", 1, 16, "FAST_LEAN", "fov5"), ("tsc", "soa", 1, 6, "FAST_LEAN", "fov0.6"),
    ("ngp", "aos", 1, 4, "FAST_LEAN", "fov0.6"), ("ngp", "soa", 1, 1, "FAST_LEAN", "fov5"),
    ("tsc", "aos", 3, 3, "FAST_LEAN", "fov0.6"), ("tsc", "soa", 8, 2, "FAST_LEAN", "fov5"),
    ("ngp", "aos", 3, 3, "FAST_LEAN", "fov5"), ("ngp", "soa", 3, 3, "FAST_LEAN", "fov0.6"),

    ("tsc", "aos", 1, 6, "EMIT_LEAN", "fov0.6"), ("tsc", "soa", 1, 16, "EMIT_LEAN", "fov5"),
    ("ngp", "aos", 1, 1, "EMIT_LEAN", "fov5"), ("ngp", "soa", 1, 4, "EMIT_LEAN", "fov0.6"),
    ("tsc", "aos", 8, 2, "EMIT_LEAN", "fov5"), ("tsc", "soa", 3, 3, "EMIT_LEAN", "fov0.6"),
    ("ngp", "aos", 3, 3, "EMIT_LEAN", "fov0.6"), ("ngp", "soa", 3, 3, "EMIT_LEAN", "fov5"),

    ("tsc", "aos", 1, 4, "FAST", "box"), ("tsc", "soa", 1, 1, "FAST", "centre"),
    ("ngp", "aos", 1, 16, "FAST", "fov0.9"), ("ngp", "soa", 1, 6, "FAST", "mixed"),
    ("tsc", "aos", 3, 3, "FAST", "mixed"), ("tsc", "soa", 3, 3, "FAST", "fov0.9"),
    ("ngp", "aos", 8, 2, "FAST", "centre"), ("ngp", "soa", 3, 3, "FAST", "box"),

    ("tsc", "aos", 1, 1, "EMIT", "fov0.9"), ("tsc", "soa", 1, 4, "EMIT", "box"),
    ("ngp", "aos", 1, 6, "EMIT", "centre"), ("ngp", "soa", 1, 16, "EMIT", "fov0.9"),
    ("tsc", "aos", 3, 3, "EMIT", "centre"), ("tsc", "soa", 3, 3, "EMIT", "box"),
    ("ngp", "aos", 3, 3, "EMIT", "box"), ("ngp", "soa", 8, 2, "EMIT", "centre"),

    ("tsc", "aos", 1, 1, "GENERIC", "npix333-narrow"), ("tsc", "soa", 1, 16, "GENERIC", "overlap-wide"),
    ("ngp", "aos", 1, 6, "GENERIC", "nrep1-narrow"), ("ngp", "soa", 1, 4, "GENERIC", "npix333-wide"),
    ("tsc", "aos", 3, 3, "GENERIC", "nrep1-wide"), ("tsc", "soa", 3, 3, "GENERIC", "overlap-narrow"),
    ("ngp", "aos", 8, 2, "GENERIC", "overlap-wide"), ("ngp", "soa", 3, 3, "GENERIC", "npix333-narrow"),

    ("tsc", "aos", 3, 3, "SIMPLE", "nrep1-narrow"), ("ngp", "soa", 3, 3, "SIMPLE", "npix333-wide"),
]
ROW_IDS = [f"{i:02d}-{m}-{l}-x{nx}p{npl}-{path}-{why}" for i, (m, l, nx, npl, path, why) in enumerate(ROWS)]
SGNS = [(-1, 1, 1), (1, -1, 1), (1, 1, -1), (-1, -1, 1), (-1, 1, -1), (1, -1, -1), (-1, -1, -1)]
MASS1 = 1.5  # type 1 (massarr); type 4 carries per-particle masses
N_UNIFORM = (60000, 40000)
K_SWEEP = 200


def consecutive(v, k, stride=1):
    """2k+1 consecutive float32 values around float32(v) (every stride-th with stride > 1), without negative ones (the
    reference aborts on those)."""
    i = int(np.array(v, np.float32).view(np.int32))
    out = (i + stride * np.arange(-k, k + 1, dtype=np.int64)).astype(np.int32).view(np.float32)
    return out[np.isfinite(out) & ~np.signbit(out)]


def exact_ld(z, box):
    """ld (Mpc/h) whose minDist = ld / box * 1e3 is exactly z."""
    ld = z * box / 1e3
    for _ in range(64):
        d = ld / box * 1.e+3
        if d == z:
            return ld
        ld = np.nextafter(ld, np.inf if d < z else -np.inf)
    raise AssertionError(f"no ld gives minDist == {z}")


def row_geometry(i):
    """-> box, planes (dicts the oracle and plane_desc take, with npix), kernel, deposit mode, mas, layout, per-type maps."""
    mas, layout, nx, npl, path, why = ROWS[i]
    rng = np.random.default_rng(7000 + i)
    base = why.split("-")[-1] if "-" in why else why
    fov, rcases = FIELDS[base]
    rcase = float(rcases[i % len(rcases)])
    box = 123456.789 if why == "box" else 128000.0
    T = fov * (1 + 2.0 / 256) * 0.5
    depth = min(0.95, 0.45 / math.tan(T) - rcase)  # the field edges of every slab stay inside the box's cross-section
    assert depth > 0.2, (i, depth)
    planes = []
    for t in range(nx):
        face = (i + t) % 6 + 1
        rot = [SGNS[(i + 3 * t + j) % len(SGNS)] for j in range(len(SGNS))]
        # one randomisation: output x and y of opposite signs, so that the two lanes of the packed box transform differ
        sgn = next(s for s in rot if s[PERM[face][0]] != s[PERM[face][1]]) if nx == 1 else rot[0]
        centre = [f32(c) for c in rng.uniform(0.05, 0.95, 3)]
        if rcase == 0.0:  # multiples of 2^-12: box * centre is a float, so a particle can sit exactly at the observer
            centre = [float(c) / 4096 for c in rng.integers(205, 3892, 3)]
        if why == "centre" and t == 0:
            centre[1] = 0.1
        edges = [rcase + depth * k / npl for k in range(npl + 1)]
        for k in range(npl):
            lo, hi = edges[k], edges[min(k + 2, npl)] if why.startswith("overlap") else edges[k + 1]
            if why.startswith("overlap") and k == npl - 1 and npl > 1:
                lo = edges[k - 1] + 0.5 * (edges[k] - edges[k - 1])  # the last slab overlaps the one before it too
            npix = 333 if why.startswith("npix333") else (128 if why == "mixed" and k % 2 else 256)
            planes.append(dict(boxsize=box, sgn=list(sgn), face=face, centre=centre, rcase=rcase,
                               ld=exact_ld(lo, box) if k == 0 else lo * box / 1e3, ld2=hi * box / 1e3,
                               nrepperp=1 if why.startswith("nrep1") else 0, fovradiants=fov, npix=npix))
    kernel = capi.KERNEL_SIMPLE if path == "SIMPLE" else capi.KERNEL_PIPELINED
    mode = capi.DEPOSIT_BINNED if path.startswith("EMIT") else capi.DEPOSIT_DIRECT
    return dict(box=box, planes=planes, kernel=kernel, mode=mode, mas=MAS_OF[mas], layout=LAYOUT_OF[layout], per_type=i % 2 == 0)


# ---- particles: sweeps placed by inverting a randomisation -------------------------------------------------------------
def invert(v, p, box):
    """Raw float32 coordinates whose transform under p's randomisation is ~v = (x, y, z) (z with rcase): output axis k is fed
    by raw axis perm[k]; b = (v_k + c_k) mod 1, raw = box b (sgn > 0) or box (1 - b) (sgn < 0)."""
    raw = np.empty(3)
    for k, a in enumerate(PERM[p["face"]]):
        b = ((v[k] - (p["rcase"] if k == 2 else 0.0)) + p["centre"][k]) % 1.0
        raw[a] = box * b if p["sgn"][a] > 0 else box * (1.0 - b)
    return raw.astype(np.float32)


def transform(oracle, pos, p, box):
    return oracle.transform(pos, box, p["sgn"], p["face"], p["centre"], p["rcase"])


def snap(oracle, raw, k, target, p, box):
    """Move the raw coordinate feeding output axis k to the float whose transform is closest to target (exact when one is)."""
    a = PERM[p["face"]][k]
    cand = consecutive(raw[a], 64)
    pos = np.tile(raw, (len(cand), 1))
    pos[:, a] = cand
    out = transform(oracle, pos, p, box)[k].astype(np.float64)
    raw = raw.copy()
    raw[a] = cand[int(np.argmin(np.abs(out - target)))]
    return raw


def sweep(oracle, v, k, p, box, kk=K_SWEEP):
    """Consecutive raw floats along the raw axis feeding output axis k, across output value v[k]; the other two output
    coordinates at v exactly where a float lands there.  Where the raw floats are much finer than the output's (a small raw
    coordinate, or z beside a large rcase), a strided run across some 50 output floats is added."""
    raw = invert(v, p, box)
    for j in range(3):
        if j != k:
            raw = snap(oracle, raw, j, v[j], p, box)
    a = PERM[p["face"]][k]
    vals = consecutive(raw[a], kk)
    stride = int(np.spacing(np.float32(v[k])) / (np.spacing(raw[a]) / box) / 2)
    if stride > 1:
        vals = np.union1d(vals, consecutive(raw[a], kk // 2, stride))
    pos = np.tile(raw, (len(vals), 1))
    pos[:, a] = vals
    return pos


def plane_sweeps(oracle, p, box, first):
    """[(label, positions)] across every decision of plane p (first: the first plane of its randomisation)."""
    c = plane_consts(p, box)
    lo, hi = p["ld"] / box * 1e3, p["ld2"] / box * 1e3
    zmid = 0.5 * (lo + hi)
    out = [("slab-lo" if not first else "slab-lo=z-wrap", sweep(oracle, (0.5, 0.5, lo), 2, p, box)),
           ("slab-hi", sweep(oracle, (0.5, 0.5, hi), 2, p, box))]
    edges = [("ra", 1, s * zmid * math.tan(c["T"])) for s in (-1, 1)] + [("dec", 0, s * zmid * math.tan(c["T"])) for s in (-1, 1)]
    centre = (p["npix"] // 2 / p["npix"] - 0.5) * p["fovradiants"]  # the pixel edge at (or next to) the map centre
    edges += [("pixel-centre", 0, zmid * math.tan(centre)), ("pixel-border-x", 0, zmid * math.tan(0.5 * p["fovradiants"])),
              ("pixel-border-y", 1, -zmid * math.tan(0.5 * p["fovradiants"]))]
    for label, k, off in edges:
        if abs(off) < 0.47:
            v = [0.5, 0.5, zmid]
            v[k] = 0.5 + off
            out.append((label, sweep(oracle, v, k, p, box)))
    return out


def face_values(box):
    B = np.float32(box)
    raw_hi = float_floor(box * (1.0 - 1e-6))
    vals = [np.float32(0.0), np.float32(np.finfo(np.float32).smallest_subnormal)]
    for v in (LEAN_UMIN, raw_hi, B):
        vals += list(consecutive(v, 6))
    vals += [np.float32(B * np.float32(1.0 + 2.0 ** -12)), np.float32(B * np.float32(1.25))]
    return np.array(vals, np.float32)


def face_particles(oracle, p, box):
    """Each raw axis on and around the box faces, the other two inside the field at the middle of plane p's slab."""
    zmid = 0.5 * (p["ld"] + p["ld2"]) / box * 1e3
    raw = invert((0.5, 0.5, zmid), p, box)
    for k in range(3):
        raw = snap(oracle, raw, k, (0.5, 0.5, zmid)[k], p, box)
    vals = face_values(box)
    rows = []
    for a in range(3):
        pos = np.tile(raw, (len(vals), 1))
        pos[:, a] = vals
        rows.append(pos)
    return np.concatenate(rows)


def observer_particles(oracle, p, box):
    """Plane at rcase 0 with ld 0: particles exactly at the observer and on the plane z = 0 (x, y off the axis)."""
    rows = []
    for v in ((0.5, 0.5, 0.0), (0.5 + 2.0 ** -10, 0.5, 0.0), (0.5, 0.5 - 2.0 ** -12, 0.0), (0.25, 0.75, 0.0)):
        raw = invert(v, p, box)
        for k in range(3):
            raw = snap(oracle, raw, k, v[k], p, box)
        rows.append(raw[None])
    return np.concatenate(rows)


@functools.lru_cache(maxsize=None)
def row_inputs(i):
    """-> geometry, the two segments [(type, positions, masses or None)], and the labelled sweeps of the row."""
    from oracle.oracle_bindings import Oracle
    oracle = Oracle()
    g = row_geometry(i)
    box, planes = g["box"], g["planes"]
    sweeps, extra = [], []
    seen = set()
    for q, p in enumerate(planes):
        key = xform_key(p)
        first = key not in seen
        seen.add(key)
        sweeps += [(f"plane {q} {label}", pos) for label, pos in plane_sweeps(oracle, p, box, first)]
        if first:
            extra.append(face_particles(oracle, p, box))
            if p["rcase"] == 0.0 and p["ld"] == 0.0:
                extra.append(observer_particles(oracle, p, box))
    special = np.concatenate([pos for _, pos in sweeps] + extra).astype(np.float32)
    u1 = synth.uniform_positions(N_UNIFORM[0], box, 100 + i)
    u4 = synth.uniform_positions(N_UNIFORM[1], box, 200 + i)
    rng = np.random.default_rng(300 + i)
    m_uniform = (0.05 + 2.0 * rng.random(len(u4))).astype(np.float32)
    # every 16th: the next of the consecutive floats around MAX_M (either side of the cut); sparse, so that the mass of a plane stays
    # within the 2^(63 - 40) units the mass-conservation check can sum in int64
    m_special = (0.05 + 2.0 * rng.random(len(special))).astype(np.float32)
    m_special[::16] = consecutive(MAX_M, 40)[np.arange(len(m_special[::16])) % 81]
    segs = [(1, np.concatenate([u1, special]), None), (4, np.concatenate([u4, special]), np.concatenate([m_uniform, m_special]))]
    return g, segs, sweeps


def oracle_types(segs):
    return [dict(type=ty, raw=pos, const_mass=MASS1) if m is None else dict(type=ty, raw=pos, masses=m, cut=True) for ty, pos, m in segs]


# ---- CPU: the planner, the coverage and the sweeps ----------------------------------------------------------------------
@pytest.mark.parametrize("i", range(len(ROWS)), ids=ROW_IDS)
def test_planner_puts_row_in_its_cell(i):
    mas, layout, nx, npl, path, why = ROWS[i]
    g = row_geometry(i)
    pl = plan(g["box"], g["planes"], g["kernel"], g["mode"], g["mas"], g["layout"])
    assert pl["path"] == path and pl["nx"] == nx, pl
    assert len(g["planes"]) == nx * npl
    assert all(-1 in p["sgn"] for p in g["planes"])
    assert all(0.0 < f32(c) < 1.0 for p in g["planes"] for c in p["centre"])
    assert all(plane_consts(p, g["box"])["zlo"] == p["rcase"] for p in g["planes"][::npl])  # first slab starts at rcase
    # the reason the row names is what decides
    if why == "fov5":
        assert 0 < pl["K"] <= 6
    if why == "fov0.6":
        assert pl["K"] > 6
    if why in ("box", "centre", "mixed") or why.endswith("narrow"):
        assert pl["nt"] > 0
    if why == "fov0.9" or why.endswith("wide"):
        assert pl["nt"] == 0
    if why == "mixed":
        assert g["mode"] == capi.DEPOSIT_DIRECT and len({p["npix"] for p in g["planes"]}) == 2
    if path in ("FAST", "EMIT"):  # the same pass with the reason removed would be lean
        fixed = [dict(p, centre=[f32(c) for c in p["centre"]], fovradiants=0.3, npix=256) for p in g["planes"]]
        assert plan(128000.0, fixed, g["kernel"], g["mode"], g["mas"], g["layout"])["lean"]


def test_planner_reasons():
    """The field-width limits the rows rely on: 0.65 rad is the widest lean field at 256^2, 0.7 rad is not."""
    def lean(fov):
        p = dict(sgn=[1, 1, -1], face=1, centre=[0.5, 0.5, 0.5], rcase=0.0, ld=0.0, ld2=64.0, nrepperp=0, fovradiants=fov, npix=256)
        return plan(128000.0, [p], capi.KERNEL_PIPELINED, capi.DEPOSIT_DIRECT, 0, 0)["lean"]
    assert lean(LEAN_WIDE_FOV) and not lean(0.7)


def test_rows_cover_every_variant():
    """The rows' kernels, together: every non-empty entry of pipelined_table (32 of 40: no NGP record kernels for either layout or
    randomisation count) and the simple kernel for TSC and NGP."""
    bits = set()
    reasons = {}
    for i, (mas, layout, nx, npl, path, why) in enumerate(ROWS):
        g = row_geometry(i)
        bits.add(plan(g["box"], g["planes"], g["kernel"], g["mode"], g["mas"], g["layout"])["bit"])
        reasons.setdefault(path, set()).add(why)
    assert len(nonempty_variants()) == 32
    assert bits == nonempty_variants() | {VARIANTS + capi.MAS_TSC, VARIANTS + capi.MAS_NGP}
    assert reasons["FAST_LEAN"] == reasons["EMIT_LEAN"] == {"fov5", "fov0.6"}
    assert reasons["FAST"] == {"box", "centre", "fov0.9", "mixed"} and reasons["EMIT"] == {"box", "centre", "fov0.9"}
    assert {w.split("-")[0] for w in reasons["GENERIC"]} == {"npix333", "nrep1", "overlap"}
    assert {w.split("-")[1] for w in reasons["GENERIC"]} == {"narrow", "wide"}
    single = {npl for (_, _, nx, npl, path, _) in ROWS if nx == 1 and path == "FAST_LEAN"}
    assert single == {1, 4, 6, 16}  # fixed slab tests, the > 4 loop, both words of count_round and its loop beyond 8
    assert {(nx, npl) for (_, _, nx, npl, _, _) in ROWS if nx > 1} == {(3, 3), (8, 2)}
    assert {ROWS[i][0:2] for i in range(len(ROWS))} == {(m, l) for m in MAS_OF for l in LAYOUT_OF}
    assert {row_geometry(i)["planes"][0]["rcase"] for i in range(len(ROWS))} == {0.0, 1.0, 2.0, 3.0}
    assert {p["face"] for i in range(len(ROWS)) for p in row_geometry(i)["planes"]} == set(range(1, 7))


def test_inversion_matches_the_oracle_transform(oracle):
    """invert() against orc_transform for every face and several sign patterns: a sweep placed around an output value lands
    on both sides of it."""
    box = 128000.0
    for face in range(1, 7):
        for sgn in SGNS:
            p = dict(sgn=list(sgn), face=face, centre=[f32(0.3), f32(0.71), f32(0.6)], rcase=1.0)
            for k in range(3):
                for target in (0.2371, 0.5, 0.8123):
                    v = [0.5, 0.5, 1.5]
                    v[k] = target + (1.0 if k == 2 else 0.0)
                    pos = sweep(oracle, v, k, p, box)
                    out = transform(oracle, pos, p, box)
                    assert np.all(np.abs(out[k] - v[k]) < 1e-4), (face, sgn, k)
                    assert np.count_nonzero(out[k] < v[k]) > 0 and np.count_nonzero(out[k] > v[k]) > 0, (face, sgn, k)
                    for j in range(3):
                        if j != k:
                            assert np.all(out[j] == np.float32(v[j])), (face, sgn, k, j)


def decisions(oracle, pos, planes, box):
    """Per particle: the (plane, NGP cell) pairs the oracle accepts it into, over every plane of the pass."""
    idx = (np.arange(len(pos)) + 1).astype(np.float32)  # carried through as a mass (no MAX_M cut): which particle a pair is
    sig = [[] for _ in range(len(pos))]
    for q, p in enumerate(planes):
        x, y, z = transform(oracle, pos, p, box)
        xs, ys, ms = oracle.select_project(x, y, z, p["ld"], p["ld2"], box, p["nrepperp"], p["fovradiants"], p["npix"],
                                           per_particle=idx, max_m=-1.0, cap=9 * len(pos) + 16)
        for j, cell in zip(ms.astype(np.int64) - 1, oracle.ngp_cells_fast(xs, ys, p["npix"])):
            sig[j].append((q, int(cell)))
    return [tuple(s) for s in sig]


@pytest.mark.parametrize("i", range(len(ROWS)), ids=ROW_IDS)
def test_sweeps_straddle_their_decisions(oracle, i):
    """For the oracle alone, every sweep of the row crosses its decision: some of its particles are accepted and some not, or
    they land in different planes or pixels.  The observer particles of the planes at ld = 0 sit exactly at (0.5, 0.5, 0)."""
    g, segs, sweeps = row_inputs(i)
    assert len(sweeps) >= 4 * len(g["planes"])
    assert any("ra" in lab for lab, _ in sweeps) and any("dec" in lab for lab, _ in sweeps)
    for label, pos in sweeps:
        assert len(set(decisions(oracle, pos, g["planes"], g["box"]))) >= 2, label
    p = g["planes"][0]
    if p["rcase"] == 0.0:
        x, y, z = transform(oracle, segs[0][1], p, g["box"])
        assert np.any((x == 0.5) & (y == 0.5) & (z == 0.0)) and np.count_nonzero(z == 0.0) >= 4
    assert len(segs[0][1]) + len(segs[1][1]) >= 100000


# ---- GPU: every row against the oracle ----------------------------------------------------------------------------------
def run_row(i):
    g, segs, _ = row_inputs(i)
    planes = g["planes"]
    npix_max = max(p["npix"] for p in planes)
    n = sum(len(pos) for _, pos, _ in segs) + 64
    descs = [capi.plane_desc(p["sgn"], p["face"], p["centre"], p["rcase"], p["ld"], p["ld2"], p["fovradiants"], p["npix"], p["nrepperp"])
             for p in planes]
    out = []
    with capi.Slicer(npix_max=npix_max, max_planes=len(planes), mas=g["mas"], particle_capacity=n, mass_capacity=n,
                     per_type_maps=g["per_type"], kernel=g["kernel"], deposit_mode=g["mode"]) as s:
        s.begin_snapshot(g["box"], [0, MASS1, 0, 0, 0, 0], True)
        for ty, pos, m in segs:
            s.stage(ty, pos if g["layout"] == capi.LAYOUT_AOS else np.ascontiguousarray(pos.T), m, layout=g["layout"])
        assert s.kernels_run() == 0
        s.deposit(descs)
        mask = s.kernels_run()
        for k, p in enumerate(planes):
            npix = p["npix"]
            _, counts, ingrid = s.fetch(k, -1, npix, want_map=False)
            got = dict(counts=counts, ingrid=ingrid, frac_bits=s.frac_bits, maps={}, fixed={})
            for ty in ((1, 4) if g["per_type"] else (-1,)):
                got["maps"][ty] = s.fetch(k, ty, npix)[0].reshape(-1)
                got["fixed"][ty] = s.fetch_fixed(k, ty, npix).reshape(-1)
            out.append(got)
        s.reset_stats()
        assert s.kernels_run() == 0
    return mask, out


@pytest.mark.gpu
@pytest.mark.parametrize("i", range(len(ROWS)), ids=ROW_IDS)
def test_variant_matrix(oracle, i):
    g, segs, _ = row_inputs(i)
    pl = plan(g["box"], g["planes"], g["kernel"], g["mode"], g["mas"], g["layout"])
    assert pl["path"] == ROWS[i][4]
    mask, got = run_row(i)
    assert mask == 1 << pl["bit"], (hex(mask), pl)
    types = oracle_types(segs)
    do_ngp = g["mas"] == capi.MAS_NGP
    for k, p in enumerate(g["planes"]):
        try:
            if g["per_type"]:
                res = check_against_oracle(oracle, types, p, p["npix"], got[k], do_ngp, MAX_M, strict_float=False)
            else:
                res = oracle.plane_from_particles(types, p, p["npix"], do_ngp=do_ngp, frac_bits=got[k]["frac_bits"])
                assert got[k]["counts"].tolist() == res["counts"].tolist()
                assert got[k]["ingrid"].tolist() == res["ingrid"].tolist()
                want = res["fixed"].sum(0)
                if not np.array_equal(got[k]["fixed"][-1], want):
                    bad = np.flatnonzero(got[k]["fixed"][-1] != want)
                    pytest.fail(f"{len(bad)} cells differ, first (gy, gx) = {divmod(int(bad[0]), p['npix'])}")
                np.testing.assert_allclose(got[k]["maps"][-1], res["f64"].sum(0), rtol=1e-6, atol=1e-9 * MAX_M)
        except AssertionError as e:
            raise AssertionError(f"plane {k} ({p}): {e}") from None
        assert res["counts"][1] > 0 and res["counts"][4] > 0, k


@pytest.mark.gpu
def test_checked_build_traps_nothing_in_variant_matrix():
    """The matrix against libslicer_b200_chk.so (device-side bounds checks: queue slots, record regions, sort and tile cells).  A
    violated check traps and the run fails with the CUDA error.  Fresh interpreter: the library is loaded once per process."""
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    chk = os.path.join(root, "slicer_b200", "_build", "libslicer_b200_chk.so")
    if not os.path.exists(chk):
        pytest.skip("checked build not present (python -c 'import __graft_entry__ as g; g.build()')")
    r = subprocess.run([sys.executable, "-m", "pytest", os.path.abspath(__file__), "-x", "-q", "-m", "gpu", "-k", "test_variant_matrix and not checked_build",
                        "-p", "no:cacheprovider"], env=dict(os.environ, SLICER_B200_LIB=chk), cwd=root, capture_output=True, text=True)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-2000:]
