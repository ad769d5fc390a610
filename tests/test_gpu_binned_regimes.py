"""The binned deposit's sort regimes against the oracle, bit for bit.  All tests need a B200.

The binned path (csrc/deposit_binned.cuh, planned by `binned_gshift` / `binned_pass` in csrc/slicer_capi.cu) picks its sort
layout from the map size and the number of planes of a pass: tile groups of 1, 2 or 4 tiles, one or several sort windows over
the same records, the record kernel's own histogram for small passes, and four scatter variants.  `plan` below restates that
planner; every row of the matrix pins one regime through it, checks through the launch count that the library ran that
regime, checks that every tile of every plane holds records, and compares counts and int64 maps with the oracle.

Further: planes smaller than the handle's npix_max (alone, after a larger plane in the same slot, and mixed in one pass),
the fixed-point scale at other `frac_bits` than the default, and per-particle masses on either side of MAX_M.
"""
import os
import subprocess
import sys

import numpy as np
import pytest

from oracle.oracle_bindings import MAX_M
from slicer_b200 import capi, synth
from test_gpu_parity import check_against_oracle

pytestmark = pytest.mark.gpu

# ---- the planner, restated (csrc/deposit_binned.cuh constants; csrc/slicer_capi.cu: binned_tiles, binned_gshift, binned_alloc,
# binned_pass, run_pass) --------------------------------------------------------------------------------------------------
TILE = 166          # binned::TILE: interior cells per tile side
MAX_BINS = 5120     # binned::MAX_BINS: bins per sort window
HIST_BINS = 1024    # binned::HIST_BINS: up to this many bins the record kernel builds the histogram (no bin_histogram_kernel)
SMALL_BINS = 4096   # binned::SMALL_BINS: table of the single-window scatter kernel
CHUNK = 1024        # pipe::CHUNK: slices are whole chunks


def plan(npix, nplanes):
    """Sort layout of a binned pass over `nplanes` planes of npix^2."""
    nt = (npix + TILE - 1) // TILE                       # tiles per map side
    g = 0                                                # groups of 2^g tiles along x, as small as fits MAX_BINS
    while g < 2 and nplanes * nt * ((nt + (1 << g) - 1) >> g) > MAX_BINS:
        g += 1
    ntx = (nt + (1 << g) - 1) >> g                       # groups per tile row
    nbins = nplanes * nt * ntx                           # bin = (plane * ntile + tile row) * ntx + group
    nwin = (nbins + MAX_BINS - 1) // MAX_BINS
    wbins = (nbins + nwin - 1) // nwin
    cuts = list(range(wbins, nbins, wbins))              # bin_lo of every window but the first
    return dict(ntile=nt, gshift=g, ntx=ntx, nbins=nbins, nwin=nwin, wbins=wbins,
                k1_hist=nbins <= HIST_BINS and nbins <= MAX_BINS,
                scatter="small" if nwin == 1 and nbins <= SMALL_BINS else "windowed",
                last_group=nt - ((ntx - 1) << g),        # tiles in the last group of a row
                cut_inside_plane=all(c % (nt * ntx) for c in cuts),
                cut_inside_row=all(c % ntx for c in cuts))


def binned_slice(particle_capacity, record_capacity=0):
    """Particles per record-kernel slice of a pass with one randomisation (binned_alloc, binned_pass)."""
    s = record_capacity or (1 << 28)
    s = min(s, 1 << 31)
    s = min(s, particle_capacity or s)
    return (s + CHUNK - 1) // CHUNK * CHUNK


def pass_launches(segments, binned, pl=None, slice_=None):
    """Kernel launches of one pass (run_pass, binned_pass): one per non-empty segment (the deposit or record kernel), and per
    binned slice the scan of the bin totals plus, per window, [histogram,] region scan, scatter and tile kernel."""
    total = 0
    for n in segments:
        if n == 0:
            continue
        total += 1
        if binned:
            nslices = (n + slice_ - 1) // slice_
            total += nslices * (1 + pl["nwin"] * (3 if pl["k1_hist"] else 4))
    return total


# ---- geometry ---------------------------------------------------------------------------------------------------------
# One randomisation, rcase 1: every particle lies in the slab z in [1, 2) box units, which the planes cut into equal, disjoint
# slabs (overlapping slabs would leave the binned path).  fov 0.45 rad keeps the whole field inside the box's cross-section
# out to z = 2 (z tan(T) / cos(T) < 1/2), so that every tile of every plane, up to the far corner of the last slab, is reached.
BOX = 128000.0
FOV = 0.45
SGN, FACE, CENTRE, RCASE = [1, -1, 1], 2, [0.25, 0.5, 0.75], 1.0
MASS1 = 1.5


def slab_planes(nplanes, npix):
    edges = [128.0 + 128.0 * k / nplanes for k in range(nplanes + 1)]  # Mpc/h: box units 1 + k / nplanes
    raw = [dict(boxsize=BOX, sgn=SGN, face=FACE, centre=CENTRE, rcase=RCASE, ld=edges[k], ld2=edges[k + 1], nrepperp=0,
                fovradiants=FOV) for k in range(nplanes)]
    return raw, [capi.plane_desc(SGN, FACE, CENTRE, RCASE, p["ld"], p["ld2"], FOV, n) for p, n in zip(raw, npix)]


def hydro_masses(n, seed):
    """Per-particle float32 masses, about 1 % above MAX_M (deposited with mass 0, still counted)."""
    rng = np.random.default_rng(seed)
    m = (0.05 + 2.0 * rng.random(n)).astype(np.float32)
    heavy = rng.random(n) < 0.01
    m[heavy] = (MAX_M * (1.0 + 2.0 * rng.random(int(heavy.sum())))).astype(np.float32)
    return m


def segments_for(n, masses, seed):
    """[(type, positions, masses or None)]: one constant-mass segment, or a constant-mass and a per-particle-mass segment."""
    if not masses:
        return [(1, synth.uniform_positions(n, BOX, seed), None)]
    n0 = n // 2
    return [(1, synth.uniform_positions(n - n0, BOX, seed), None),
            (0, synth.uniform_positions(n0, BOX, seed + 1), hydro_masses(n0, seed + 2))]


def oracle_plane(oracle, xyz, segs, p, npix, frac_bits, do_ngp):
    """One plane through the oracle without its 18 full maps: -> counts[6], ingrid[6], int64 map summed over the types,
    accepted (xs, ys) of all types."""
    counts = np.zeros(6, np.int64)
    ingrid = np.zeros(6, np.int64)
    fixed = np.zeros(npix * npix, np.int64)
    acc = []
    for (ty, _, mass), (x, y, z) in zip(segs, xyz):
        xs, ys, ms = oracle.select_project(x, y, z, p["ld"], p["ld2"], BOX, 0, FOV, npix, const_mass=MASS1, per_particle=mass,
                                           max_m=MAX_M, cap=len(x) + 16)
        counts[ty] += len(xs)
        ingrid[ty] += int(np.count_nonzero(oracle.ngp_cells_fast(xs, ys, npix) >= 0))
        oracle.gridist_w_fixed(xs, ys, ms, npix, frac_bits, do_ngp, out=fixed)  # adds
        acc.append((xs, ys))
    return counts, ingrid, fixed, acc


def tiles_hit(acc, npix, nt):
    """Records per tile of one plane, as binned::bin_of assigns them (clamped NGP cell / TILE)."""
    hits = np.zeros(nt * nt, np.int64)
    for xs, ys in acc:
        gx = np.clip(np.floor(xs.astype(np.float64) * npix).astype(np.int64), 0, npix - 1) // TILE
        gy = np.clip(np.floor(ys.astype(np.float64) * npix).astype(np.int64), 0, npix - 1) // TILE
        hits += np.bincount(gy * nt + gx, minlength=nt * nt)
    return hits


# ---- 1. the regime matrix ----------------------------------------------------------------------------------------------
# (id, npix, planes, masses, mas list, deposit mode, record_capacity as a fraction of n, particles, what the row pins)
N = 1 << 22
ROWS = [
    ("2048x6", 2048, 6, False, ["tsc"], capi.DEPOSIT_BINNED, 0, N, dict(nbins=1014, k1_hist=True)),
    ("2048x7-mass", 2048, 7, True, ["ngp"], capi.DEPOSIT_BINNED, 0, N, dict(nbins=1183, k1_hist=False, scatter="small")),
    ("4096x8-mass", 4096, 8, True, ["tsc"], capi.DEPOSIT_BINNED, 0, N, dict(gshift=0, nbins=5000, nwin=1, scatter="windowed")),
    ("4096x16", 4096, 16, False, ["tsc"], capi.DEPOSIT_BINNED, 0, N, dict(gshift=2, last_group=1, nwin=1)),
    ("8192x3-mass", 8192, 3, True, ["tsc", "ngp"], capi.DEPOSIT_BINNED, 0, N, dict(gshift=1, nwin=1, scatter="small")),
    ("8192x6-auto", 8192, 6, False, ["tsc"], capi.DEPOSIT_AUTO, 0, N, dict(gshift=2, last_group=2, nwin=1)),
    ("8192x9-mass", 8192, 9, True, ["tsc"], capi.DEPOSIT_BINNED, 0, N, dict(gshift=2, nwin=2, cut_inside_plane=True)),
    ("8192x16", 8192, 16, False, ["tsc", "ngp"], capi.DEPOSIT_BINNED, 0, 1 << 23, dict(gshift=2, nwin=3, cut_inside_row=True)),
    ("8192x9-slices", 8192, 9, False, ["tsc"], capi.DEPOSIT_BINNED, 1 / 3, N, dict(gshift=2, nwin=2)),
    ("16384x3", 16384, 3, False, ["tsc"], capi.DEPOSIT_BINNED, 0, N, dict(ntile=99, gshift=2, last_group=3, nwin=2)),
]
MATRIX = [pytest.param(r, mas, id=f"{r[0]}-{mas}") for r in ROWS for mas in r[4]]
SEEDS = {r[0]: 100 + 10 * i for i, r in enumerate(ROWS)}


@pytest.mark.parametrize("row,mas", MATRIX)
def test_regime_matrix(oracle, row, mas):
    """One pass over all planes of a row: (a) the launches of the pass are those of the regime the row pins, (b) every tile of
    every plane holds records (so does every bin: the last group of every row and both sides of every window boundary), (c) for
    every plane the accepted counts, the in-grid counts and the full int64 map equal the oracle's."""
    name, npix, nplanes, masses, _, mode, rc_frac, n, pins = row
    pl = plan(npix, nplanes)
    assert {k: pl[k] for k in pins} == pins, pl  # the row still exercises the regime it is meant to
    segs = segments_for(n, masses, SEEDS[name])
    raw, descs = slab_planes(nplanes, [npix] * nplanes)
    cap = sum(len(pos) for _, pos, _ in segs) + 64
    record_capacity = int(n * rc_frac) + 1 if rc_frac else 0
    slice_ = binned_slice(cap, record_capacity)
    if rc_frac:
        assert all((len(pos) + slice_ - 1) // slice_ >= 3 for _, pos, _ in segs)
    do_ngp = mas == "ngp"
    with capi.Slicer(npix_max=npix, max_planes=nplanes, mas=capi.MAS_NGP if do_ngp else capi.MAS_TSC, particle_capacity=cap,
                     mass_capacity=cap if masses else 0, per_type_maps=False, deposit_mode=mode, record_capacity=record_capacity) as s:
        s.begin_snapshot(BOX, [0, MASS1, 0, 0, 0, 0], masses)
        for ty, pos, mass in segs:
            s.stage(ty, pos, mass)
        l0 = s.stats().launches
        s.deposit(descs)
        launches = s.stats().launches - l0
        assert launches == pass_launches([len(pos) for _, pos, _ in segs], True, pl, slice_), (launches, pl)
        fb = s.frac_bits
        xyz = [oracle.transform(pos, BOX, SGN, FACE, CENTRE, RCASE) for _, pos, _ in segs]
        for k, p in enumerate(raw):
            counts, ingrid, want, acc = oracle_plane(oracle, xyz, segs, p, npix, fb, do_ngp)
            hits = tiles_hit(acc, npix, pl["ntile"])
            assert hits.min() > 0, (k, np.flatnonzero(hits == 0)[:10])
            _, c, g = s.fetch(k, -1, npix, want_map=False)
            assert c.tolist() == counts.tolist(), (k, c, counts)
            assert g.tolist() == ingrid.tolist(), (k, g, ingrid)
            got = s.fetch_fixed(k, -1, npix).reshape(-1)
            if not np.array_equal(got, want):
                bad = np.flatnonzero(got != want)
                pytest.fail(f"plane {k}: {len(bad)} cells differ, first at (gy, gx) = {divmod(int(bad[0]), npix)}, "
                            f"tiles {sorted(set(((b // npix) // TILE * pl['ntile'] + (b % npix) // TILE) for b in bad[:1000].tolist()))[:10]}")
            del got, want, acc


# ---- 2. planes smaller than npix_max -----------------------------------------------------------------------------------
PATHS = [pytest.param(capi.KERNEL_SIMPLE, capi.DEPOSIT_AUTO, id="simple"), pytest.param(capi.KERNEL_PIPELINED, capi.DEPOSIT_DIRECT, id="direct"),
         pytest.param(capi.KERNEL_PIPELINED, capi.DEPOSIT_BINNED, id="binned")]


def _fetch_types(s, k, npix, types):
    _, counts, ingrid = s.fetch(k, -1, npix, want_map=False)
    return dict(counts=counts, ingrid=ingrid, frac_bits=s.frac_bits,
                maps={t["type"]: s.fetch(k, t["type"], npix)[0].reshape(-1) for t in types},
                fixed={t["type"]: s.fetch_fixed(k, t["type"], npix).reshape(-1) for t in types})


MAS = [pytest.param(capi.MAS_TSC, id="tsc"), pytest.param(capi.MAS_NGP, id="ngp")]


@pytest.mark.parametrize("mas", MAS)
@pytest.mark.parametrize("kernel,mode", PATHS)
def test_planes_below_npix_max(oracle, kernel, mode, mas):
    """A handle with npix_max = 1024: two planes at 1024, then the same slots at 512, then at 256 (no cell of the earlier, larger
    pass may survive), then one pass with a 256^2 and a 512^2 plane (which leaves the binned path).  Counts, int64 maps and
    float maps of each plane at its own npix equal the oracle's."""
    n0, n1 = 60000, 140000
    pos1 = synth.uniform_positions(n1, BOX, 71)
    pos0 = synth.uniform_positions(n0, BOX, 72)
    m0 = hydro_masses(n0, 73)
    types = [dict(type=1, raw=pos1, const_mass=MASS1), dict(type=0, raw=pos0, masses=m0, cut=True)]
    do_ngp = mas == capi.MAS_NGP
    with capi.Slicer(npix_max=1024, max_planes=2, mas=mas, particle_capacity=n0 + n1 + 64, mass_capacity=n0 + 64, per_type_maps=True,
                     kernel=kernel, deposit_mode=mode) as s:
        s.begin_snapshot(BOX, [0, MASS1, 0, 0, 0, 0], True)
        s.stage(1, pos1)
        s.stage(0, pos0, m0)
        for npix in ([1024, 1024], [512, 512], [256, 256], [256, 512]):
            raw, descs = slab_planes(2, npix)
            l0 = s.stats().launches
            s.deposit(descs)
            binned = mode == capi.DEPOSIT_BINNED and npix[0] == npix[1]
            want = pass_launches([n1, n0], binned, plan(npix[0], 2), binned_slice(n0 + n1 + 64))
            assert s.stats().launches - l0 == want, npix
            for k in range(2):
                got = _fetch_types(s, k, npix[k], types)
                res = check_against_oracle(oracle, types, raw[k], npix[k], got, do_ngp, MASS1, strict_float=False)
                assert res["counts"][1] > 1000 and res["counts"][0] > 500


# ---- 3. fixed-point scale and the MAX_M cut ----------------------------------------------------------------------------
@pytest.mark.parametrize("mas", MAS)
@pytest.mark.parametrize("frac_bits", [20, 52])
def test_frac_bits_other_than_default(oracle, frac_bits, mas):
    """The tile kernel folds 2^frac_bits into the x weights (tile_tsc), the direct paths scale the product: both must round like
    the oracle's llrint(float contribution * 2^frac_bits) at a coarse and at a fine scale, on the simple, direct and binned paths."""
    n0, n1 = 100000, 200000
    pos1 = synth.uniform_positions(n1, BOX, 81)
    pos0 = synth.uniform_positions(n0, BOX, 82)
    m0 = (0.05 + 2.0 * np.random.default_rng(83).random(n0)).astype(np.float32)
    npix = 256
    raw, descs = slab_planes(1, [npix])
    p = raw[0]
    want = {}
    for ty, pos, kw in ((1, pos1, dict(const_mass=MASS1)), (0, pos0, dict(per_particle=m0))):
        x, y, z = oracle.transform(pos, BOX, SGN, FACE, CENTRE, RCASE)
        xs, ys, ms = oracle.select_project(x, y, z, p["ld"], p["ld2"], BOX, 0, FOV, npix, cap=len(x) + 16, **kw)
        want[ty] = (len(xs), oracle.gridist_w_fixed(xs, ys, ms, npix, frac_bits, mas == capi.MAS_NGP))
    for kernel, mode in ((capi.KERNEL_SIMPLE, capi.DEPOSIT_AUTO), (capi.KERNEL_PIPELINED, capi.DEPOSIT_DIRECT),
                         (capi.KERNEL_PIPELINED, capi.DEPOSIT_BINNED)):
        with capi.Slicer(npix_max=npix, max_planes=1, mas=mas, particle_capacity=n0 + n1 + 64, mass_capacity=n0 + 64, per_type_maps=True,
                         kernel=kernel, deposit_mode=mode, frac_bits=frac_bits) as s:
            assert s.frac_bits == frac_bits
            s.begin_snapshot(BOX, [0, MASS1, 0, 0, 0, 0], True)
            s.stage(1, pos1)
            s.stage(0, pos0, m0)
            l0 = s.stats().launches
            s.deposit(descs)
            binned = mode == capi.DEPOSIT_BINNED
            assert s.stats().launches - l0 == pass_launches([n1, n0], binned, plan(npix, 1), binned_slice(n0 + n1 + 64))
            _, c, _ = s.fetch(0, -1, npix, want_map=False)
            for ty in (1, 0):
                assert c[ty] == want[ty][0] and want[ty][0] > 10000
                assert np.array_equal(s.fetch_fixed(0, ty, npix).reshape(-1), want[ty][1]), (kernel, mode, ty)


@pytest.mark.parametrize("mas", MAS)
@pytest.mark.parametrize("mode", [pytest.param(capi.DEPOSIT_DIRECT, id="direct"), pytest.param(capi.DEPOSIT_BINNED, id="binned")])
def test_per_particle_mass_at_max_m(oracle, mode, mas):
    """Masses {the float below MAX_M, MAX_M, the float above}: the reference keeps m == MAX_M (m > MAX_M in double) and deposits
    the next float up with mass 0 (still counted).  Counts and int64 maps equal select_project(max_m=MAX_M)'s."""
    n = 150000
    pos = synth.uniform_positions(n, BOX, 91)
    vals = np.array([np.nextafter(np.float32(MAX_M), np.float32(0)), np.float32(MAX_M), np.nextafter(np.float32(MAX_M), np.float32(np.inf))],
                    np.float32)
    m = vals[np.arange(n) % 3]
    npix = 256
    raw, descs = slab_planes(1, [npix])
    p = raw[0]
    x, y, z = oracle.transform(pos, BOX, SGN, FACE, CENTRE, RCASE)
    xs, ys, ms = oracle.select_project(x, y, z, p["ld"], p["ld2"], BOX, 0, FOV, npix, per_particle=m, max_m=MAX_M, cap=n + 16)
    assert set(np.unique(ms).tolist()) == {0.0, float(vals[0]), float(vals[1])}
    with capi.Slicer(npix_max=npix, max_planes=1, mas=mas, particle_capacity=n + 64, mass_capacity=n + 64, per_type_maps=True,
                     deposit_mode=mode) as s:
        s.begin_snapshot(BOX, [0, 0, 0, 0, 0, 0], True)
        s.stage(0, pos, m)
        l0 = s.stats().launches
        s.deposit(descs)
        assert s.stats().launches - l0 == pass_launches([n], mode == capi.DEPOSIT_BINNED, plan(npix, 1), binned_slice(n + 64))
        fb = s.frac_bits
        _, c, g = s.fetch(0, -1, npix, want_map=False)
        got = s.fetch_fixed(0, 0, npix).reshape(-1)
    assert c[0] == len(xs) and g[0] == int(np.count_nonzero(oracle.ngp_cells_fast(xs, ys, npix) >= 0))
    assert np.array_equal(got, oracle.gridist_w_fixed(xs, ys, ms, npix, fb, mas == capi.MAS_NGP))


# ---- 4. the same file against the build with device-side bounds checks -------------------------------------------------
def test_checked_build_traps_nothing_in_binned_regimes():
    """This file (up to the 8192^2 x 9 rows) against libslicer_b200_chk.so: the SLICER_CHECK bounds assertions of the scatter and
    tile kernels (destination inside its bin's range, cells inside the tile) are what a windowing or grouping error violates.  A
    violated check traps and the run fails with the CUDA error.  Fresh interpreter: the library is loaded once per process."""
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    chk = os.path.join(root, "slicer_b200", "_build", "libslicer_b200_chk.so")
    if not os.path.exists(chk):
        pytest.skip("checked build not present (python -c 'import __graft_entry__ as g; g.build()')")
    sel = "not checked_build and not 8192x16 and not 16384x3"
    r = subprocess.run([sys.executable, "-m", "pytest", os.path.abspath(__file__), "-x", "-q", "-m", "gpu", "-k", sel, "-p", "no:cacheprovider"],
                       env=dict(os.environ, SLICER_B200_LIB=chk), cwd=root, capture_output=True, text=True)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-2000:]
