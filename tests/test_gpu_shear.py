"""Shear maps (SLICER_b200 --shear; slicer_shear / slicer_shear_fetch): Kaiser–Squires γ1, γ2 of every convergence map through a
deterministic, zero-padded FFT on the GPU (csrc/shear.cuh, DESIGN §12).

`restated_shear` restates the definition pass by pass in numpy: the same Stockham stages in the same real double operations, the
same twiddle table from libm, the same skipped rows.  CPU: the restatement against numpy.fft, periodic analytic modes, the
tangential shear of a Gaussian peak, and the driver's refusals.  GPU: the library against the restatement bit for bit (and the
same physics checks on the device), its refusals, the checked build; the driver's γ files against numpy KS of its own κ files,
their byte identity across ways of running, and resume."""
import math
import os
import subprocess
import sys

import numpy as np
import pytest

import fits_standard
from slicer_b200 import capi, host, synth
from test_gpu_driver import make_dataset
from test_gpu_kappa import deposit_random_slots, gpus
from test_gpu_realisations import ini_text, realisation_inis, run_exe, tree

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


# ---- the definition, restated ---------------------------------------------------------------------------------------------------
def twiddles(P):
    """The table the library fills: cos(2.0*M_PI*k/P), sin(2.0*M_PI*k/P) with the same libm"""
    return (np.array([math.cos(2.0 * math.pi * k / P) for k in range(P)]), np.array([math.sin(2.0 * math.pi * k / P) for k in range(P)]))


def stage(re, im, n, R, inv, wc, ws):
    """One Stockham stage of radix R on sub-transforms of n points along the last axis"""
    L, P = re.shape
    m = P // (n * R)
    xr, xi = re.reshape(L, R, m, n), im.reshape(L, R, m, n)
    j = np.arange(n)
    t = [(xr[:, 0], xi[:, 0])]
    for q in range(1, R):
        a, b = xr[:, q], xi[:, q]
        c, s = wc[q * j * m], ws[q * j * m]
        t.append((a * c - b * s, b * c + a * s) if inv else (a * c + b * s, b * c - a * s))
    if R == 2:
        y = [(t[0][0] + t[1][0], t[0][1] + t[1][1]), (t[0][0] - t[1][0], t[0][1] - t[1][1])]
    else:
        a0 = (t[0][0] + t[2][0], t[0][1] + t[2][1])
        a1 = (t[0][0] - t[2][0], t[0][1] - t[2][1])
        a2 = (t[1][0] + t[3][0], t[1][1] + t[3][1])
        a3 = (t[1][0] - t[3][0], t[1][1] - t[3][1])
        minus_i = (a1[0] + a3[1], a1[1] - a3[0])  # a1 - i a3
        plus_i = (a1[0] - a3[1], a1[1] + a3[0])  # a1 + i a3
        y = [(a0[0] + a2[0], a0[1] + a2[1]), plus_i if inv else minus_i, (a0[0] - a2[0], a0[1] - a2[1]), minus_i if inv else plus_i]
    outr, outi = np.empty((L, m, R, n)), np.empty((L, m, R, n))
    for r in range(R):
        outr[:, :, r, :], outi[:, :, r, :] = y[r]
    return outr.reshape(L, P), outi.reshape(L, P)


def transform_lines(re, im, inv, wc, ws):
    """Radix 4 while at least 4 points remain per sub-transform, then one radix 2"""
    P, n = re.shape[1], 1
    while n < P:
        R = 4 if P // n >= 4 else 2
        re, im = stage(re, im, n, R, inv, wc, ws)
        n *= R
    return re, im


def multiplier(P):
    """D1, D2 [f2, f1]"""
    f = np.arange(P)
    s = np.where(f < P // 2, f, f - P).astype(np.float64)
    s1, s2 = s[None, :], s[:, None]
    d = s1 * s1 + s2 * s2
    with np.errstate(invalid="ignore", divide="ignore"):
        D1 = (s1 * s1 - s2 * s2) / d
        D2 = (2.0 * s1 * s2) / d
    D1[0, 0] = D2[0, 0] = 0.0
    D2[:, P // 2] = 0.0
    D2[P // 2, :] = 0.0
    return D1, D2


def restated_shear(k, P):
    """γ1, γ2 [gy, gx] of κ [gy, gx] on a P x P grid, operation for operation as the library forms them"""
    n = k.shape[0]
    wc, ws = twiddles(P)
    K = np.zeros((n, P))
    K[:, :n] = k
    rr, ri = transform_lines(K, np.zeros((n, P)), False, wc, ws)  # forward rows: the npix rows of κ only
    re, im = np.zeros((P, P)), np.zeros((P, P))  # the other rows stay +0
    re[:n], im[:n] = rr, ri
    cr, ci = transform_lines(np.ascontiguousarray(re.T), np.ascontiguousarray(im.T), False, wc, ws)  # forward columns
    re, im = cr.T, ci.T
    D1, D2 = multiplier(P)
    gr, gi = D1 * re - D2 * im, D1 * im + D2 * re
    cr, ci = transform_lines(np.ascontiguousarray(gr.T), np.ascontiguousarray(gi.T), True, wc, ws)  # inverse columns
    rr, ri = transform_lines(np.ascontiguousarray(cr.T[:n]), np.ascontiguousarray(ci.T[:n]), True, wc, ws)  # inverse rows of the window
    sc = 1.0 / (P * P)
    return rr[:, :n] * sc, ri[:, :n] * sc


def numpy_shear(k, P):
    """The same definition through numpy.fft"""
    n = k.shape[0]
    K = np.zeros((P, P))
    K[:n, :n] = k
    D1, D2 = multiplier(P)
    G = np.fft.ifft2((D1 + 1j * D2) * np.fft.fft2(K))
    return G.real[:n, :n], G.imag[:n, :n]


def driver_fft(npix):
    """The driver's P: the smallest power of two >= 2 npix"""
    return 1 << math.ceil(math.log2(2 * npix))


def device_shear(k, P):
    n = k.shape[0]
    with capi.Slicer(npix_max=n, max_planes=1) as s:
        s.kappa_maps(1, n)
        s.kappa_load(0, k)
        s.shear(0, P)
        return s.shear_fetch()


def shear_by(where, k, P):
    return restated_shear(k, P) if where == "restated" else device_shear(k, P)


WHERE = ["restated", pytest.param("device", marks=pytest.mark.gpu)]


def same_bits(a, b):
    return np.array_equal(np.ascontiguousarray(a).view(np.uint64), np.ascontiguousarray(b).view(np.uint64))


def random_kappa(npix, seed):
    return np.random.default_rng(seed).standard_normal((npix, npix)) * 0.01 + 0.003


# ---- CPU: the restatement and the physics ---------------------------------------------------------------------------------------
@pytest.mark.parametrize("npix", [8, 100, 333, 512])
def test_restatement_matches_numpy_fft(npix):
    k = random_kappa(npix, npix)
    P = driver_fft(npix)
    got, want = restated_shear(k, P), numpy_shear(k, P)
    err = max(np.abs(got[0] - want[0]).max(), np.abs(got[1] - want[1]).max())
    assert err <= 1e-14 * np.abs(k).max(), err


@pytest.mark.parametrize("where", WHERE)
def test_periodic_analytic_modes(where):
    """P = npix = 64: κ = cos(2 pi (a x + b y) / P) has γ1 = D1(a, b) κ and γ2 = D2(a, b) κ; D2 = 0 on the Nyquist row and column."""
    P = 64
    x, y = np.arange(P)[None, :], np.arange(P)[:, None]
    for a, b in ((3, 5), (-7, 2), (0, 9), (32, 4), (5, 32), (32, 32)):
        k = np.cos(2 * np.pi * (a * x + b * y) / P)
        g1, g2 = shear_by(where, k, P)
        d = a * a + b * b
        D1 = (a * a - b * b) / d
        D2 = 0.0 if 32 in (abs(a), abs(b)) else 2 * a * b / d
        assert np.abs(g1 - D1 * k).max() <= 1e-13, (a, b)
        assert np.abs(g2 - D2 * k).max() <= 1e-13, (a, b)


@pytest.mark.parametrize("where", WHERE)
def test_tangential_shear_of_a_gaussian_peak(where):
    """npix 128, σ = 3 px, centre off the grid, the driver's P: γ_t = -(γ1 cos 2φ + γ2 sin 2φ) equals κ̄(<r) - κ(r) within 3 % for
    2σ <= r <= 0.4 npix, and the cross component stays below 3 % of it.  This pins the sign and the axes (φ from gx towards gy)."""
    n, sig = 128, 3.0
    c = n // 2 + 0.3
    yy, xx = np.mgrid[0:n, 0:n].astype(float)
    dx, dy = xx - c, yy - c
    r2 = dx * dx + dy * dy
    k = np.exp(-r2 / (2 * sig * sig))
    g1, g2 = shear_by(where, k, driver_fft(n))
    phi = np.arctan2(dy, dx)
    gt = -(g1 * np.cos(2 * phi) + g2 * np.sin(2 * phi))
    gx = -(g2 * np.cos(2 * phi) - g1 * np.sin(2 * phi))
    want = 2 * sig * sig / r2 * (1 - np.exp(-r2 / (2 * sig * sig))) - k
    m = (np.sqrt(r2) >= 2 * sig) & (np.sqrt(r2) <= 0.4 * n)
    assert np.max(np.abs(gt[m] - want[m]) / want[m]) <= 0.03
    assert np.max(np.abs(gx[m]) / want[m]) <= 0.03


# ---- CPU: refusals ---------------------------------------------------------------------------------------------------------------
REFUSALS = {
    "physical": (dict(npix=-500), ["--shear"], "physical pixels"),
    "npix 16385": (dict(npix=16385), ["--shear"], "at most 32768^2"),
    "non-flat": ({}, ["--shear"], "not flat"),
    "zs above the ini's": ({}, ["--shear", "--kappa-zs", "0.1,0.3"], "outside (0, 0.2]"),
    "nine sources": ({}, ["--shear", "--kappa-zs", ",".join(str(0.02 * (i + 1)) for i in range(9))], "at most 8"),
}


@pytest.mark.parametrize("case", sorted(REFUSALS))
def test_refused_before_anything_is_written(tmp_path, case):
    kw, args, msg = REFUSALS[case]
    if case == "non-flat":
        snapdir = tmp_path / "snaps"
        for i in range(2):
            synth.write_snapshot(str(snapdir / f"snap_{i:03d}"), {1: synth.uniform_positions(512, 128000.0, 5 + i)}, [0, 1.0375, 0, 0, 0, 0],
                                 0.1 * i, 128000.0, numfiles=1, om0=0.3, oml=0.6)
        lst = tmp_path / "snapshot_list.txt"
        lst.write_text("snap_000\nsnap_001")
        snapdir, lst = str(snapdir) + "/", str(lst)
    else:
        snapdir, lst = make_dataset(tmp_path, ng=8, nsnap=2, numfiles=1)
    out = tmp_path / "out"
    out.mkdir()
    ini = tmp_path / "a.ini"
    ini.write_text(ini_text(lst, snapdir, str(out) + "/t_", **kw))
    r = run_exe([*args, ini], tmp_path, quiet=False, timeout=120)
    assert r.returncode != 0
    assert msg in r.stderr, r.stderr
    assert os.listdir(out) == []


# ---- GPU: the library ------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("npix,P", [(8, 16), (100, 256), (333, 1024), (1000, 2048), (256, 256)])
def test_library_bit_for_bit_against_the_restatement(npix, P):
    k = random_kappa(npix, 11 + npix)
    got = device_shear(k, P)
    want = restated_shear(k, P)
    assert same_bits(got[0], want[0]) and same_bits(got[1], want[1])
    assert np.count_nonzero(got[1]) > 0


@pytest.mark.gpu
def test_library_bit_for_bit_on_a_deposited_map():
    """κ formed by slicer_kappa_add from a deposited pass; two maps in a row at one P, then another P on the same handle (the
    workspace is made again)."""
    npix, nslots = 64, 4
    rng = np.random.default_rng(5)
    scale, offset = rng.uniform(1e-6, 1e-3, (nslots, 2)), -rng.uniform(1e-6, 1e-3, (nslots, 2))
    with capi.Slicer(npix_max=npix, max_planes=nslots, particle_capacity=(1 << 17) + 64) as s:
        deposit_random_slots(s, npix, nslots, 1 << 17, 900)
        s.kappa_maps(2, npix)
        s.kappa_add(0, [0] * nslots, scale, offset)
        kappa = [s.kappa_fetch(m) for m in range(2)]
        got = []
        for m, P in ((0, 128), (1, 128), (0, 256)):
            s.shear(m, P)
            got.append((m, P, s.shear_fetch()))
    assert np.std(kappa[0]) > 0
    for m, P, (g1, g2) in got:
        w1, w2 = restated_shear(kappa[m], P)
        assert same_bits(g1, w1) and same_bits(g2, w2), (m, P)


@pytest.mark.gpu
def test_library_against_numpy_fft_at_2048():
    k = random_kappa(2048, 3)
    g1, g2 = device_shear(k, 4096)
    w1, w2 = numpy_shear(k, 4096)
    assert max(np.abs(g1 - w1).max(), np.abs(g2 - w2).max()) <= 1e-14 * np.abs(k).max()


@pytest.mark.gpu
def test_library_refusals():
    with capi.Slicer(npix_max=64, max_planes=1) as s:
        with pytest.raises(capi.SlicerError, match="no convergence maps"):
            s.shear(0, 128)
        s.kappa_maps(2, 64)
        with pytest.raises(capi.SlicerError, match="no shear map"):
            s.shear_fetch()
        for P in (96, 32, 65536, 0):
            with pytest.raises(capi.SlicerError, match="power of two"):
                s.shear(0, P)
        for m in (-1, 2):
            with pytest.raises(capi.SlicerError, match="outside 0..1"):
                s.shear(m, 128)


@pytest.mark.gpu
def test_overflowed_kappa_map_fails_the_fetch():
    """The accumulator overflow of tests/test_gpu_parity.py, summed into a κ map: neither the map nor its shear is returned."""
    box, n = 128000.0, 48
    pos = np.tile(np.array([[0.5, 0.5, 0.3]], np.float32) * np.float32(box), (n, 1))
    d = capi.plane_desc([1, 1, 1], 1, [0.0, 0.0, 0.0], 0.0, 10.0, 100.0, 0.5, 64)
    with capi.Slicer(npix_max=64, max_planes=1, mas=capi.MAS_NGP, particle_capacity=n + 64, frac_bits=58) as s:
        s.begin_snapshot(box, [0, 1.0, 0, 0, 0, 0], False)
        s.stage(1, pos)
        s.deposit([d])
        s.kappa_maps(1, 64)
        s.kappa_add(0, [0], [[1e-3]], [[0.0]])
        s.shear(0, 128)
        with pytest.raises(capi.SlicerError, match="exceeded 2\\^63"):
            s.shear_fetch()
        with pytest.raises(capi.SlicerError, match="frac_bits"):
            s.kappa_fetch(0)


@pytest.mark.gpu
def test_checked_build_traps_nothing_in_the_shear_kernels():
    """The bit-for-bit library tests against libslicer_b200_chk.so (SLICER_CHECK bounds assertions in shear_fft_pass)."""
    chk = os.path.join(ROOT, "slicer_b200", "_build", "libslicer_b200_chk.so")
    if not os.path.exists(chk):
        pytest.skip("checked build not present (python -c 'import __graft_entry__ as g; g.build()')")
    r = subprocess.run([sys.executable, "-m", "pytest", os.path.abspath(__file__), "-x", "-q", "-m", "gpu", "-k", "bit_for_bit", "-p",
                        "no:cacheprovider"], env=dict(os.environ, SLICER_B200_LIB=chk), cwd=ROOT, capture_output=True, text=True)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-2000:]


# ---- GPU: the driver -------------------------------------------------------------------------------------------------------------
KEYS = ("ZSOURCE", "DS", "PHYSICALSIZE", "NPLANES", "HUBBLE", "OMEGAMATTER", "OMEGALAMBDA")


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["tsc", "ngp", "hydro_per_type"])
def test_driver_gamma_files_equal_numpy_on_its_own_kappa(tmp_path, case):
    """Two source redshifts: each γ file against numpy KS of the same run's κ file (float32 of the same double κ) within
    1e-6 max|κ|; the files pass the standard-driven reader and carry κ's keys plus FFTSIZE."""
    npix = 64
    snapdir, lst = make_dataset(tmp_path, nsnap=4, numfiles=2, hydro=case == "hydro_per_type")
    out = tmp_path / "out"
    out.mkdir()
    ini = tmp_path / "a.ini"
    ini.write_text(ini_text(lst, snapdir, str(out) + "/t_", npix=npix, pip=1 if case == "hydro_per_type" else 0))
    r = run_exe([*(["--ngp"] if case == "ngp" else []), "--shear", "--kappa-zs", "0.2,0.1", ini], tmp_path)
    assert r.returncode == 0, r.stderr[-3000:]
    P = driver_fft(npix)
    for z in (0.2, 0.1):
        khdr, k = host.read_fits(str(out / f"t_gadget.kappa_{npix}_zs{z:.4f}_0.fits"))
        want = numpy_shear(k.astype(np.float64), P)
        for i, name in enumerate(("gamma1", "gamma2")):
            f = str(out / f"t_gadget.{name}_{npix}_zs{z:.4f}_0.fits")
            hdr, g = host.read_fits(f)
            assert np.abs(g - want[i]).max() <= 1e-6 * np.abs(k).max(), (z, name)
            assert np.std(g) > 0
            std_hdr, rows = fits_standard.read_primary_image(f)
            assert np.array_equal(np.asarray(rows, np.float32).reshape(npix, npix), g)
            assert all(hdr[key] == khdr[key] for key in KEYS) and hdr["FFTSIZE"] == P and std_hdr["FFTSIZE"] == P


def shear_files(files):
    return sorted(f for f in files if ".gamma1_" in f or ".gamma2_" in f)


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["no_planes", "separately", "max_slots", "two_gpus", "two_procs"])
def test_gamma_files_are_byte_identical(tmp_path, case):
    snapdir, lst = make_dataset(tmp_path, ng=40, nsnap=3, numfiles=4)
    args = ["--shear", "--kappa-zs", "0.1,0.05"]

    def inis(tag):
        return realisation_inis(tmp_path, tag, lst, snapdir, 2, zs=0.1)

    r = run_exe([*args, *inis("base")], tmp_path)
    assert r.returncode == 0, r.stderr[-3000:]
    ref = tree(tmp_path / "base")
    if case in ("two_gpus", "two_procs") and gpus() < 2:
        pytest.skip("needs 2 GPUs")
    if case == "no_planes":
        r = run_exe([*args, "--no-planes", *inis("other")], tmp_path)
    elif case == "separately":
        for ini in inis("other"):
            r = run_exe([*args, ini], tmp_path)
            assert r.returncode == 0, r.stderr[-3000:]
    elif case == "max_slots":
        r = run_exe([*args, "--max-slots", "3", *inis("other")], tmp_path)
    elif case == "two_gpus":
        r = run_exe([*args, "--gpus", "0,1", *inis("other")], tmp_path)
    else:
        from test_multiprocess import run_job

        res = run_job(inis("other"), tmp_path, [[0], [1]], extra=args)
        assert all(rc == 0 for rc, _, _ in res), [e[-2000:] for _, _, e in res]
    if case != "two_procs":
        assert r.returncode == 0, r.stderr[-3000:]
    got = tree(tmp_path / "other")
    sf = shear_files(ref)
    assert len(sf) == 8
    assert all(got[f] == ref[f] for f in sf), [f for f in sf if got.get(f) != ref[f]]


@pytest.mark.gpu
def test_resume(tmp_path):
    """Two light cones with two source redshifts.  All files present: nothing is deposited.  One γ2 file gone: that light cone is
    deposited again and only that file is written, byte for byte as before; no other FITS file's modification time changes
    (planes_list is written by every run)."""
    snapdir, lst = make_dataset(tmp_path, ng=24, nsnap=3, numfiles=2)
    inis = realisation_inis(tmp_path, "out", lst, snapdir, 2, npix=32, zs=0.1, fov=5.0)
    args = ["--shear", "--kappa-zs", "0.1,0.05"]
    assert run_exe([*args, *inis], tmp_path).returncode == 0
    before = tree(tmp_path / "out")
    stamp = {f: os.stat(tmp_path / "out" / f).st_mtime_ns for f in before}
    assert len(shear_files(before)) == 8
    r = run_exe([*args, *inis], tmp_path, quiet=False)
    assert r.returncode == 0, r.stderr[-3000:]
    assert " sub-file " not in r.stdout and tree(tmp_path / "out") == before
    gone = [f for f in shear_files(before) if ".gamma2_" in f and f.endswith("_r1.fits")][0]
    os.remove(tmp_path / "out" / gone)
    r = run_exe([*args, *inis], tmp_path, quiet=False)
    assert r.returncode == 0, r.stderr[-3000:]
    assert " sub-file " in r.stdout
    assert r.stdout.count(" Already exists") == sum(f.endswith(".fits") for f in before) - 1
    assert tree(tmp_path / "out") == before
    rewritten = {f for f in before if f.endswith(".fits") and os.stat(tmp_path / "out" / f).st_mtime_ns != stamp[f]}
    assert rewritten == {gone}
