"""Convergence maps (SLICER_b200 --kappa / --kappa-zs / --no-planes; slicer_kappa_*): flat-sky, thin-plane Born sums of a light
cone's planes, formed on the GPU from the int64 accumulators.

CPU: the Born weights against a numpy restatement of their definition; every refused configuration exits before anything is
written.  GPU: the library's maps against numpy on the same integer planes bit for bit (per-type handles, two realisations in
one call, planes beyond a source, a 2-GPU reduce, odd and even map sides, the checked build); the driver's maps against its own
plane files; byte identity of the map files over --no-planes, several inis, --max-slots, GPUs and processes; resume; and the
mean convergence of a uniform universe."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

from slicer_b200 import capi, host, synth
from test_gpu_driver import make_dataset
from test_gpu_realisations import BOX, desc, random_planes, realisation_inis, run_exe, seed_triples, tree, SEEDS, ini_text

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SPEEDC = 2.99792458e3
RHO_C = 27.753662724817193  # 3 (100 km/s/Mpc)^2 / (8 pi G) in 1e10 Msun/h per (Mpc/h)^3


def numpy_weights(ld, ld2, z, chis, om0, fov_deg, npix):
    """The definition, restated: scale, offset [plane, source]"""
    A = 1.5 / (SPEEDC * SPEEDC)
    pix = fov_deg / 180.0 * np.pi / npix
    omega = pix * pix
    chi = (ld + ld2) / 2.0
    V = (ld2 * ld2 * ld2 - ld * ld * ld) / (3.0 * chi * chi)
    scale, offset = np.zeros((len(ld), len(chis))), np.zeros((len(ld), len(chis)))
    for k, cs in enumerate(chis):
        on = chi < cs
        g = (1.0 + z) * chi * (cs - chi) / cs
        scale[:, k] = np.where(on, A * g / (RHO_C * omega * chi * chi), 0.0)
        offset[:, k] = np.where(on, -(A * om0 * g * V), 0.0)
    return scale, offset


def numpy_kappa(planes, scale, offset, fb):
    """kappa += scale * (double(acc) * 2^-fb) + offset, plane after plane (numpy: IEEE double, no contraction)"""
    k = np.zeros(planes[0].shape)
    for acc, sc, of in zip(planes, scale, offset):
        if sc == 0 and of == 0:
            continue
        k = k + (sc * (acc.astype(np.float64) * 2.0 ** -fb) + of)
    return k


# ---- CPU: weights and refusals -----------------------------------------------------------------------------------------------
def test_weights_match_the_definition(tmp_path):
    """The weights restated from their definition to 1 ulp.  The restatement covers the formula; its inputs z_i = getZl(chi_i)
    and chi_s = getDl(zs_k) come from the plan's distance tables (the existing, separately tested CosmoTable), cross-checked here
    only against planes_list's plane redshifts (6 digits) and the plan's Ds."""
    snapred, snapbox = [0.0, 0.15, 0.3, 0.45, 0.6], [128000.0, 128000.0, 256000.0, 256000.0, 256000.0]
    om0, zs, fov, npix = 0.3, 0.5, 4.0, 128
    zs_list = [0.5, 0.2, 0.05]
    w = host.kappa_weights(om0, 1 - om0, -1.0, zs, snapred, snapbox, fov, npix, zs_list)
    plan = host.plan(om0, 1 - om0, -1.0, zs, snapred, snapbox, str(tmp_path) + "/", "t")
    assert np.array_equal(w["ld"], plan["ld"]) and np.array_equal(w["ld2"], plan["ld2"])
    assert w["chis"][0] == plan["Ds"]  # getDl(zs): the table the plan uses
    # z = getZl(chi) agrees with planes_list's plane redshift (column 2, printed to 6 digits) where chi is the plane's middle
    listed = np.loadtxt(tmp_path / "planes_list_t.txt", usecols=1)
    np.testing.assert_allclose(w["z"], listed, rtol=2e-5)
    scale, offset = numpy_weights(w["ld"], w["ld2"], w["z"], w["chis"], om0, fov, npix)
    for got, want in ((w["scale"], scale), (w["offset"], offset)):
        assert np.all(np.abs(got - want) <= np.spacing(np.abs(want))), np.max(np.abs(got - want) / np.spacing(np.abs(want) + 1e-300))
    # planes behind a source do not contribute; the first plane's slab depth is not ld2 - ld
    chi = (w["ld"] + w["ld2"]) / 2
    for k, cs in enumerate(w["chis"]):
        assert np.all((w["scale"][:, k] == 0) == (chi >= cs)) and np.count_nonzero(w["scale"][:, k]) >= 1
    assert np.all(w["scale"][chi < w["chis"][0], 0] > 0) and np.all(w["offset"][chi < w["chis"][0], 0] < 0)


REFUSALS = {
    "physical": (dict(npix=-500), ["--kappa"], "physical pixels"),
    "zs above the ini's": ({}, ["--kappa-zs", "0.1,0.3"], "outside (0, 0.2]"),
    "zs not positive": ({}, ["--kappa-zs", "0"], "outside (0, 0.2]"),
    "nine sources": ({}, ["--kappa-zs", ",".join(str(0.02 * (i + 1)) for i in range(9))], "at most 8"),
    "no planes alone": ({}, ["--no-planes"], "--no-planes"),
    "non-flat": ({}, ["--kappa"], "not flat"),
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


def gpus():
    try:
        return capi.device_count()
    except capi.SlicerError:  # no CUDA device on this machine
        return 0


@pytest.mark.parametrize("given,refused", [("0.7", False), ("0.7000001", True)])
def test_the_ini_source_redshift_given_as_a_number(tmp_path, given, refused):
    """Entry 2 is read as a float (0.7 -> 0.699999988): the same value given to --kappa-zs is accepted, anything beyond that float
    refused.  (Without a GPU an accepted run stops later, at the device.)"""
    snapdir, lst = make_dataset(tmp_path, ng=8, nsnap=2, numfiles=1)
    assert float(np.float32(0.7)) < 0.7
    out = tmp_path / "out"
    out.mkdir()
    ini = tmp_path / "a.ini"
    ini.write_text(ini_text(lst, snapdir, str(out) + "/t_", zs=0.7, fov=2.0, npix=32))
    r = run_exe(["--kappa-zs", given, ini], tmp_path, quiet=False, timeout=300)
    assert ("outside (0, 0.7]" in r.stderr) == refused, r.stderr
    if refused:
        assert r.returncode != 0 and os.listdir(out) == []
    elif gpus() > 0:
        assert r.returncode == 0, r.stderr[-3000:]
        assert any(".kappa_32_zs0.7000_0.fits" in f for f in os.listdir(out))


# ---- GPU: the library against numpy ------------------------------------------------------------------------------------------
def deposit_random_slots(s, npix, nslots, n, seed, types=(1,)):
    """nslots planes of two randomisations into slots 0 .. nslots-1, particles of `types` -> int64 planes summed over the types"""
    planes = random_planes(seed_triples(2, seed), [(8.0 + 24.0 * i, 32.0 + 24.0 * i, 0.0) for i in range(nslots // 2)], 0.5, npix)
    s.begin_snapshot(BOX, [0, 1.0375, 0, 0, 0.5, 0], False)
    for t in types:
        s.stage(t, synth.uniform_positions(n, BOX, seed + t))
    s.deposit_slots([desc(p, npix) for p in planes], 0)
    return [s.fetch_fixed(q, -1, npix).reshape(-1) for q in range(nslots)]


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["even", "odd", "per_type", "two_realisations", "zero_coefficients"])
def test_library_maps_equal_numpy_bit_for_bit(case):
    npix = 63 if case == "odd" else 64
    n, nslots, nsrc = 1 << 18, 8, 3
    rng = np.random.default_rng(7)
    scale = rng.uniform(1e-6, 1e-3, (nslots, nsrc))
    offset = -rng.uniform(1e-6, 1e-3, (nslots, nsrc))
    if case == "zero_coefficients":
        scale[2, :] = offset[2, :] = 0.0  # a plane beyond every source
        scale[5, 1] = offset[5, 1] = 0.0  # beyond one
    maps = [0] * nslots if case != "two_realisations" else [0] * (nslots // 2) + [nsrc] * (nslots // 2)
    nmaps = max(maps) + nsrc
    per_type = case == "per_type"
    with capi.Slicer(npix_max=npix, max_planes=nslots, particle_capacity=2 * n + 64, per_type_maps=per_type) as s:
        fb = s.frac_bits
        acc = deposit_random_slots(s, npix, nslots, n, 300, types=(1, 4) if per_type else (1,))
        assert all(a.sum() > 0 for a in acc)
        s.kappa_maps(nmaps, npix)
        l0 = s.stats().launches
        # two calls: the second adds to what the first left (slots 0-3, then 4-7)
        s.kappa_add(0, maps[:4], scale[:4], offset[:4])
        s.kappa_add(4, maps[4:], scale[4:], offset[4:])
        assert s.stats().launches == l0 + 2
        got = [s.kappa_fetch(m).reshape(-1) for m in range(nmaps)]
    for m in range(nmaps):
        js = [j for j in range(nslots) if maps[j] <= m < maps[j] + nsrc]
        k = m - maps[js[0]]
        want = numpy_kappa([acc[j] for j in js], scale[js, k], offset[js, k], fb)
        assert np.array_equal(got[m].view(np.uint64), want.view(np.uint64)), (case, m)
        assert np.count_nonzero(got[m]) > 0


@pytest.mark.gpu
def test_library_maps_after_a_two_gpu_reduce():
    if capi.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    npix, n, nslots = 64, 1 << 17, 4
    scale = np.array([[2e-4], [3e-4], [5e-4], [7e-4]])
    offset = -scale / 3
    hs = [capi.Slicer(npix_max=npix, max_planes=nslots, particle_capacity=n + 64, device=d) for d in range(2)]
    try:
        arr = (C.c_void_p * 2)(*[s.h.value for s in hs])
        capi._check(capi.lib().slicer_comm_init_all(arr, 2))
        planes = random_planes(seed_triples(2, 40), [(8.0, 40.0, 0.0), (40.0, 90.0, 0.0)], 0.5, npix)
        per_gpu = []
        for r, s in enumerate(hs):
            s.begin_snapshot(BOX, [0, 1.0375, 0, 0, 0, 0], False)
            s.stage(1, synth.uniform_positions(n, BOX, 60 + r))
            s.deposit_slots([desc(p, npix) for p in planes], 0)
        for r, s in enumerate(hs):
            per_gpu.append([s.fetch_fixed(q, -1, npix).reshape(-1) for q in range(nslots)])
        capi._check(capi.lib().slicer_reduce_all_slots(arr, 2, 0, nslots, 0))
        hs[0].kappa_maps(1, npix)
        hs[0].kappa_add(0, [0] * nslots, scale, offset)
        got = hs[0].kappa_fetch(0).reshape(-1)
        fb = hs[0].frac_bits
    finally:
        for s in hs:
            s.close()
    want = numpy_kappa([per_gpu[0][q] + per_gpu[1][q] for q in range(nslots)], scale[:, 0], offset[:, 0], fb)
    assert np.array_equal(got.view(np.uint64), want.view(np.uint64))


@pytest.mark.gpu
def test_checked_build_traps_nothing_in_the_kappa_kernel():
    """The library tests above against libslicer_b200_chk.so (SLICER_CHECK bounds assertions in kappa_add_kernel)."""
    chk = os.path.join(ROOT, "slicer_b200", "_build", "libslicer_b200_chk.so")
    if not os.path.exists(chk):
        pytest.skip("checked build not present (python -c 'import __graft_entry__ as g; g.build()')")
    r = subprocess.run([sys.executable, "-m", "pytest", os.path.abspath(__file__), "-x", "-q", "-m", "gpu", "-k", "library_maps", "-p",
                        "no:cacheprovider"], env=dict(os.environ, SLICER_B200_LIB=chk), cwd=ROOT, capture_output=True, text=True)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-2000:]


# ---- GPU: the driver ---------------------------------------------------------------------------------------------------------
def kappa_files(root):
    return sorted(f for f in tree(root) if ".kappa_" in f)


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["tsc", "ngp", "hydro_per_type", "degrade"])
def test_driver_maps_equal_numpy_on_its_own_planes(tmp_path, case):
    """The κ FITS of a 64^2 light cone against numpy κ from the same run's float plane files and the plan's weights: within
    1e-6 of the sum of |terms| per pixel (the planes are float32 roundings of the integer sums)."""
    nsnap, zs, fov, npix = 4, 0.2, 6.0, 64
    snapdir, lst = make_dataset(tmp_path, nsnap=nsnap, numfiles=2, hydro=case == "hydro_per_type")
    out = tmp_path / "out"
    out.mkdir()
    ini = tmp_path / "a.ini"
    ini.write_text(ini_text(lst, snapdir, str(out) + "/t_", npix=npix, zs=zs, fov=fov, pip=1 if case == "hydro_per_type" else 0,
                            snopt=1 if case == "degrade" else 0))
    zs_list = [0.2, 0.1]
    r = run_exe([*(["--ngp"] if case == "ngp" else []), "--kappa-zs", "0.2,0.1", ini], tmp_path)
    assert r.returncode == 0, r.stderr[-3000:]
    check_maps_against_planes(out, nsnap, zs, zs_list, fov, npix, per_type=case == "hydro_per_type")


def check_maps_against_planes(out, nsnap, zs, zs_list, fov, npix, per_type=False):
    """Every κ map of `out` against numpy κ from the same run's plane files (snapshots z = 0.1 i of 128 Mpc/h boxes)"""
    # (the ini's zs is read as a float: the plan's distance table is built for float(zs), and its getDl depends on that)
    w = host.kappa_weights(0.3, 0.7, -1.0, float(np.float32(zs)), [0.1 * i for i in range(nsnap)], [128000.0] * nsnap, fov, npix, zs_list)
    files = os.listdir(out)
    for k, z in enumerate(zs_list):
        hdr, got = host.read_fits(str(out / f"t_gadget.kappa_{npix}_zs{z:.4f}_0.fits"))
        h = hdr["HUBBLE"]
        assert hdr["ZSOURCE"] == z and hdr["NPLANES"] == np.count_nonzero(w["scale"][:, k])
        assert abs(hdr["DS"] - w["chis"][k] / h) <= 1e-9 * hdr["DS"] and hdr["PHYSICALSIZE"] == fov
        want, bound = np.zeros((npix, npix)), np.zeros((npix, npix))
        for i in range(len(w["ld"])):
            if w["scale"][i, k] == 0:
                continue
            if per_type:
                mass = np.zeros((npix, npix))
                for f in files:
                    if f.startswith(f"t_gadget.{i:03d}.ptype"):
                        ph, img = host.read_fits(str(out / f))
                        mass += img
            else:
                ph, mass = host.read_fits(str(out / f"t_gadget.{i:03d}.plane_{npix}_0.fits"))
            assert abs(ph["DlLOW"] * h - w["ld"][i]) <= 1e-9 * w["ld2"][i]
            term = w["scale"][i, k] * mass.astype(np.float64) + w["offset"][i, k]
            want += term
            bound += np.abs(term)
        assert np.all(np.abs(got - want) <= 1e-6 * bound), np.max(np.abs(got - want) / bound)
        assert np.std(got) > 0


@pytest.mark.gpu
def test_maps_survive_a_rebuild_of_the_handles(tmp_path):
    """The last snapshot's sub-files hold more particles than the staging pools sized from the first: the driver rebuilds the
    handles before that snapshot (ensure_capacity) and carries the partial maps over (slicer_kappa_fetch / slicer_kappa_load).
    The maps still equal numpy κ from the run's own planes."""
    nsnap, zs, fov, npix, box = 3, 0.2, 6.0, 64, 128000.0  # (the list ends at the first snapshot at the source: z = 0.2)
    snapdir = tmp_path / "snaps"
    names = []
    for i in range(nsnap):
        ng = 64 if i == nsnap - 1 else 24  # 131072 particles per sub-file against pools for 6912 * 5/4 + 65536
        synth.write_snapshot(str(snapdir / f"snap_{i:03d}"), {1: synth.uniform_positions(ng ** 3, box, 1000 + i)}, [0, 1.0375, 0, 0, 0, 0],
                             0.1 * i, box, numfiles=2)
        names.append(f"snap_{i:03d}")
    lst = tmp_path / "snapshot_list.txt"
    lst.write_text("\n".join(names))
    out = tmp_path / "out"
    out.mkdir()
    ini = tmp_path / "a.ini"
    ini.write_text(ini_text(str(lst), str(snapdir) + "/", str(out) + "/t_", npix=npix, zs=zs, fov=fov))
    r = subprocess.run([host.EXE_PATH, "--quiet", "--kappa-zs", "0.2,0.1", str(ini)], cwd=tmp_path, capture_output=True, text=True, timeout=900,
                       env=dict(os.environ, SLICER_B200_TIMING="1"))
    assert r.returncode == 0, r.stderr[-3000:]
    assert r.stderr.count("[timing] slicer_create(") >= 2, r.stderr[-3000:]  # the handles were made again
    planes = open(out / "t_planes_list_0.txt").read().split()
    assert f"snap_{nsnap - 1:03d}" in planes  # the large snapshot feeds planes
    check_maps_against_planes(out, nsnap, zs, [0.2, 0.1], fov, npix)


def byte_identity_case(tmp_path, case):
    snapdir, lst = make_dataset(tmp_path, ng=40, nsnap=3, numfiles=4)
    kz = ["--kappa-zs", "0.1,0.05"]

    def inis(tag, count=2):
        return realisation_inis(tmp_path, tag, lst, snapdir, count, zs=0.1)

    base = inis("base")
    r = run_exe([*kz, *base], tmp_path)
    assert r.returncode == 0, r.stderr[-3000:]
    ref = tree(tmp_path / "base")
    if case == "no_planes":
        other = inis("other")
        r = run_exe([*kz, "--no-planes", *other], tmp_path)
        got = tree(tmp_path / "other")
        assert not any(f.endswith(".fits") and ".kappa_" not in f for f in got)
        lists = [f for f in ref if "planes_list" in f]
        assert len(lists) == 2 and {f for f in got if "planes_list" in f} == set(lists)
        assert all(got[f] == ref[f] for f in lists)
    elif case == "separately":
        for ini in inis("other"):
            r = run_exe([*kz, ini], tmp_path)
            assert r.returncode == 0, r.stderr[-3000:]
        got = tree(tmp_path / "other")
    elif case == "max_slots":
        r = run_exe([*kz, "--max-slots", "3", *inis("other")], tmp_path)
        got = tree(tmp_path / "other")
    elif case == "two_gpus":
        if capi.device_count() < 2:
            pytest.skip("needs 2 GPUs")
        r = run_exe([*kz, "--gpus", "0,1", *inis("other")], tmp_path)
        got = tree(tmp_path / "other")
    else:  # two processes of one job, one GPU each
        if capi.device_count() < 2:
            pytest.skip("needs 2 GPUs")
        from test_multiprocess import run_job

        res = run_job(inis("other"), tmp_path, [[0], [1]], extra=kz)
        assert all(rc == 0 for rc, _, _ in res), [e[-2000:] for _, _, e in res]
        got = tree(tmp_path / "other")
    if case not in ("two_procs",):
        assert r.returncode == 0, r.stderr[-3000:]
    kf = [f for f in ref if ".kappa_" in f]
    assert len(kf) == 4
    assert all(got[f] == ref[f] for f in kf), [f for f in kf if got.get(f) != ref[f]]
    return ref, got


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["no_planes", "separately", "max_slots", "two_gpus", "two_procs"])
def test_kappa_files_are_byte_identical(tmp_path, case):
    ref, got = byte_identity_case(tmp_path, case)
    if case != "no_planes":
        assert got == ref  # planes too


@pytest.mark.gpu
@pytest.mark.parametrize("sources", [["--kappa"], ["--kappa-zs", "0.1,0.05"]])
def test_resume(tmp_path, sources):
    """Two light cones with one or two maps each.  All maps present: nothing is read or deposited.  One map of the second light
    cone gone: that light cone is deposited again and only the missing map is written, bit for bit as before; its other map and
    every plane file keep their bytes and modification times."""
    snapdir, lst = make_dataset(tmp_path, ng=24, nsnap=3, numfiles=2)
    inis = realisation_inis(tmp_path, "out", lst, snapdir, 2, npix=32, zs=0.1, fov=5.0)
    S = 1 if sources == ["--kappa"] else 2
    assert run_exe([*sources, *inis], tmp_path).returncode == 0
    before = tree(tmp_path / "out")
    stamp = {f: os.stat(tmp_path / "out" / f).st_mtime_ns for f in before}
    kf = sorted(f for f in before if ".kappa_" in f)
    assert len(kf) == 2 * S
    r = run_exe([*sources, *inis], tmp_path, quiet=False)
    assert r.returncode == 0, r.stderr[-3000:]
    assert " sub-file " not in r.stdout and r.stdout.count(".kappa_") == 2 * S
    assert tree(tmp_path / "out") == before
    gone = [f for f in kf if f.endswith("_r1.fits")][-1]
    os.remove(tmp_path / "out" / gone)
    r = run_exe([*sources, *inis], tmp_path, quiet=False)
    assert r.returncode == 0, r.stderr[-3000:]
    assert " sub-file " in r.stdout
    assert r.stdout.count(" Already exists") == sum(f.endswith(".fits") for f in before) - 1
    assert tree(tmp_path / "out") == before
    rewritten = {f for f in before if f.endswith(".fits") and os.stat(tmp_path / "out" / f).st_mtime_ns != stamp[f]}
    assert rewritten == {gone}


@pytest.mark.gpu
def test_uniform_universe_has_zero_mean_convergence(tmp_path):
    """Uniform snapshots whose particle mass makes the mean density Omega_m rho_c: the mean κ over interior pixels is 0 within 5
    sigma, sigma^2 = sum_i (scale_i m)^2 N_i / (P P_int) the Poisson noise of the mean of the plane masses (N_i = nparttype1 of
    plane i, P = npix^2 pixels, P_int interior ones), plus 0.2 % of the mean term for the cos(dec) of the flat-sky pixel area.
    A unit slip of h moves the mean by 30 % of sum_i |offset_i| (several times 5 sigma), one of 1e3 by orders of magnitude more."""
    ng, box, om0, nsnap, npix, zs, fov = 96, 128000.0, 0.3, 4, 64, 0.2, 6.0
    m = om0 * RHO_C * (box / 1e3) ** 3 / ng ** 3
    snapdir = tmp_path / "snaps"
    names = []
    for i in range(nsnap):
        synth.write_snapshot(str(snapdir / f"snap_{i:03d}"), {1: synth.uniform_positions(ng ** 3, box, 77 + i)}, [0, m, 0, 0, 0, 0], 0.1 * i, box,
                             numfiles=2, om0=om0, oml=1 - om0)
        names.append(f"snap_{i:03d}")
    lst = tmp_path / "snapshot_list.txt"
    lst.write_text("\n".join(names))
    out = tmp_path / "out"
    out.mkdir()
    ini = tmp_path / "a.ini"
    ini.write_text(ini_text(str(lst), str(snapdir) + "/", str(out) + "/t_", npix=npix, zs=zs, fov=fov))
    r = run_exe(["--kappa", ini], tmp_path)
    assert r.returncode == 0, r.stderr[-3000:]
    w = host.kappa_weights(om0, 1 - om0, -1.0, float(np.float32(zs)), [0.1 * i for i in range(nsnap)], [box] * nsnap, fov, npix,
                           [float(np.float32(zs))])
    _, kappa = host.read_fits(str(out / f"t_gadget.kappa_{npix}_zs{zs:.4f}_0.fits"))
    interior = kappa[2:-2, 2:-2].astype(np.float64)
    P, Pint = npix * npix, interior.size
    var, mean_term = 0.0, 0.0
    for i in range(len(w["ld"])):
        if w["scale"][i, 0] == 0:
            continue
        hdr, _ = host.read_fits(str(out / f"t_gadget.{i:03d}.plane_{npix}_0.fits"))
        var += (w["scale"][i, 0] * m) ** 2 * hdr["nparttype1"] / (P * Pint)
        mean_term += abs(w["offset"][i, 0])
    sigma = np.sqrt(var) + 2e-3 * mean_term
    mean = interior.mean()
    assert abs(mean) < 5 * sigma, (mean, sigma, mean_term)
    assert 5 * sigma < 0.15 * mean_term  # a unit slip of h (30 % of the mean term) or 1e3 is far outside the band
