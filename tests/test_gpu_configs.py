"""Parity at the shapes BASELINE.json states (SURVEY.md §8d): C1 / C2 end to end through the driver against the reference
executable, and one sub-file x one plane group at the C3, C4 and C5 geometries against the oracle (the reference's CPU path needs
~130 ns per particle and plane, so the full 1024^3 / 2048^3 light cones are checked through these windows and through the
bench's self-checks).  All tests need a B200."""
import os
import subprocess

import numpy as np
import pytest

import fits_standard
from slicer_b200 import capi, host, synth
from test_gpu_driver import INI, REF_EXE, REF_EXE_NGP, read_shim_fits

pytestmark = pytest.mark.gpu
LENS_PER_SNAP = 4


def _light_cone_planes(box, fov_deg, ngroups):
    """Plane parameters of a light cone of piled boxes (the plan arithmetic of bench.py, from the product's C++ plan stage)."""
    import bench

    _, raw = bench.c3_planes(box, 64, fov_deg, ngroups)  # npix is not part of the raw parameters
    return raw


@pytest.mark.parametrize("mas", ["tsc", "ngp"])
def test_c1_c2_example_light_cone_matches_reference_executable(tmp_path, mas):
    """BASELINE.json configs[0] (C1) and configs[1] (C2, DO_NGP): the shape of examples/InputParams.ini — box 128 Mpc/h, 7 snapshots
    z = 0 .. 0.6, 256^2 map, 2 deg, zs = 0.5, seeds -229/-230/-231, 42 planes — with 128^3 particles per snapshot (the reference
    executable needs ~15 s for them; 256^3 takes it two minutes: tests/e2e_c1.py).  Every plane of SLICER_b200 against the
    reference executable's: keys, pixels within 1e-6 (TSC), identical pixel counts (NGP), identical planes_list."""
    exe = REF_EXE if mas == "tsc" else REF_EXE_NGP
    if not os.path.exists(exe):
        pytest.skip("reference executable not built (oracle/Makefile)")
    ng, box = 128, 128000.0
    snapdir = tmp_path / "snaps"
    names = []
    for i in range(7):
        synth.write_snapshot(str(snapdir / f"snap_{i:03d}"), {1: synth.hash_positions(ng ** 3, box, 1000 + i)}, [0, 1.0375, 0, 0, 0, 0], 0.1 * i,
                             box, numfiles=4)
        names.append(f"snap_{i:03d}")
    lst = tmp_path / "snapshot_list.txt"
    lst.write_text("\n".join(names))
    outs = {}
    for tag, cmd in (("ref", [exe]), ("gpu", [host.EXE_PATH, "--quiet"] + (["--ngp"] if mas == "ngp" else []))):
        out = tmp_path / f"out_{tag}"
        out.mkdir()
        ini = tmp_path / f"{tag}.ini"
        ini.write_text(INI.format(npix=256, zs=0.5, fov=2.0, list=str(lst), snapdir=str(snapdir) + "/", outdir=str(out) + "/test_", pip=0, snopt=0))
        r = subprocess.run(cmd + [str(ini)], cwd=tmp_path, capture_output=True, text=True, timeout=1500)
        assert r.returncode == 0, r.stderr[-2000:]
        outs[tag] = out
    files = sorted(f for f in os.listdir(outs["ref"]) if f.endswith(".fits"))
    assert files == sorted(f for f in os.listdir(outs["gpu"]) if f.endswith(".fits")) and len(files) == 42
    assert open(outs["ref"] / "test_planes_list_0.txt").read() == open(outs["gpu"] / "test_planes_list_0.txt").read()
    m = np.float32(1.0375)
    accepted = 0
    for f in files:
        rk, rimg = read_shim_fits(outs["ref"] / f)
        hdr, rows = fits_standard.read_primary_image(str(outs["gpu"] / f))  # the independent, standard-driven reader
        gimg = np.array(rows, np.float32)
        assert gimg.shape == rimg.shape == (256, 256)
        for k in ("REDSHIFT", "PHYSICALSIZE", "PIXELUNIT", "DlLOW", "DlUP", "HUBBLE", "OMEGAMATTER", "OMEGALAMBDA", "m1"):
            assert hdr[k] == rk[k], (f, k)
        assert hdr["DLLOW"] == rk["DlLOW"] and hdr["NAXIS1"] == 256  # as Lens/kslicer.py:39-40,84-86 spells them
        if mas == "ngp":
            assert np.array_equal(np.rint(gimg / m), np.rint(rimg / m)), f  # identical pixel indices <=> identical counts per pixel
            assert hdr["nparttype1"] >= int(np.rint(gimg / m).sum())        # in-grid hits <= accepted pairs
        np.testing.assert_allclose(gimg, rimg, rtol=1e-6, atol=1e-9)
        accepted += hdr["nparttype1"]
    assert accepted > 200_000


def _oracle_group(oracle, pos, planes, npix, massarr1, frac_bits, do_ngp=False):
    """One sub-file through the oracle for each plane of a group -> list of (counts[6], ingrid[6], fixed int64 map)."""
    out = []
    for p in planes:
        x, y, z = oracle.transform(pos, p["boxsize"], p["sgn"], p["face"], p["centre"], p["rcase"])
        xs, ys, ms = oracle.select_project(x, y, z, p["ld"], p["ld2"], p["boxsize"], 0, p["fovradiants"], npix, const_mass=massarr1,
                                           cap=len(x) + 16)
        fixed = oracle.gridist_w_fixed(xs, ys, ms, npix, frac_bits, do_ngp)
        cells = oracle.ngp_cells_fast(xs, ys, npix)
        out.append((len(xs), int(np.count_nonzero(cells >= 0)), fixed))
    return out


@pytest.mark.parametrize("name,box,npix,ngroups,group", [("C3", 256000.0, 2048, 9, 8), ("C3", 256000.0, 2048, 9, 2), ("C5", 1000000.0, 8192, 6, 5)])
def test_one_subfile_at_c3_and_c5_geometry_matches_oracle(oracle, name, box, npix, ngroups, group):
    """SURVEY.md §8(d): 'one sub-file x one plane' parity at the C3 (2048^2, 5 deg) and C5 (8192^2, 5 deg, piled boxes) geometries:
    a 2^22-particle window of the bench's synthetic snapshot through the production path (AUTO: binned for these groups; at
    8192^2 the four planes sort by groups of two tiles in a single window of 5000 bins) and through the forced-direct path, all
    four planes of the group against the oracle: accepted counts, in-grid counts and int64 maps bit for bit.  The windowed
    sorts and groups of four are held to the oracle in test_gpu_binned_regimes.py."""
    n = 1 << 22
    mass = 5.2
    raw = _light_cone_planes(box, 5.0, ngroups)[group * LENS_PER_SNAP:(group + 1) * LENS_PER_SNAP]
    descs = [capi.plane_desc(p["sgn"], p["face"], p["centre"], p["rcase"], p["ld"], p["ld2"], p["fovradiants"], npix) for p in raw]
    pos = synth.hash_positions(n, box, 1000)
    want = None
    for mode in (capi.DEPOSIT_AUTO, capi.DEPOSIT_BINNED, capi.DEPOSIT_DIRECT):
        with capi.Slicer(npix_max=npix, max_planes=LENS_PER_SNAP, mas=capi.MAS_TSC, particle_capacity=n + 64, deposit_mode=mode) as s:
            s.begin_snapshot(box, [0, mass, 0, 0, 0, 0], False)
            s.stage(1, pos)
            s.deposit(descs)
            if want is None:
                want = _oracle_group(oracle, pos, raw, npix, mass, s.frac_bits)
                assert sum(w[0] for w in want) > (900_000 if group >= 5 else 150_000)
            for k in range(LENS_PER_SNAP):
                _, counts, ingrid = s.fetch(k, -1, npix, want_map=False)
                assert (int(counts[1]), int(ingrid[1])) == want[k][:2], (name, mode, k)
                assert np.array_equal(s.fetch_fixed(k, -1, npix).reshape(-1), want[k][2]), (name, mode, k)


def test_c4_shape_three_species_per_type_maps_match_oracle(oracle):
    """BASELINE.json configs[3] (C4) at the createDensityMaps output (SURVEY.md §8a row 12): gas / DM / stars in one sub-file, per-particle
    masses for gas and stars with ~1 % above MAX_M (counted, deposited as 0), Part. in Planes = 1 (one map per type), 1024^2 map,
    the four planes of a dense C3-geometry group in one pass: per-type counts and int64 maps against the oracle."""
    box, npix, n = 256000.0, 1024, 1 << 20
    raw = _light_cone_planes(box, 5.0, 9)[7 * LENS_PER_SNAP:8 * LENS_PER_SNAP]
    descs = [capi.plane_desc(p["sgn"], p["face"], p["centre"], p["rcase"], p["ld"], p["ld2"], p["fovradiants"], npix) for p in raw]
    rng = np.random.default_rng(9)
    types = []
    for k, ty in enumerate((0, 1, 4)):
        t = dict(type=ty, raw=synth.hash_positions(n, box, 4000 + k))
        if ty == 1:
            t["const_mass"] = 5.2
        else:
            m = (rng.random(n, dtype=np.float32) * 2 + 0.05).astype(np.float32)
            m[::100] = 2000.0
            t["masses"] = m
        types.append(t)
    for mode in (capi.DEPOSIT_AUTO, capi.DEPOSIT_DIRECT):
        with capi.Slicer(npix_max=npix, max_planes=LENS_PER_SNAP, mas=capi.MAS_TSC, particle_capacity=3 * n + 64, mass_capacity=3 * n + 64,
                         per_type_maps=True, deposit_mode=mode) as s:
            s.begin_snapshot(box, [0, 5.2, 0, 0, 0, 0], True)
            for t in types:
                s.stage(t["type"], t["raw"], t.get("masses"))
            s.deposit(descs)
            fb = s.frac_bits
            for k, p in enumerate(raw):
                res = oracle.plane_from_particles(types, p, npix, frac_bits=fb)
                _, counts, ingrid = s.fetch(k, -1, npix, want_map=False)
                assert counts.tolist() == res["counts"].tolist() and ingrid.tolist() == res["ingrid"].tolist()
                assert counts[0] > 100_000 and counts[4] > 100_000
                for t in types:
                    assert np.array_equal(s.fetch_fixed(k, t["type"], npix).reshape(-1), res["fixed"][t["type"]]), (mode, k, t["type"])
