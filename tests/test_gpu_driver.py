"""End to end on a B200: the C++ driver (SLICER_b200: ini -> plan -> GADGET-2 sub-files -> CUDA passes -> FITS planes)
against the reference's own executable (oracle/_ref/SLICER_ref, the unmodified sources built by oracle/Makefile) on the
same synthetic snapshots and the same InputParams.ini."""
import os
import subprocess

import numpy as np
import pytest

from slicer_b200 import host, synth

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF_EXE = os.path.join(ROOT, "oracle", "_ref", "SLICER_ref")
REF_EXE_NGP = os.path.join(ROOT, "oracle", "_ref", "SLICER_ref_ngp")

INI = """##### 1. Number of Map Pixels ##
{npix}
##### 2. Source Redshift #######
{zs}
##### 3. Field of View #########
{fov}
##### 4. File with Snapshots ###
{list}
##### 5. Snapshots Directory ###
{snapdir}
##### 6. PLC Sim. Name #########
gadget
##### 7. Seed for Pos. Center ##
-229
##### 8. Seed for Pos. Reflec. #
-230
##### 9. Seed for Axis Sel. ####
-231
##### 10. Part. in Planes ######
{pip}
##### 11. PLC Directory ########
{outdir}
##### 12. PLC Suffix ###########
0
##### 13. Part. Degradation ####
{snopt}
##### 14. DE-EOS w #############
-1.0
"""


def read_shim_fits(path):
    """The reference build's CCfits stand-in dumps keys as text and then raw float32 pixels (oracle/shim/CCfits/CCfits)."""
    raw = open(path, "rb").read()
    end = raw.index(b"END\n") + 4
    keys, naxis = {}, []
    for line in raw[:end].decode().splitlines():
        parts = line.split("\t")
        if line.startswith("NAXIS") and " " in line and not line.startswith("NAXIS "):
            naxis.append(int(line.split()[1]))
        if parts[0].startswith("KEY "):
            keys[parts[0][4:]] = float(parts[2])
    img = np.frombuffer(raw, dtype="<f4", offset=end).reshape(naxis[1], naxis[0])
    return keys, img


def make_dataset(tmp_path, ng=48, nsnap=4, numfiles=2, hydro=False):
    box = 128000.0
    snapdir = tmp_path / "snaps"
    names = []
    for i in range(nsnap):
        n = ng ** 3
        if hydro:
            rng = np.random.default_rng(50 + i)
            pos = {0: synth.uniform_positions(n // 2, box, 1000 + i), 1: synth.uniform_positions(n // 2, box, 2000 + i),
                   4: synth.uniform_positions(n // 8, box, 3000 + i)}
            masses = {0: (rng.random(n // 2) * 0.3).astype(np.float32), 4: (rng.random(n // 8) * 2).astype(np.float32)}
            masses[4][::13] = 5e3  # above MAX_M: counted, deposited with mass 0
            synth.write_snapshot(str(snapdir / f"snap_{i:03d}"), pos, [0, 1.0375, 0, 0, 0, 0], 0.1 * i, box, numfiles=numfiles, masses=masses)
        else:
            synth.write_snapshot(str(snapdir / f"snap_{i:03d}"), {1: synth.uniform_positions(n, box, 1000 + i)}, [0, 1.0375, 0, 0, 0, 0],
                                 0.1 * i, box, numfiles=numfiles)
        names.append(f"snap_{i:03d}")
    lst = tmp_path / "snapshot_list.txt"
    lst.write_text("\n".join(names))  # no trailing newline (SURVEY.md App. C)
    return str(snapdir) + "/", str(lst)


def run_both(tmp_path, npix, zs, fov, ref_exe, extra=(), pip=0, hydro=False, numfiles=2, snopt=0):
    snapdir, lst = make_dataset(tmp_path, hydro=hydro, numfiles=numfiles)
    outs = {}
    for tag, exe in (("ref", [ref_exe]), ("gpu", [host.EXE_PATH, "--quiet", *extra])):
        out = tmp_path / f"out_{tag}"
        out.mkdir()
        ini = tmp_path / f"InputParams_{tag}.ini"
        ini.write_text(INI.format(npix=npix, zs=zs, fov=fov, list=lst, snapdir=snapdir, outdir=str(out) + "/test_", pip=pip, snopt=snopt))
        r = subprocess.run(exe + [str(ini)], cwd=tmp_path, capture_output=True, text=True, timeout=900)
        assert r.returncode == 0, r.stderr[-2000:] + r.stdout[-2000:]
        outs[tag] = out
    return outs


@pytest.mark.parametrize("mas", ["tsc", "ngp"])
def test_driver_matches_reference_executable(tmp_path, mas):
    if not os.path.exists(REF_EXE):
        pytest.skip("oracle/_ref/SLICER_ref not built")
    outs = run_both(tmp_path, 64, 0.2, 6.0, REF_EXE if mas == "tsc" else REF_EXE_NGP, extra=("--ngp",) if mas == "ngp" else ())
    ref_files = sorted(f for f in os.listdir(outs["ref"]) if f.endswith(".fits"))
    gpu_files = sorted(f for f in os.listdir(outs["gpu"]) if f.endswith(".fits"))
    assert ref_files == gpu_files and len(ref_files) >= 16
    # planes_list: identical text (same plan, same formatting)
    assert open(outs["ref"] / "test_planes_list_0.txt").read() == open(outs["gpu"] / "test_planes_list_0.txt").read()
    total = 0.0
    for f in ref_files:
        rk, rimg = read_shim_fits(outs["ref"] / f)
        gk, gimg = host.read_fits(str(outs["gpu"] / f))
        assert gimg.shape == rimg.shape == (64, 64)
        for k in ("REDSHIFT", "PHYSICALSIZE", "PIXELUNIT", "DlLOW", "DlUP", "HUBBLE", "OMEGAMATTER", "OMEGALAMBDA", "m1"):
            assert gk[k] == rk[k], (f, k)
        if mas == "ngp":
            # NGP with one constant particle mass: pixel = count * m; identical pixel indices <=> identical counts
            assert np.array_equal(np.rint(gimg / np.float32(1.0375)), np.rint(rimg / np.float32(1.0375))), f
        np.testing.assert_allclose(gimg, rimg, rtol=1e-6, atol=1e-9)
        assert gk["nparttype1"] >= np.count_nonzero(rimg) / 9  # real counts (the reference always writes 0 here)
        total += float(rimg.sum(dtype=np.float64))
    assert total > 100.0


def test_driver_hydro_per_type_files(tmp_path):
    """C4 shape: gas / DM / stars with per-particle masses, Part. in Planes = 1.  The shipped reference writes no FITS in
    this mode (densitymaps.cpp:497 shadows the counts, :593 gates on them), so parity is checked against its total map
    (partinplanes = 0 run of the reference) = sum of our per-type files."""
    if not os.path.exists(REF_EXE):
        pytest.skip("oracle/_ref/SLICER_ref not built")
    snapdir, lst = make_dataset(tmp_path, hydro=True, numfiles=3)
    out_ref, out_gpu = tmp_path / "out_ref", tmp_path / "out_gpu"
    out_ref.mkdir()
    out_gpu.mkdir()
    ini_ref, ini_gpu = tmp_path / "ref.ini", tmp_path / "gpu.ini"
    ini_ref.write_text(INI.format(npix=128, zs=0.2, fov=6.0, list=lst, snapdir=snapdir, outdir=str(out_ref) + "/test_", pip=0, snopt=0))
    ini_gpu.write_text(INI.format(npix=128, zs=0.2, fov=6.0, list=lst, snapdir=snapdir, outdir=str(out_gpu) + "/test_", pip=1, snopt=0))
    assert subprocess.run([REF_EXE, str(ini_ref)], cwd=tmp_path, capture_output=True, timeout=900).returncode == 0
    r = subprocess.run([host.EXE_PATH, "--quiet", str(ini_gpu)], cwd=tmp_path, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-2000:]
    ref_files = sorted(f for f in os.listdir(out_ref) if f.endswith(".fits"))
    assert len(ref_files) >= 16
    for f in ref_files:
        _, rimg = read_shim_fits(out_ref / f)
        acc = np.zeros_like(rimg, dtype=np.float64)
        ntypes = 0
        for t in range(6):
            g = out_gpu / f.replace(".plane_", f".ptype{t}_plane_")
            if g.exists():
                hk, gimg = host.read_fits(str(g))
                assert hk["nparttype0"] > 0
                acc += gimg
                ntypes += 1
        assert ntypes >= 2 or rimg.sum() == 0
        np.testing.assert_allclose(acc, rimg, rtol=3e-6, atol=1e-8)


def test_driver_resume_skips_existing_planes(tmp_path):
    snapdir, lst = make_dataset(tmp_path, ng=24, nsnap=3, numfiles=1)
    out = tmp_path / "out"
    out.mkdir()
    ini = tmp_path / "p.ini"
    ini.write_text(INI.format(npix=32, zs=0.1, fov=5.0, list=lst, snapdir=snapdir, outdir=str(out) + "/t_", pip=0, snopt=0))
    assert subprocess.run([host.EXE_PATH, "--quiet", str(ini)], cwd=tmp_path, capture_output=True, timeout=600).returncode == 0
    files = sorted(f for f in os.listdir(out) if f.endswith(".fits"))
    assert len(files) >= 8
    keep = {f: open(out / f, "rb").read() for f in files}
    os.remove(out / files[3])
    r = subprocess.run([host.EXE_PATH, str(ini)], cwd=tmp_path, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "Already exists" in r.stdout
    assert {f: open(out / f, "rb").read() for f in files} == keep  # the missing plane is rebuilt bit for bit, the rest untouched


@pytest.mark.parametrize("snopt", [0, 1])
def test_driver_two_gpus_matches_one_gpu(tmp_path, snopt):
    """Sub-files dealt over two GPUs + ncclReduce(int64) of the planes == the single-GPU run, bit for bit
    (integer accumulators make the sum independent of how the particles are sharded), also with Part. Degradation: its two
    sweeps over the sub-files run on both GPUs at once."""
    from slicer_b200 import capi

    if capi.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    snapdir, lst = make_dataset(tmp_path, ng=40, nsnap=3, numfiles=5)
    outs = {}
    for tag, gpus in (("g1", "0"), ("g2", "0,1")):
        out = tmp_path / tag
        out.mkdir()
        ini = tmp_path / f"{tag}.ini"
        ini.write_text(INI.format(npix=64, zs=0.1, fov=6.0, list=lst, snapdir=snapdir, outdir=str(out) + "/t_", pip=0, snopt=snopt))
        r = subprocess.run([host.EXE_PATH, "--quiet", "--gpus", gpus, str(ini)], cwd=tmp_path, capture_output=True, text=True, timeout=900)
        assert r.returncode == 0, r.stderr[-2000:]
        outs[tag] = out
    files = sorted(f for f in os.listdir(outs["g1"]) if f.endswith(".fits"))
    assert len(files) >= 8
    for f in files:
        assert open(outs["g1"] / f, "rb").read() == open(outs["g2"] / f, "rb").read(), f


@pytest.mark.parametrize("snopt,hydro", [(1, False), (2, True)])
def test_driver_part_degradation_matches_reference(tmp_path, snopt, hydro):
    """Part. Degradation = 1, 2: the reference's serial rand() stream (continuing from randomizeBox, plane after plane,
    sub-file after sub-file) is reproduced exactly, so every plane matches the reference executable's."""
    if not os.path.exists(REF_EXE):
        pytest.skip("oracle/_ref/SLICER_ref not built")
    outs = run_both(tmp_path, 64, 0.2, 6.0, REF_EXE, snopt=snopt, hydro=hydro, numfiles=3)
    ref_files = sorted(f for f in os.listdir(outs["ref"]) if f.endswith(".fits"))
    assert ref_files == sorted(f for f in os.listdir(outs["gpu"]) if f.endswith(".fits")) and len(ref_files) >= 16
    total = 0.0
    for f in ref_files:
        _, rimg = read_shim_fits(outs["ref"] / f)
        _, gimg = host.read_fits(str(outs["gpu"] / f))
        np.testing.assert_allclose(gimg, rimg, rtol=1e-6, atol=1e-9)
        total += float(rimg.sum(dtype=np.float64))
    assert total > 100.0


def _compare_dirs(out_ref, out_gpu, npix=None, min_files=8):
    ref_files = sorted(f for f in os.listdir(out_ref) if f.endswith(".fits"))
    assert ref_files == sorted(f for f in os.listdir(out_gpu) if f.endswith(".fits")) and len(ref_files) >= min_files
    total = 0.0
    for f in ref_files:
        rk, rimg = read_shim_fits(out_ref / f)
        gk, gimg = host.read_fits(str(out_gpu / f))
        assert gimg.shape == rimg.shape
        if npix:
            assert rimg.shape == (npix, npix)
        for k in ("REDSHIFT", "DlLOW", "DlUP"):
            assert gk[k] == rk[k]
        np.testing.assert_allclose(gimg, rimg, rtol=1e-6, atol=1e-9)
        total += float(rimg.sum(dtype=np.float64))
    assert total > 50.0
    return ref_files


def test_driver_perpendicular_replication(tmp_path):
    """CMake USE_REPLICATION (-DReplicationOnPerpendicularPlane): a field wider than the box is filled with
    replicas (computeReplications, densitymaps.cpp:275-283; mapParticles' ni, nj loops :377-378)."""
    exe = os.path.join(ROOT, "oracle", "_ref", "SLICER_ref_repl")
    if not os.path.exists(exe):
        pytest.skip("oracle/_ref/SLICER_ref_repl not built")
    outs = run_both(tmp_path, 64, 0.2, 25.0, exe, extra=("--replication",))  # 25 deg at 590 Mpc/h = 257 Mpc/h > 128 Mpc/h box
    _compare_dirs(outs["ref"], outs["gpu"], 64, 16)


def test_driver_fixed_plc_vertex(tmp_path):
    """CMake USE_FIXED_PLC_VERTEX (-DFixedPLCVertex): no random centre shift (densitymaps.cpp:186-196)."""
    exe = os.path.join(ROOT, "oracle", "_ref", "SLICER_ref_fixed")
    if not os.path.exists(exe):
        pytest.skip("oracle/_ref/SLICER_ref_fixed not built")
    outs = run_both(tmp_path, 64, 0.2, 6.0, exe, extra=("--fixed-vertex",))
    _compare_dirs(outs["ref"], outs["gpu"], 64, 16)


def test_driver_physical_pixel_mode(tmp_path):
    """npix < 0: `physical` mode, -npix kpc/h pixels, map side recomputed per plane (data.cpp:64-78, slicer-v2.cpp:142-143)."""
    if not os.path.exists(REF_EXE):
        pytest.skip("oracle/_ref/SLICER_ref not built")
    outs = run_both(tmp_path, -500, 0.2, 6.0, REF_EXE)
    files = _compare_dirs(outs["ref"], outs["gpu"], None, 16)
    assert all("_500_kpc_" in f for f in files)
    sides = {host.read_fits(str(outs["gpu"] / f))[0]["NAXIS1"] for f in files}
    assert len(sides) > 4  # the map grows with distance
