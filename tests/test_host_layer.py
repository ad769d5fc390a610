"""The C++ host layer (slicer_b200/host/): plan, ini parser, GADGET-2 reader and FITS writer.  CPU only: the plan is
pinned bit for bit to the golden vectors generated from the reference build (oracle/make_golden.py)."""
import os

import numpy as np
import pytest

from conftest import unhex
from slicer_b200 import host, synth


def test_cosmo_table_matches_reference(kat):
    for c in kat["cosmo_table"]:
        zl, dl = host.cosmo_table(c["om0"], c["oml"], c["w"], c["zs"])
        assert [zl[i] for i in c["idx"]] == [unhex(v) for v in c["zl"]]
        assert [dl[i] for i in c["idx"]] == [unhex(v) for v in c["dl"]]


def test_plan_matches_reference(kat, tmp_path):
    for pl in kat["plan"]:
        got = host.plan(pl["om0"], pl["oml"], pl["w"], pl["zs"], pl["snapred"], [pl["box"]] * len(pl["snapred"]), str(tmp_path) + "/")
        assert got["nplanes"] == pl["nplanes"]
        assert got["Ds"] == unhex(pl["Ds"])
        for k in ("ld", "ld2", "zsimlens"):
            assert got[k].tolist() == [unhex(v) for v in pl[k]], k
        assert got["fromsnapi"].tolist() == pl["fromsnapi"]
        assert got["randomize"].tolist() == pl["randomize"]
        assert got["replication"].tolist() == pl["replication"]
        # planes_list_<suffix>.txt: column 6 (snapshot name) is what Lens/kslicer.py:29 reads
        rows = [l.split() for l in open(tmp_path / "planes_list_t.txt")]
        assert len(rows) == len(got["ld"]) and rows[0][0] == "0" and rows[0][5].startswith("snap_") and len(rows[0]) == 8
        os.remove(tmp_path / "planes_list_t.txt")


def test_plan_known_answers(tmp_path):
    # SURVEY.md App. A: 7 snapshots z = 0 .. 0.6, L = 128 Mpc/h, zs = 0.5 -> 42 planes, Ds = 1330.6066
    got = host.plan(0.3, 0.7, -1.0, 0.5, [0.0, 0.1, 0.2, 0.3, 0.4, 0.5, 0.6], [128000.0] * 7, str(tmp_path) + "/")
    assert got["nplanes"] == 42 and abs(got["Ds"] - 1330.6066) < 1e-3
    assert (got["ld"][5], got["ld2"][5], got["fromsnapi"][5], got["randomize"][5]) == (160.0, 192.0, 1, 0)
    assert (got["ld"][41], got["ld2"][41], got["fromsnapi"][41]) == (1312.0, 1344.0, 5)


def test_randomize_box_matches_reference(kat, oracle):
    for r in kat["randomize_box"]:
        got = host.randomize_box(*r["seeds"], r["randomize"])
        for k in ("x0", "y0", "z0"):
            assert got[k].tolist() == [unhex(v) for v in r[k]]
        for k in ("face", "sgnX", "sgnY", "sgnZ"):
            assert got[k].tolist() == r[k]
    fv = host.randomize_box(1, 2, 3, [1, 0, 0, 0, 1], fixed_vertex=True)
    assert fv["x0"].tolist() == [0.0] * 5 and fv["z0"].tolist() == [0.5] * 5  # -DFixedPLCVertex (densitymaps.cpp:191-195)
    assert fv["face"].tolist() == oracle.randomize_box(1, 2, 3, [1, 0, 0, 0, 1], fixed_vertex=True)["face"].tolist()


def test_read_input(tmp_path):
    ini = tmp_path / "InputParams.ini"
    ini.write_text("##### 1. Number of Map Pixels ##\n256\n##### 2. Source Redshift #######\n0.5\n##### 3. Field of View #########\n2.1\n"
                   "##### 4. File with Snapshots ###\nsnapshot_list.txt\n##### 5. Snapshots Directory ###\n/data/L128N256/\n"
                   "##### 6. PLC Sim. Name #########\ngadget\n##### 7. Seed for Pos. Center ##\n-229\n##### 8. Seed for Pos. Reflec. #\n-230\n"
                   "##### 9. Seed for Axis Sel. ####\n-231\n##### 10. Part. in Planes ######\n0\n##### 11. PLC Directory ########\n/out/test_\n"
                   "##### 12. PLC Suffix ###########\n0\n##### 13. Part. Degradation ####\n0\n##### 14. DE-EOS w #############\n-1.0\n")
    p = host.read_input(str(ini))
    assert (p["npix"], p["seedcenter"], p["seedface"], p["seedsign"], p["snopt"], p["partinplanes"]) == (256, -229, -230, -231, 0, False)
    assert p["fov"] == float(np.float32(2.1)) and p["zs"] == 0.5 and p["w"] == -1.0  # stof precision (data.cpp:26,29,62)
    assert (p["filredshiftlist"], p["pathsnap"], p["simulation"], p["directory"], p["suffix"], p["snpix"]) == (
        "snapshot_list.txt", "/data/L128N256/", "gadget", "/out/test_", "0", "256")
    ini.write_text(ini.read_text().replace("\n256\n", "\n-50\n", 1))
    q = host.read_input(str(ini))
    assert q["physical"] and q["rgrid"] == 50 and q["snpix"] == "50_kpc"  # data.cpp:64-78


def test_reader_matches_reference_reader(tmp_path, oracle, golden):
    """The GADGET-2 reader against the reference's reader (header, readPos) where the reference build is present, and always
    against what the writer put into the sub-files.  Without the build, against the reference's stored readPos output instead:
    tests/golden/cases.npz holds x, y, z that readPos returned for sub-files written by synth.write_snapshot from the stored
    inputs (oracle/make_golden.py).  The same files are written again here, read with our reader and taken through the box
    transform of the C restatement (itself pinned to those vectors by test_oracle_golden.py)."""
    from oracle import ref_bindings

    reflib = ref_bindings.RefLib(ngp=False) if ref_bindings.available() else None
    if reflib is None:
        for name in golden.names():
            m, plane = golden.meta[name], golden.plane(name)
            tys = golden.types(name)
            masses = {t["type"]: t["masses"] for t in tys if "masses" in t}
            base = str(tmp_path / name)
            synth.write_snapshot(base, {t["type"]: t["raw"] for t in tys}, m["massarr"], 0.0, m["box"], numfiles=1, masses=masses,
                                 bh_masses=masses.get(5))
            s = host.read_subfile(base + ".0", bool(m["hydro"]), sum(len(t["raw"]) for t in tys))
            assert s["npart"].tolist() == [int(m["npart"].get(str(t), 0)) for t in range(6)] and s["boxsize"] == m["box"]
            got = oracle.transform(s["pos"], plane["boxsize"], plane["sgn"], plane["face"], plane["centre"], plane["rcase"])
            for k, key in enumerate("xyz"):
                assert np.array_equal(got[k].view(np.uint32), golden.arr[f"{name}/{key}"].view(np.uint32)), (name, key)
    rng = np.random.default_rng(3)
    box = 75000.0
    pos = {0: synth.uniform_positions(700, box, 1), 1: synth.uniform_positions(900, box, 2), 4: synth.uniform_positions(300, box, 3),
           5: synth.uniform_positions(50, box, 4)}
    masses = {t: rng.random(len(pos[t])).astype(np.float32) for t in (0, 4, 5)}
    bh = rng.random(50).astype(np.float32) + 10
    base = str(tmp_path / "snap_007")
    synth.write_snapshot(base, pos, [0, 0.25, 0, 0, 0, 0], 0.3, box, numfiles=2, masses=masses, bh_masses=bh)
    for ff in range(2):
        s = host.read_subfile(f"{base}.{ff}", True, 4000)
        assert s["numfiles"] == 2
        if reflib is not None:
            ref = reflib.read_header(f"{base}.{ff}")
            assert s["npart"].tolist() == ref["npart"].tolist()
            for k in ("redshift", "boxsize", "om0", "oml", "h", "time"):
                assert s[k] == ref[k]
            # identity transform through the reference's readPos == raw/box
            x, y, z, _ = reflib.read_pos(f"{base}.{ff}", [1, 1, 1], 1, [0.0, 0.0, 0.0], 0.0)
            assert np.array_equal((s["pos"][:, 0].astype(np.float64) / box).astype(np.float32), x)
        off = 0
        for t in range(6):
            n = int(s["npart"][t])
            lo, hi = synth.split_counts(len(pos.get(t, [])), 2)[1][ff: ff + 2] if t in pos else (0, 0)
            if t in pos:
                assert np.array_equal(s["pos"][off: off + n], pos[t][lo:hi])
            if t in (0, 4):
                assert np.array_equal(s["mass"][off: off + n], masses[t][lo:hi])
            if t == 5:
                assert np.array_equal(s["mass"][off: off + n], bh[lo:hi])  # BHMA, not the MASS entries (densitymaps.cpp:361-365)
            if t == 1:
                assert not s["mass"][off: off + n].any()
            off += n


def test_fits_writer_layout(tmp_path):
    img = np.arange(12 * 12, dtype=np.float32).reshape(12, 12) * 0.5
    f = str(tmp_path / "gadget.005.plane_12_0.fits")
    assert host.write_fits(f, img, [("REDSHIFT", 0.0593), ("PHYSICALSIZE", 2.0), ("DlLOW", 228.57142857142858), ("DlUP", 274.0)],
                           [("nparttype1", 1224)]) == 0
    raw = open(f, "rb").read()
    assert len(raw) % 2880 == 0 and raw.startswith(b"SIMPLE  =                    T")
    hdr, back = host.read_fits(f)
    assert (hdr["BITPIX"], hdr["NAXIS"], hdr["NAXIS1"], hdr["NAXIS2"]) == (-32, 2, 12, 12)
    assert hdr["DlLOW"] == 228.57142857142858 and hdr["nparttype1"] == 1224 and hdr["PHYSICALSIZE"] == 2.0
    assert np.array_equal(back, img)  # element [gy, gx] <-> map[gx + npix*gy], big-endian on disk
    assert host.write_fits(f, img, [], []) == 1  # an existing file is not overwritten (FITS::CantCreate)


def test_fits_output_conforms_to_the_standard(tmp_path):
    """The plane files are read by astropy in Lens/kslicer.py:39-40,84-86 (DLLOW, DLUP, PHYSICALSIZE, NAXIS1/2; case-insensitive,
    HIERARCH-transparent).  astropy / CFITSIO are not on this box, so tests/fits_standard.py restates what a conforming reader
    checks (FITS 4.0 + the HIERARCH convention) independently of the repo's own reader, and validates a file with the full key
    set of writeMaps (densitymaps.cpp:563-583), awkward values included."""
    import fits_standard

    rng = np.random.default_rng(3)
    img = (rng.random((37, 37)) * 1e3).astype(np.float32)
    img[0, 0], img[36, 36], img[5, 7] = 0.0, np.float32(3.4e38), np.float32(1e-38)
    dkeys = [("REDSHIFT", 0.059314673648001914), ("PHYSICALSIZE", 2.0), ("PIXELUNIT", 14285714285.714287), ("DlLOW", 228.57142857142858),
             ("DlUP", 274.28571428571428), ("HUBBLE", 0.7), ("OMEGAMATTER", 0.3), ("OMEGALAMBDA", 0.7)] + \
            [(f"m{i}", v) for i, v in enumerate([0.0, 1.0375, 0.0, 0.0, 1e-300, 123456789012.5])]
    ikeys = [(f"nparttype{i}", v) for i, v in enumerate([0, 1224, 0, 0, 2 ** 40, 7])]
    f = str(tmp_path / "gadget.041.plane_37_t.fits")
    assert host.write_fits(f, img, dkeys, ikeys) == 0
    hdr, rows = fits_standard.read_primary_image(f)
    assert (hdr["BITPIX"], hdr["NAXIS"], hdr["NAXIS1"], hdr["NAXIS2"]) == (-32, 2, 37, 37)
    # the keys the consumer reads, the way it spells them
    assert hdr["DLLOW"] == 228.57142857142858 and hdr["DLUP"] == 274.28571428571428 and hdr["PHYSICALSIZE"] == 2.0
    for k, v in dkeys:
        assert hdr[k] == v, k          # %.17G round-trips every double
    for k, v in ikeys:
        assert hdr[k] == v and isinstance(hdr[k], int), k
    assert np.array_equal(np.array(rows, np.float32), img)  # row gy holds map[gx + npix*gy], gx fastest
    # and the repo's own test reader agrees with the independent one
    h2, back = host.read_fits(f)
    assert np.array_equal(back, img) and h2["DlLOW"] == hdr["DLLOW"]


def test_glibc_rand_restatement_matches_libc():
    """slicer::GlibcRand (private state) == libc srand/rand, which the reference uses (densitymaps.cpp:187-223, :393)."""
    from oracle.oracle_bindings import libc_rand, libc_srand

    for seed in (1, 0, -229, -230, -231, 12345, 2 ** 31 - 1, 2 ** 32 - 5):
        libc_srand(seed)
        want = [libc_rand() for _ in range(3000)]
        assert host.glibc_rand(seed, 3000).tolist() == want


def test_reader_parallel_bulk_read(tmp_path):
    """Payloads >= 8 MiB are read by several threads (pread on disjoint ranges): same bytes as the plain read
    (SLICER_B200_IO_THREADS=1, in a fresh process because the thread count is latched), for POS and MASS blocks."""
    import subprocess, sys, textwrap
    box = 100000.0
    n0, n1 = 2_300_000, 1_000_003  # gas MASS block 9.2 MB, POS block 39.6 MB: not multiples of the 1 MiB chunk rounding
    pos = {0: synth.uniform_positions(n0, box, 11), 1: synth.uniform_positions(n1, box, 12)}
    masses = {0: (np.arange(n0, dtype=np.float32) % 977) + 1}
    base = str(tmp_path / "snap_big")
    synth.write_snapshot(base, pos, [0, 0.5, 0, 0, 0, 0], 0.1, box, numfiles=1, masses=masses)
    s = host.read_subfile(f"{base}.0", True, n0 + n1 + 10)
    assert s["npart"].tolist() == [n0, n1, 0, 0, 0, 0]
    assert np.array_equal(s["pos"][:n0], pos[0]) and np.array_equal(s["pos"][n0:], pos[1])
    assert np.array_equal(s["mass"][:n0], masses[0]) and not s["mass"][n0:].any()
    code = textwrap.dedent(f"""
        import sys, zlib, numpy as np
        sys.path.insert(0, {str(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))!r})
        from slicer_b200 import host
        s = host.read_subfile({base + '.0'!r}, True, {n0 + n1 + 10})
        print(zlib.crc32(s['pos'].tobytes()), zlib.crc32(s['mass'].tobytes()))
    """)
    import zlib
    out = subprocess.run([sys.executable, "-c", code], env=dict(os.environ, SLICER_B200_IO_THREADS="1"), capture_output=True, text=True, check=True)
    assert out.stdout.split() == [str(zlib.crc32(s["pos"].tobytes())), str(zlib.crc32(s["mass"].tobytes()))]


@pytest.mark.parametrize("n", [50_000, 1_200_000])  # plain fread path and the multi-threaded path (>= 8 MiB)
def test_reader_rejects_truncated_pos_block(tmp_path, n):
    """A sub-file cut off inside its POS payload is an error (the reference reads garbage silently; here: loud, rc != 0)."""
    box = 100000.0
    base = str(tmp_path / "snap_cut")
    synth.write_snapshot(base, {1: synth.uniform_positions(n, box, 21)}, [0, 0.5, 0, 0, 0, 0], 0.1, box, numfiles=1, with_vel_id=False)
    size = os.path.getsize(base + ".0")
    with open(base + ".0", "r+b") as f:
        f.truncate(size - n * 6)  # lose the second half of the positions
    with pytest.raises(RuntimeError):
        host.read_subfile(base + ".0", False, n + 10)
