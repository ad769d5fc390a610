"""Several light-cone realisations in one run (SLICER_b200 A.ini B.ini ...): one read of every snapshot for all of them.

Driver: every realisation's files are byte-identical to a run of its ini alone (TSC, NGP, perpendicular replication,
per-type files, physical pixels; more realisations than accumulator slots; resume; two GPUs; a degrading ini among normal
ones); mismatched inis are refused before anything is written (CPU).  Library: accumulator slots above 16 per handle, three slot ranges deposited interleaved
with the rounding guard's libm path busy, and eight randomisations from different seed triples in one dense pass, all
against the oracle bit for bit."""
import itertools
import os
import subprocess
import sys

import numpy as np
import pytest

from slicer_b200 import capi, host, synth
from test_gpu_driver import INI, make_dataset

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SEEDS = [(-229, -230, -231), (17, 4242, -5), (-1001, 3, 77), (5, 6, 7)]


def ini_text(lst, snapdir, outdir, seeds=SEEDS[0], suffix="0", sim="gadget", npix=64, zs=0.2, fov=6.0, pip=0, snopt=0, w="-1.0"):
    """test_gpu_driver.INI with the seeds (entries 7-9), simulation name, suffix and w of one realisation."""
    t = INI.format(npix=npix, zs=zs, fov=fov, list=lst, snapdir=snapdir, outdir=outdir, pip=pip, snopt=snopt)
    for old, new in zip((-229, -230, -231), seeds):
        t = t.replace(f"\n{old}\n", f"\n{new}\n")
    t = t.replace("PLC Sim. Name #########\ngadget\n", f"PLC Sim. Name #########\n{sim}\n")
    t = t.replace("PLC Suffix ###########\n0\n", f"PLC Suffix ###########\n{suffix}\n")
    return t.replace("DE-EOS w #############\n-1.0\n", f"DE-EOS w #############\n{w}\n")


def run_exe(args, cwd, quiet=True, timeout=900):
    cmd = [host.EXE_PATH] + (["--quiet"] if quiet else []) + [str(a) for a in args]
    return subprocess.run(cmd, cwd=cwd, capture_output=True, text=True, timeout=timeout)


def tree(root):
    """relative path -> bytes of every file below root"""
    out = {}
    for d, _, files in os.walk(root):
        for f in files:
            p = os.path.join(d, f)
            out[os.path.relpath(p, root)] = open(p, "rb").read()
    return out


def realisation_inis(tmp_path, tag, lst, snapdir, count=3, **kw):
    """`count` inis with different seed triples: the first two write to one directory (other suffixes), the rest to another."""
    inis = []
    for k in range(count):
        out = tmp_path / tag / ("d1" if k < 2 else "d2")
        out.mkdir(parents=True, exist_ok=True)
        seeds = SEEDS[k] if k < len(SEEDS) else (11 * k, -7 * k, 3 * k + 1)
        ini = tmp_path / f"{tag}_{k}.ini"
        ini.write_text(ini_text(lst, snapdir, str(out) + "/t_", seeds=seeds, suffix=f"r{k}", **kw))
        inis.append(ini)
    return inis


def separate_runs_match(tmp_path, lst, snapdir, extra=(), count=3, together_extra=(), **kw):
    together = realisation_inis(tmp_path, "together", lst, snapdir, count, **kw)
    r = run_exe([*extra, *together_extra, *together], tmp_path, quiet=False)
    assert r.returncode == 0, r.stderr[-3000:]
    log = r.stdout
    for ini in realisation_inis(tmp_path, "alone", lst, snapdir, count, **kw):
        r = run_exe([*extra, ini], tmp_path)
        assert r.returncode == 0, r.stderr[-3000:]
    a, b = tree(tmp_path / "together"), tree(tmp_path / "alone")
    assert sorted(a) == sorted(b)
    assert all(a[f] == b[f] for f in a), [f for f in a if a[f] != b[f]]
    for k in range(count):
        assert f"{'d1' if k < 2 else 'd2'}/t_planes_list_r{k}.txt" in a
    return a, log


def snapshot_runs(planes_list):
    """lengths of the runs of consecutive planes cut from one snapshot (planes_list column 6)"""
    return [len(list(g)) for _, g in itertools.groupby(line.split()[5] for line in open(planes_list))]


# ---- driver: byte identity with separate runs ------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("case", ["tsc", "ngp", "replication", "hydro_per_type", "physical"])
def test_several_inis_write_what_separate_runs_write(tmp_path, case):
    """Three inis with different seed triples (two share an output directory) on 4 snapshots of 3 sub-files: every FITS file
    and planes_list of `SLICER_b200 A B C` equals, byte for byte, what `SLICER_b200 X` writes for each ini alone."""
    snapdir, lst = make_dataset(tmp_path, nsnap=4, numfiles=3, hydro=case == "hydro_per_type")
    kw, extra = {}, ()
    if case == "ngp":
        extra = ("--ngp",)
    elif case == "replication":
        extra, kw = ("--replication",), dict(fov=25.0)  # wider than the box at the far planes: the general chain with replicas
    elif case == "hydro_per_type":
        kw = dict(pip=1, npix=128)
    elif case == "physical":
        kw = dict(npix=-500)
    files, _ = separate_runs_match(tmp_path, lst, snapdir, extra, **kw)
    fits = [f for f in files if f.endswith(".fits")]
    assert len(fits) >= 3 * 16
    if case == "hydro_per_type":
        assert any(".ptype0_plane_" in f for f in fits) and any(".ptype4_plane_" in f for f in fits)
    if case == "physical":
        sides = {host.read_fits(str(tmp_path / "together" / f))[0]["NAXIS1"] for f in fits}
        assert len(sides) > 4
    # the realisations differ: the same plane of two seed triples is not the same map
    a = [f for f in fits if f.startswith("d1/") and f.endswith("_r0.fits")][-1]
    assert files[a] != files[a.replace("_r0.fits", "_r1.fits")]


@pytest.mark.gpu
def test_more_realisations_than_accumulator_slots(tmp_path):
    """20 realisations x up to 4 planes per snapshot exceed SLICER_MAX_SLOTS (64): each snapshot is read once per group of
    realisations that fits, and every file is still the bytes of the realisation's own run (here through the Python API)."""
    snapdir, lst = make_dataset(tmp_path, ng=24, nsnap=4, numfiles=2)
    count = 20
    together = realisation_inis(tmp_path, "together", lst, snapdir, count, npix=32)
    r = run_exe(together, tmp_path, quiet=False)
    assert r.returncode == 0, r.stderr[-3000:]
    # runs of consecutive planes cut from one snapshot (planes_list column 6): each is read once per group of realisations whose
    # planes fill the 64 slots (a realisation's planes in one pass, passes of up to 16 planes)
    runs = snapshot_runs(tmp_path / "together" / "d1" / "t_planes_list_r0.txt")
    reads = r.stdout.count(" sub-file 0: ")
    assert reads == sum(-(-count * n // capi.MAX_SLOTS) for n in runs) and reads > len(runs), (reads, runs)
    for ini in realisation_inis(tmp_path, "alone", lst, snapdir, count, npix=32):
        assert host.run_light_cone(str(ini)) == 0
    a, b = tree(tmp_path / "together"), tree(tmp_path / "alone")
    assert sorted(a) == sorted(b) and len(a) > count * 8
    assert all(a[f] == b[f] for f in a), [f for f in a if a[f] != b[f]]
    again = tmp_path / "api"
    for k, ini in enumerate(together):
        ini.write_text(ini.read_text().replace(str(tmp_path / "together"), str(again)))
    (again / "d1").mkdir(parents=True)
    (again / "d2").mkdir()
    assert host.run_light_cones([str(i) for i in together]) == 0
    assert tree(again) == a


@pytest.mark.gpu
@pytest.mark.parametrize("slots", [3, 6, 10])
def test_fewer_slots_than_a_merged_pass(tmp_path, slots):
    """--max-slots N below what the realisations' planes of a snapshot take (as when device memory holds only N accumulators,
    or a caller makes an engine with max_planes N): passes are cut to N planes, a realisation's planes of a snapshot are split
    over passes when they exceed N (3 slots, 4 planes), and a snapshot is read once per group of N slots.  Every file is still
    the bytes of the realisation's own run with all the slots it wants."""
    snapdir, lst = make_dataset(tmp_path, nsnap=4, numfiles=2)
    count = 3
    _, log = separate_runs_match(tmp_path, lst, snapdir, (), count, together_extra=("--max-slots", slots))
    runs = snapshot_runs(tmp_path / "together" / "d1" / "t_planes_list_r0.txt")
    assert max(runs) > min(slots, 16) or count * max(runs) > slots
    reads = log.count(" sub-file 0: ")
    assert reads >= sum(-(-count * n // slots) for n in runs) and reads > len(runs), (reads, runs)


@pytest.mark.gpu
def test_resume_rewrites_only_the_missing_planes(tmp_path):
    snapdir, lst = make_dataset(tmp_path, ng=24, nsnap=3, numfiles=2)
    inis = realisation_inis(tmp_path, "out", lst, snapdir, 3, npix=32, zs=0.1, fov=5.0)
    assert run_exe(inis, tmp_path).returncode == 0
    before = tree(tmp_path / "out")
    fits = sorted(f for f in before if f.endswith("_r1.fits"))
    assert len(fits) >= 8
    gone = [fits[1], fits[-2]]
    stamp = {f: os.stat(tmp_path / "out" / f).st_mtime_ns for f in before}
    for f in gone:
        os.remove(tmp_path / "out" / f)
    r = run_exe(inis, tmp_path, quiet=False)
    assert r.returncode == 0, r.stderr[-3000:]
    assert r.stdout.count("Already exists") == sum(1 for f in before if f.endswith(".fits")) - len(gone)
    assert tree(tmp_path / "out") == before  # the deleted planes are rebuilt bit for bit
    rewritten = {f for f in before if f.endswith(".fits") and os.stat(tmp_path / "out" / f).st_mtime_ns != stamp[f]}
    assert rewritten == set(gone)


@pytest.mark.gpu
def test_two_gpus_match_one_gpu(tmp_path):
    if capi.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    snapdir, lst = make_dataset(tmp_path, ng=40, nsnap=3, numfiles=5)
    outs = {}
    for tag, gpus in (("g1", "0"), ("g2", "0,1")):
        inis = realisation_inis(tmp_path, tag, lst, snapdir, 3, zs=0.1)
        r = run_exe(["--gpus", gpus, *inis], tmp_path)
        assert r.returncode == 0, r.stderr[-3000:]
        outs[tag] = tree(tmp_path / tag)
    assert len(outs["g1"]) >= 3 * 8 and outs["g1"] == outs["g2"]


@pytest.mark.gpu
def test_a_degrading_ini_among_normal_ones(tmp_path):
    """Part. Degradation = 1 in the second of three inis (4 snapshots of 3 sub-files): the degrading light cone takes its own two
    sweeps over each snapshot after the shared passes of the others, and every file is still the bytes of each ini's own run."""
    snapdir, lst = make_dataset(tmp_path, nsnap=4, numfiles=3)

    def inis(tag):
        out = realisation_inis(tmp_path, tag, lst, snapdir, 3)
        out[1].write_text(out[1].read_text().replace("Part. Degradation ####\n0\n", "Part. Degradation ####\n1\n"))
        return out

    r = run_exe(inis("together"), tmp_path, quiet=False)
    assert r.returncode == 0, r.stderr[-3000:]
    reads = [line for line in r.stdout.splitlines() if line.startswith(" sub-file ")]
    degraded = [line for line in reads if line.endswith(" (degradation 2^-1)")]
    assert degraded and 2 * len(degraded) == len(reads)  # sweep 2 logs each sub-file the shared passes log; sweep 1 is silent
    for ini in inis("alone"):
        r = run_exe([ini], tmp_path)
        assert r.returncode == 0, r.stderr[-3000:]
    a, b = tree(tmp_path / "together"), tree(tmp_path / "alone")
    assert sorted(a) == sorted(b) and sum(f.endswith("_r1.fits") for f in a) >= 8
    assert all(a[f] == b[f] for f in a), [f for f in a if a[f] != b[f]]


# ---- library: slots above 16, interleaved sets, eight randomisations --------------------------------------------------------
BOX = 128000.0


def random_planes(seeds, layers, fov, npix):
    """One randomisation per seed triple (randomizeBox of a plan whose first plane opens a group), `layers` planes each."""
    out = []
    for sc, sf, ss in seeds:
        r = host.randomize_box(sc, sf, ss, [1])
        for ld, ld2, rcase in layers:
            out.append(dict(boxsize=BOX, sgn=[int(r["sgnX"][0]), int(r["sgnY"][0]), int(r["sgnZ"][0])], face=int(r["face"][0]),
                            centre=[float(r["x0"][0]), float(r["y0"][0]), float(r["z0"][0])], rcase=rcase, ld=ld, ld2=ld2, nrepperp=0,
                            fovradiants=fov))
    return out


def desc(p, npix):
    return capi.plane_desc(p["sgn"], p["face"], p["centre"], p["rcase"], p["ld"], p["ld2"], p["fovradiants"], npix)


def seed_triples(n, base):
    return [(base + 7 * i, -base - 3 * i, 1000 + base + i) for i in range(n)]


def expect(oracle, batches, planes, npix, fb):
    """-> per plane (counts, ingrid, int64 map) of all batches together (integer accumulators add exactly)"""
    out = []
    for p in planes:
        c, g, m = np.zeros(6, np.int64), np.zeros(6, np.int64), 0
        for pos in batches:
            r = oracle.plane_from_particles([dict(type=1, raw=pos, const_mass=1.0375)], p, npix, frac_bits=fb)
            c, g, m = c + r["counts"], g + r["ingrid"], m + r["fixed"][1]
        out.append((c, g, m))
    return out


@pytest.mark.gpu
def test_slots_above_sixteen(oracle):
    """max_planes = 64: passes of 16 planes (8 randomisations x 2) into slots 0-15, 16-31 and 48-63 over two batches of one
    snapshot (non-accumulating, then accumulating).  Every slot's counts and int64 map equal the oracle's on both batches."""
    npix, n = 64, 1 << 17
    batches = [synth.uniform_positions(n, BOX, 71), synth.uniform_positions(n, BOX, 72)]
    ranges = [0, 16, 48]
    sets = [random_planes(seed_triples(8, 100 * (i + 1)), [(8.0, 40.0, 0.0), (40.0, 100.0, 0.0)], 0.3, npix) for i in range(3)]
    with capi.Slicer(npix_max=npix, max_planes=capi.MAX_SLOTS, particle_capacity=n + 64, staging_buffers=2) as s:
        fb = s.frac_bits
        for b, pos in enumerate(batches):
            if b == 0:
                s.begin_snapshot(BOX, [0, 1.0375, 0, 0, 0, 0], False)
            else:
                s.next_batch()
            s.stage(1, pos)
            for first, planes in zip(ranges, sets):
                s.deposit_slots([desc(p, npix) for p in planes], first, accumulate=b > 0)
        for first, planes in zip(ranges, sets):
            for k, (c, g, m) in enumerate(expect(oracle, batches, planes, npix, fb)):
                _, counts, ingrid = s.fetch(first + k, -1, npix, want_map=False)
                assert counts.tolist() == c.tolist() and ingrid.tolist() == g.tolist(), (first, k)
                assert np.array_equal(s.fetch_fixed(first + k, -1, npix).reshape(-1), m), (first, k)
                assert c[1] > 0
        too_many = [desc(p, npix) for p in sets[0]] + [desc(sets[1][0], npix)]
        with pytest.raises(capi.SlicerError, match="SLICER_MAX_PLANES"):
            s.deposit_slots(too_many, 0)
        with pytest.raises(capi.SlicerError):
            s.deposit_slots([desc(p, npix) for p in sets[0][:8]], 60)
        with pytest.raises(capi.SlicerError):
            s.fetch(64, -1, npix)
    with capi.Slicer(npix_max=npix, max_planes=20, particle_capacity=n + 64) as s:
        s.begin_snapshot(BOX, [0, 1.0375, 0, 0, 0, 0], False)
        s.stage(1, batches[0])
        s.deposit_slots([desc(sets[0][0], npix)], 19)
        with pytest.raises(capi.SlicerError):
            s.deposit_slots([desc(sets[0][0], npix)], 20)
        with pytest.raises(capi.SlicerError):
            s.count_accepted(too_many)
    with pytest.raises(capi.SlicerError, match="SLICER_MAX_SLOTS"):
        capi.Slicer(npix_max=npix, max_planes=capi.MAX_SLOTS + 1)


@pytest.mark.gpu
@pytest.mark.parametrize("finish", ["settle", "reduce", "reduce_in_one_rank"])
def test_interleaved_sets_with_the_libm_path(oracle, finish):
    """guard_eta = 2^-34 sends thousands of pairs per pass to the host's libm.  Three slot ranges are deposited as the driver
    does with three realisations: A, B, C non-accumulating over batch 1, then A, B, C accumulating over batch 2; then each
    range is settled (or reduced, also as the only rank of a communicator) and read.  Every plane equals the oracle on batch 1 +
    batch 2 bit for bit."""
    npix, n = 256, 1 << 20
    batches = [synth.uniform_positions(n, BOX, 81), synth.uniform_positions(n, BOX, 82)]
    sets = [random_planes(seed_triples(1, 500 + 10 * i), [(40.0, 100.0, 0.0), (100.0, 128.0, 0.0)], 0.55, npix) for i in range(3)]
    ranges = [0, 2, 4]
    with capi.Slicer(npix_max=npix, max_planes=6, particle_capacity=n + 64, staging_buffers=2, guard_eta=2.0 ** -34) as s:
        if finish == "reduce_in_one_rank":
            s.comm_init_rank(capi.Slicer.comm_unique_id(), 1, 0)
        fb = s.frac_bits
        f0 = int(s.stats().flagged_pairs)
        for b, pos in enumerate(batches):
            if b == 0:
                s.begin_snapshot(BOX, [0, 1.0375, 0, 0, 0, 0], False)
            else:
                s.next_batch()
            s.stage(1, pos)
            for first, planes in zip(ranges, sets):
                s.deposit_slots([desc(p, npix) for p in planes], first, accumulate=b > 0)
        for first in ranges:
            (s.settle_slots if finish == "settle" else s.reduce_slots)(first, 2)
        settled = int(s.stats().flagged_pairs) - f0
        for first, planes in zip(ranges, sets):
            for k, (c, g, m) in enumerate(expect(oracle, batches, planes, npix, fb)):
                _, counts, ingrid = s.fetch(first + k, -1, npix, want_map=False)
                assert counts.tolist() == c.tolist() and ingrid.tolist() == g.tolist(), (first, k)
                assert np.array_equal(s.fetch_fixed(first + k, -1, npix).reshape(-1), m), (first, k)
        assert int(s.stats().flagged_void) == 0
    assert settled > 3000, settled


@pytest.mark.gpu
@pytest.mark.parametrize("mode", [capi.DEPOSIT_BINNED, capi.DEPOSIT_AUTO])
def test_eight_randomisations_in_one_dense_pass(oracle, mode):
    """8 seed triples x 2 planes = 16 planes in one pass; the thick wide planes accept ~40 % of the snapshot each."""
    npix, n = 256, 1 << 20
    pos = synth.uniform_positions(n, BOX, 91)
    planes = random_planes(seed_triples(8, 900), [(40.0, 128.0, 0.0), (8.0, 40.0, 0.0)], 1.0, npix)
    with capi.Slicer(npix_max=npix, max_planes=16, particle_capacity=n + 64, deposit_mode=mode) as s:
        s.begin_snapshot(BOX, [0, 1.0375, 0, 0, 0, 0], False)
        s.stage(1, pos)
        s.deposit([desc(p, npix) for p in planes])
        fb = s.frac_bits
        want = expect(oracle, [pos], planes, npix, fb)
        for k, (c, g, m) in enumerate(want):
            _, counts, ingrid = s.fetch(k, -1, npix, want_map=False)
            assert counts.tolist() == c.tolist() and ingrid.tolist() == g.tolist(), k
            assert np.array_equal(s.fetch_fixed(k, -1, npix).reshape(-1), m), k
    assert max(c[1] for c, _, _ in want) > 0.3 * n
    assert len({(tuple(p["sgn"]), p["face"], tuple(p["centre"])) for p in planes}) == 8


@pytest.mark.gpu
def test_checked_build_traps_nothing_with_many_slots():
    """The library tests of this file against libslicer_b200_chk.so (device-side bounds checks).  Fresh interpreter: the
    library is loaded once per process."""
    chk = os.path.join(ROOT, "slicer_b200", "_build", "libslicer_b200_chk.so")
    if not os.path.exists(chk):
        pytest.skip("checked build not present (python -c 'import __graft_entry__ as g; g.build()')")
    sel = "slots_above or interleaved or eight_randomisations"
    r = subprocess.run([sys.executable, "-m", "pytest", os.path.abspath(__file__), "-x", "-q", "-m", "gpu", "-k", sel, "-p", "no:cacheprovider"],
                       env=dict(os.environ, SLICER_B200_LIB=chk), cwd=ROOT, capture_output=True, text=True)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-2000:]


# ---- refusal of inis that cannot share a run (CPU: checked before any device call) ------------------------------------------
MISMATCHES = {
    "map pixels": dict(npix=32),
    "source redshift": dict(zs=0.3),
    "field of view": dict(fov=5.0),
    "snapshot list": "list",
    "snapshot path": "snapdir",
    "one map per particle type": dict(pip=1),
    "dark-energy w": dict(w="-0.9"),
}


@pytest.mark.parametrize("key", sorted(MISMATCHES) + ["same output", "two degradations"])
def test_mismatched_inis_are_refused_before_any_output(tmp_path, key):
    snapdir, lst = make_dataset(tmp_path, ng=8, nsnap=2, numfiles=1)
    outs = [tmp_path / "o0", tmp_path / "o1"]
    for o in outs:
        o.mkdir()
    first = dict(seeds=SEEDS[0], suffix="a")
    second = dict(seeds=SEEDS[1], suffix="b")
    base = dict(lst=lst, snapdir=snapdir)
    change = MISMATCHES.get(key)
    if change == "list":
        other = tmp_path / "other_list.txt"
        other.write_text(open(lst).read())
        base2 = dict(base, lst=str(other))
    elif change == "snapdir":
        os.symlink(snapdir, tmp_path / "snaps_link")
        base2 = dict(base, snapdir=str(tmp_path / "snaps_link") + "/")
    else:
        base2 = dict(base)
        second.update(change or {})
    if key == "same output":
        second.update(suffix="a")
    if key == "two degradations":
        first.update(snopt=1)
        second.update(snopt=2)
    inis = [tmp_path / "a.ini", tmp_path / "b.ini"]
    inis[0].write_text(ini_text(base["lst"], base["snapdir"], str(outs[0]) + "/t_", **first))
    inis[1].write_text(ini_text(base2["lst"], base2["snapdir"], str(outs[0 if key == "same output" else 1]) + "/t_", **second))
    r = run_exe(inis, tmp_path, quiet=False, timeout=120)
    assert r.returncode != 0
    want = {"same output": "output directory", "two degradations": "particle degradation"}.get(key, key)
    assert want in r.stderr and "b.ini" in r.stderr, r.stderr
    assert [os.listdir(o) for o in outs] == [[], []]
    if key in MISMATCHES:
        assert "must agree" in r.stderr
