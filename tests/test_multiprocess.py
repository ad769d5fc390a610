"""SLICER_b200 as one job of several processes (mpirun -np N / srun / torchrun): launcher parsing, the TCP control channel
between the ranks, the job's sub-file assignment (CPU); and on the GPU, N processes whose FITS files and planes_list are byte-identical
to one process on one GPU, a rank that fails making every rank stop, and a world-size-1 run that is today's run."""
import json
import os
import socket
import subprocess
import sys
import time

import pytest

from slicer_b200 import capi, host

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LAUNCHER_VARS = ("OMPI_COMM_WORLD_RANK", "OMPI_COMM_WORLD_SIZE", "OMPI_COMM_WORLD_LOCAL_RANK", "PMI_RANK", "PMI_SIZE", "MPI_LOCALRANKID",
                 "SLURM_PROCID", "SLURM_STEP_NUM_TASKS", "SLURM_LOCALID", "RANK", "WORLD_SIZE", "LOCAL_RANK", "MASTER_ADDR", "MASTER_PORT",
                 "TORCHELASTIC_RUN_ID")


def clean_env(**extra):
    """this process' environment without any launcher variable (the tests may run under a launcher), plus `extra`"""
    env = {k: v for k, v in os.environ.items() if k not in LAUNCHER_VARS}
    env.update({k: str(v) for k, v in extra.items()})
    return env


def free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def wait_all(procs, deadline):
    """(returncode, stdout, stderr) of every process; kills all of them if the deadline passes, and in any case on the way out"""
    out = []
    try:
        for p in procs:
            o, e = p.communicate(timeout=max(1.0, deadline - time.time()))
            out.append((p.returncode, o, e))
        return out
    finally:
        for p in procs:
            if p.poll() is None:
                p.kill()
                p.communicate()


# ---- launcher parsing -------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("rank_var,size_var", [("OMPI_COMM_WORLD_RANK", "OMPI_COMM_WORLD_SIZE"), ("PMI_RANK", "PMI_SIZE"),
                                               ("SLURM_PROCID", "SLURM_STEP_NUM_TASKS"), ("RANK", "WORLD_SIZE")])
def test_launcher_families(rank_var, size_var):
    l = host.launch_from_env({rank_var: "3", size_var: "4", "MASTER_ADDR": "node7", "MASTER_PORT": "29511"})
    assert (l["rank"], l["nranks"], l["master_addr"], l["master_port"]) == (3, 4, "node7", 29511)
    assert l["local_rank"] == 3  # no local-rank variable: the global rank stands in


@pytest.mark.parametrize("local_var", ["OMPI_COMM_WORLD_LOCAL_RANK", "MPI_LOCALRANKID", "SLURM_LOCALID", "LOCAL_RANK"])
def test_local_rank_picks_the_gpu(local_var):
    base = {"RANK": "13", "WORLD_SIZE": "16", "MASTER_ADDR": "a", "MASTER_PORT": "1234", local_var: "5"}
    assert host.launch_from_env(base, ndev=8)["device"] == 5
    assert host.launch_from_env(base, ndev=4)["device"] == 1  # local rank modulo the visible devices
    assert host.launch_from_env(base, ndev=1)["device"] == 0  # CUDA_VISIBLE_DEVICES set per task: one device each


def test_world_size_one_is_a_plain_run():
    # (an sbatch script's own step: SLURM_PROCID = 0 and SLURM_NTASKS = the job's tasks, but it is one process, not an srun step)
    for env in ({}, {"RANK": "0", "WORLD_SIZE": "1"}, {"SLURM_PROCID": "0", "SLURM_STEP_NUM_TASKS": "1", "SLURM_LOCALID": "0"},
                {"SLURM_PROCID": "0", "SLURM_NTASKS": "8", "SLURM_NPROCS": "8", "SLURM_JOB_ID": "77"}):
        l = host.launch_from_env(env, ndev=8)
        assert (l["rank"], l["nranks"], l["master_addr"], l["device"]) == (0, 1, "", 0)


def test_first_family_wins_and_bad_values_are_refused():
    l = host.launch_from_env({"OMPI_COMM_WORLD_RANK": "1", "OMPI_COMM_WORLD_SIZE": "2", "RANK": "0", "WORLD_SIZE": "8", "MASTER_ADDR": "h",
                              "MASTER_PORT": "9"})
    assert (l["rank"], l["nranks"]) == (1, 2)
    for env in ({"RANK": "2", "WORLD_SIZE": "2"}, {"RANK": "x", "WORLD_SIZE": "2"}, {"RANK": "0", "WORLD_SIZE": "0"}):
        with pytest.raises(ValueError):
            host.launch_from_env(env)


def test_torchrun_leaves_master_port_to_its_agent():
    env = {"RANK": "1", "WORLD_SIZE": "2", "LOCAL_RANK": "1", "MASTER_ADDR": "127.0.0.1", "MASTER_PORT": "29500"}
    assert host.launch_from_env(env)["master_port"] == 29500
    assert host.launch_from_env(dict(env, TORCHELASTIC_RUN_ID="none"))["master_port"] == 29501
    with pytest.raises(ValueError):
        host.launch_from_env(dict(env, MASTER_PORT="65535", TORCHELASTIC_RUN_ID="none"))


def test_ranks_meet_under_torchrun(tmp_path):
    """SLICER_b200 started by torchrun itself (whose agent holds MASTER_PORT): the ranks meet before they read the ini, so a
    missing ini reported by both ranks shows that they met (no GPU needed)"""
    port = free_port()
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes", "1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
                        "--master-port", str(port), "--no-python", host.EXE_PATH, "--gpus", "0", str(tmp_path / "missing.ini")],
                       cwd=tmp_path, env=clean_env(), capture_output=True, text=True, timeout=180)
    out = r.stdout + r.stderr
    assert "cannot listen" not in out and "cannot reach rank 0" not in out, out[-3000:]
    assert out.count("cannot open the parameter file") == 2, out[-3000:]


@pytest.mark.parametrize("env", [{"RANK": "1", "WORLD_SIZE": "2"}, {"RANK": "0", "WORLD_SIZE": "2", "MASTER_ADDR": "127.0.0.1"},
                                 {"PMI_RANK": "0", "PMI_SIZE": "3", "MASTER_PORT": "29500"}])
def test_refused_without_master(env):
    with pytest.raises(ValueError) as e:
        host.launch_from_env(env)
    assert "MASTER_ADDR" in str(e.value) and "MASTER_PORT" in str(e.value)


def test_executable_refuses_without_master(tmp_path):
    """the reference's command line under a launcher but without a meeting point: stops before any work, never runs alone"""
    r = subprocess.run([host.EXE_PATH, str(tmp_path / "missing.ini")], env=clean_env(OMPI_COMM_WORLD_RANK=0, OMPI_COMM_WORLD_SIZE=4),
                       capture_output=True, text=True, timeout=60)
    assert r.returncode != 0
    assert "MASTER_ADDR" in r.stderr and "MASTER_PORT" in r.stderr
    assert not list(tmp_path.iterdir())


# ---- the job's sub-file assignment -------------------------------------------------------------------------------------------
@pytest.mark.parametrize("ngpus", [[1], [1, 1], [2, 1], [1, 3, 2], [4, 4], [2, 1, 1, 4]])
@pytest.mark.parametrize("ffmin,ffmax", [(0, 1), (0, 5), (0, 16), (3, 40)])
def test_every_subfile_on_one_gpu(ngpus, ffmin, ffmax):
    owners = host.subfile_owners(ngpus, ffmin, ffmax)
    G = sum(ngpus)
    glob = [sum(ngpus[:r]) + g for r, g in owners]  # the job's GPU index of each sub-file's owner
    assert all(0 <= g < ngpus[r] for r, g in owners)
    assert glob == [(ff - ffmin) % G for ff in range(ffmin, ffmax)]  # round-robin over all GPUs of the job, rank after rank


# ---- the control channel: N CPU processes on 127.0.0.1 ----------------------------------------------------------------------
WORKER = r"""
import json, sys, os
sys.path.insert(0, sys.argv[1])
from slicer_b200 import host
rank, n, port, mode, timeout = int(sys.argv[2]), int(sys.argv[3]), int(sys.argv[4]), sys.argv[5], float(sys.argv[6])
g = host.Group(rank, n, "127.0.0.1", port, timeout)
res = dict(rank=rank, open=g.ok)
try:
    if mode == "ops" and g.ok:
        res["bcast"] = g.bcast(b"id:" + bytes(range(128)) if rank == 0 else b"").hex()
        res["gather"] = [b.decode() for b in g.allgather((("r%d" % rank) * rank).encode(), n)]
        res["min"] = g.allreduce([rank, -rank, 10 + rank], "min")
        res["max"] = g.allreduce([rank, -rank, 10 + rank], "max")
        res["sum"] = g.allreduce([rank, 1, 1 << 40], "sum")
        res["agree_ok"] = g.agree(0)
        res["agree_one_failed"] = g.agree(1 if rank == n - 1 else 0)
        res["again"] = g.allreduce([1], "sum")
    elif mode.startswith("leave") and g.ok:
        leaver = int(mode[5:])
        g.allreduce([rank], "sum")
        if rank == leaver:
            os._exit(3)  # leaves the job without a word
        try:
            g.allreduce([rank], "sum")
            res["second"] = "ok"
        except RuntimeError:
            res["second"] = "failed"
        try:
            g.bcast(b"x")
            res["third"] = "ok"
        except RuntimeError:
            res["third"] = "failed"
finally:
    g.close()
print(json.dumps(res), flush=True)
"""


def start_ranks(n, mode, ranks=None, timeout=30.0, port=None):
    port = port or free_port()
    return [subprocess.Popen([sys.executable, "-c", WORKER, ROOT, str(r), str(n), str(port), mode, str(timeout)], env=clean_env(),
                             stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True) for r in (range(n) if ranks is None else ranks)]


@pytest.mark.parametrize("n", [2, 4])
def test_channel_operations(n):
    res = wait_all(start_ranks(n, "ops"), time.time() + 120)
    out = [json.loads(o) for rc, o, e in res]
    assert all(rc == 0 for rc, _, _ in res), [e for _, _, e in res]
    for r in out:
        assert r["open"]
        assert bytes.fromhex(r["bcast"]) == b"id:" + bytes(range(128))
        assert r["gather"] == [("r%d" % k) * k for k in range(n)]
        assert r["min"] == [0, -(n - 1), 10] and r["max"] == [n - 1, 0, 10 + n - 1]
        assert r["sum"] == [n * (n - 1) // 2, n, n << 40]
        assert r["agree_ok"] == 0 and r["agree_one_failed"] == 1 and r["again"] == [n]


def test_channel_times_out_when_a_rank_never_arrives():
    t0 = time.time()
    port = free_port()
    res = wait_all(start_ranks(3, "ops", ranks=[0, 1], timeout=3.0, port=port), time.time() + 60)
    assert time.time() - t0 < 30
    out = [json.loads(o) for _, o, _ in res]
    assert not out[0]["open"]  # rank 0 waited for rank 2 in vain
    assert f"127.0.0.1:{port}" in res[0][2] and "MASTER_ADDR" in res[0][2]
    assert not out[1]["open"]  # rank 1 got in, but rank 0 gave up and closed its connection
    # a rank whose rank 0 never listens: names the address it tried
    port2 = free_port()
    (rc, o, e), = wait_all(start_ranks(2, "ops", ranks=[1], timeout=2.0, port=port2), time.time() + 60)
    assert not json.loads(o)["open"] and f"127.0.0.1:{port2}" in e


@pytest.mark.parametrize("n,leaver", [(2, 1), (2, 0), (4, 2), (4, 0)])
def test_channel_fails_on_every_rank_when_one_leaves(n, leaver):
    res = wait_all(start_ranks(n, f"leave{leaver}"), time.time() + 120)
    for r, (rc, o, e) in enumerate(res):
        if r == leaver:
            assert rc == 3
            continue
        out = json.loads(o)
        assert out["second"] == "failed" and out["third"] == "failed", (r, e)


# ---- GPU: N SLICER_b200 processes against one process on one GPU --------------------------------------------------------------
def need_gpus(n):
    have = capi.device_count()
    if have < n:
        pytest.skip(f"needs {n} GPUs ({have} visible): NCCL refuses two ranks of one communicator on one device")


def run_job(inis, cwd, gpus_per_rank, extra=(), timeout=600):
    """one SLICER_b200 process per entry of gpus_per_rank (its --gpus list), started with torchrun's variables on 127.0.0.1"""
    port = free_port()
    n = len(gpus_per_rank)
    procs = []
    for r, gpus in enumerate(gpus_per_rank):
        env = clean_env(RANK=r, WORLD_SIZE=n, LOCAL_RANK=r, MASTER_ADDR="127.0.0.1", MASTER_PORT=port)
        cmd = [host.EXE_PATH, "--quiet", "--gpus", ",".join(map(str, gpus)), *extra, *map(str, inis)]
        procs.append(subprocess.Popen(cmd, cwd=cwd, env=env, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True))
    return wait_all(procs, time.time() + timeout)


def run_alone(inis, cwd, extra=(), env=None, timeout=600):
    r = subprocess.run([host.EXE_PATH, "--quiet", "--gpus", "0", *extra, *map(str, inis)], cwd=cwd, env=env or clean_env(),
                       capture_output=True, text=True, timeout=timeout)
    assert r.returncode == 0, r.stderr[-3000:]


def make_case(tmp_path, case):
    from test_gpu_driver import make_dataset
    from test_gpu_realisations import SEEDS, ini_text

    hydro = case == "per_type"
    snapdir, lst = make_dataset(tmp_path, ng=40 if not hydro else 32, nsnap=3, numfiles=5, hydro=hydro)
    kw = dict(npix=64, zs=0.1, fov=6.0, pip=1 if hydro else 0, snopt=1 if case == "degrade" else 0)
    count = 2 if case == "two_realisations" else 1

    def inis(tag):
        out = tmp_path / tag
        out.mkdir()
        paths = []
        for k in range(count):
            p = tmp_path / f"{tag}_{k}.ini"
            p.write_text(ini_text(lst, snapdir, str(out) + "/t_", seeds=SEEDS[k], suffix=f"r{k}", **kw))
            paths.append(p)
        return paths

    return inis


def tree(root):
    from test_gpu_realisations import tree as t

    return t(root)


CASES = ["tsc", "ngp", "per_type", "degrade", "two_realisations"]


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES)
def test_two_processes_match_one(tmp_path, case):
    need_gpus(2)
    inis = make_case(tmp_path, case)
    extra = ("--ngp",) if case == "ngp" else ()
    run_alone(inis("one"), tmp_path, extra)
    res = run_job(inis("job"), tmp_path, [[0], [1]], extra)
    assert all(rc == 0 for rc, _, _ in res), [e[-3000:] for _, _, e in res]
    a, b = tree(tmp_path / "one"), tree(tmp_path / "job")
    assert sorted(a) == sorted(b) and sum(f.endswith(".fits") for f in a) >= 8
    assert [f for f in a if a[f] != b[f]] == []


@pytest.mark.gpu
def test_two_processes_resume(tmp_path):
    need_gpus(2)
    inis = make_case(tmp_path, "tsc")
    job = inis("job")
    assert all(rc == 0 for rc, _, _ in run_job(job, tmp_path, [[0], [1]]))
    full = tree(tmp_path / "job")
    fits = sorted(f for f in full if f.endswith(".fits"))
    for f in fits[2:5]:
        os.remove(tmp_path / "job" / f)
    res = run_job(job, tmp_path, [[0], [1]], timeout=600)
    assert all(rc == 0 for rc, _, _ in res), [e[-3000:] for _, _, e in res]
    assert tree(tmp_path / "job") == full  # the deleted planes are rebuilt bit for bit, the others untouched


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["tsc", "degrade"])
def test_two_processes_of_two_gpus_match_one(tmp_path, case):
    need_gpus(4)
    inis = make_case(tmp_path, case)
    run_alone(inis("one"), tmp_path)
    res = run_job(inis("job"), tmp_path, [[0, 1], [2, 3]])
    assert all(rc == 0 for rc, _, _ in res), [e[-3000:] for _, _, e in res]
    assert tree(tmp_path / "one") == tree(tmp_path / "job")


@pytest.mark.gpu
def test_mixed_gpu_counts_per_rank_match_one(tmp_path):
    need_gpus(3)
    inis = make_case(tmp_path, "degrade")
    run_alone(inis("one"), tmp_path)
    res = run_job(inis("job"), tmp_path, [[0], [1, 2]])
    assert all(rc == 0 for rc, _, _ in res), [e[-3000:] for _, _, e in res]
    assert tree(tmp_path / "one") == tree(tmp_path / "job")


@pytest.mark.gpu
def test_a_failing_rank_stops_the_job(tmp_path):
    """rank 1's sub-files are cut short after their headers: rank 1 fails reading one, and rank 0 learns it before the reduce
    instead of waiting in NCCL for a rank that is gone"""
    need_gpus(2)
    inis = make_case(tmp_path, "tsc")
    snaps = tmp_path / "snaps"
    for f in snaps.iterdir():
        if f.name.endswith(".1") or f.name.endswith(".3"):  # of 5 sub-files: the job's GPU 1 takes 1 and 3
            with open(f, "r+b") as fh:
                fh.truncate(300)
    t0 = time.time()
    res = run_job(inis("job"), tmp_path, [[0], [1]], timeout=300)
    assert time.time() - t0 < 300
    assert all(rc != 0 for rc, _, _ in res), [(rc, e[-2000:]) for rc, _, e in res]


@pytest.mark.gpu
def test_world_size_one_is_todays_run(tmp_path):
    """one GPU: the launcher's variables for a job of one process, and the library call with rank 0 of 1, give today's bytes"""
    inis = make_case(tmp_path, "degrade")
    run_alone(inis("plain"), tmp_path)
    run_alone(inis("ws1"), tmp_path, env=clean_env(RANK=0, WORLD_SIZE=1, LOCAL_RANK=0))
    lib_inis = inis("lib")
    assert host.run_light_cones([str(i) for i in lib_inis], devices=(0,), rank=0, nranks=1) == 0
    plain = tree(tmp_path / "plain")
    assert plain == tree(tmp_path / "ws1") == tree(tmp_path / "lib")


def test_a_rank_that_stops_before_any_work_stops_the_job(tmp_path):
    """rank 0 cannot read its ini: rank 1, which can, stops at its next collective call with the job's exit code instead of
    waiting or running on alone (no GPU needed: rank 1 stops before it makes its engine)"""
    from test_gpu_driver import make_dataset
    from test_gpu_realisations import ini_text

    snapdir, lst = make_dataset(tmp_path, ng=8, nsnap=2, numfiles=1)
    (tmp_path / "out").mkdir()
    ini = tmp_path / "a.ini"
    ini.write_text(ini_text(lst, snapdir, str(tmp_path / "out") + "/t_", npix=16, zs=0.1))
    port = free_port()
    procs = [subprocess.Popen([host.EXE_PATH, "--quiet", "--gpus", "0", str(ini if r == 1 else tmp_path / "missing.ini")], cwd=tmp_path,
                              env=clean_env(RANK=r, WORLD_SIZE=2, MASTER_ADDR="127.0.0.1", MASTER_PORT=port), stdout=subprocess.PIPE,
                              stderr=subprocess.PIPE, text=True) for r in range(2)]
    res = wait_all(procs, time.time() + 60)
    assert res[0][0] != 0 and res[1][0] == 255
    assert "rank 0 left the job" in res[1][2]
    assert not list((tmp_path / "out").iterdir())
