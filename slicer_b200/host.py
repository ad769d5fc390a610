"""ctypes binding of the C++ host layer (slicer_b200/host/, libslicer_host.so): plan, GADGET-2 reader, FITS writer and
the light-cone driver.  Used by tests and examples; the driver itself is the C++ executable `SLICER_b200`."""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "_build", "libslicer_host.so")
EXE_PATH = os.path.join(HERE, "_build", "SLICER_b200")

_f32p = np.ctypeslib.ndpointer(dtype=np.float32, flags="C_CONTIGUOUS")
_f64p = np.ctypeslib.ndpointer(dtype=np.float64, flags="C_CONTIGUOUS")
_i32p = np.ctypeslib.ndpointer(dtype=np.int32, flags="C_CONTIGUOUS")
_lib = None


def lib():
    global _lib
    if _lib is None:
        L = C.CDLL(LIB_PATH)
        L.shost_cosmo_table.argtypes = [C.c_double] * 4 + [_f64p, _f64p]
        L.shost_plan.argtypes = ([C.c_double] * 4 + [C.c_int, _f64p, _f64p, C.c_char_p, C.c_char_p, C.c_int, C.POINTER(C.c_int),
                                                     C.POINTER(C.c_double)] + [_f64p] * 4 + [_i32p] * 3 + [C.POINTER(C.c_int)])
        L.shost_randomize_box.argtypes = [C.c_int] * 4 + [_i32p, C.c_int, _f64p, _f64p, _f64p, _i32p, _i32p, _i32p, _i32p]
        L.shost_glibc_rand.argtypes = [C.c_uint, C.c_int, _i32p]
        L.shost_read_input.argtypes = [C.c_char_p, _i32p, _f64p, C.c_char_p]
        L.shost_read_subfile.argtypes = [C.c_char_p, C.c_int, _i32p, _f64p, _f64p, C.POINTER(C.c_int), C.c_void_p, C.c_void_p, C.c_longlong]
        L.shost_write_fits.argtypes = [C.c_char_p, _f32p, C.c_int, C.c_int, C.POINTER(C.c_char_p), _f64p, C.c_int, C.POINTER(C.c_char_p),
                                       np.ctypeslib.ndpointer(dtype=np.int64, flags="C_CONTIGUOUS")]
        L.shost_run_light_cone.argtypes = [C.c_char_p, _i32p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int]
        L.shost_run_light_cones.argtypes = [C.POINTER(C.c_char_p), C.c_int, _i32p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                            C.c_int, C.c_char_p, C.c_int]
        L.shost_launch_from_env.argtypes = [C.POINTER(C.c_char_p), C.c_int, C.c_int, _i32p, C.c_char_p, C.c_int, C.c_char_p, C.c_int]
        L.shost_subfile_owners.argtypes = [C.c_int, _i32p, C.c_uint, C.c_uint, _i32p, _i32p]
        L.shost_group_open.restype = C.c_void_p
        L.shost_group_open.argtypes = [C.c_int, C.c_int, C.c_char_p, C.c_int, C.c_double, C.POINTER(C.c_int)]
        L.shost_group_close.argtypes = [C.c_void_p]
        L.shost_group_bcast.argtypes = [C.c_void_p, C.c_char_p, C.POINTER(C.c_longlong), C.c_longlong]
        L.shost_group_allgather.argtypes = [C.c_void_p, C.c_char_p, C.c_longlong, C.c_char_p, C.POINTER(C.c_longlong), C.c_longlong]
        L.shost_group_allreduce.argtypes = [C.c_void_p, C.POINTER(C.c_longlong), C.c_int, C.c_int]
        L.shost_group_agree.argtypes = [C.c_void_p, C.c_int]
        _lib = L
    return _lib


def cosmo_table(om0, oml, w, zs):
    zl, dl = np.zeros(1000), np.zeros(1000)
    lib().shost_cosmo_table(om0, oml, w, zs, zl, dl)
    return zl, dl


def plan(om0, oml, w, zs, snapred, snapbox, directory, suffix="t", cap=4096):
    snapred = np.ascontiguousarray(snapred, np.float64)
    snapbox = np.ascontiguousarray(snapbox, np.float64)
    nplanes, nrepl, Ds = C.c_int(), C.c_int(), C.c_double()
    ld, ld2, zsim, zfs = (np.zeros(cap) for _ in range(4))
    fromsnapi, randomize, replication = (np.zeros(cap, np.int32) for _ in range(3))
    rc = lib().shost_plan(om0, oml, w, zs, len(snapred), snapred, snapbox, directory.encode(), suffix.encode(), cap, C.byref(nplanes),
                          C.byref(Ds), ld, ld2, zsim, zfs, fromsnapi, randomize, replication, C.byref(nrepl))
    if rc:
        raise RuntimeError(f"shost_plan rc={rc}")
    n = nplanes.value
    return dict(nplanes=n, Ds=Ds.value, ld=ld[:n].copy(), ld2=ld2[:n].copy(), zsimlens=zsim[:n].copy(), zfromsnap=zfs[:n].copy(),
                fromsnapi=fromsnapi[:n].copy(), randomize=randomize[:n].copy(), replication=replication[: nrepl.value].copy())


def randomize_box(seedcenter, seedface, seedsign, randomize, fixed_vertex=False):
    randomize = np.ascontiguousarray(randomize, np.int32)
    n = len(randomize)
    x0, y0, z0 = (np.zeros(n) for _ in range(3))
    face, sx, sy, sz = (np.zeros(n, np.int32) for _ in range(4))
    lib().shost_randomize_box(seedcenter, seedface, seedsign, n, randomize, int(fixed_vertex), x0, y0, z0, face, sx, sy, sz)
    return dict(x0=x0, y0=y0, z0=z0, face=face, sgnX=sx, sgnY=sy, sgnZ=sz)


def glibc_rand(seed, n):
    out = np.zeros(n, np.int32)
    lib().shost_glibc_rand(C.c_uint(seed & 0xFFFFFFFF), n, out)
    return out


def read_input(path):
    ints = np.zeros(8, np.int32)
    dbl = np.zeros(3)
    buf = C.create_string_buffer(6 * 512)
    if lib().shost_read_input(path.encode(), ints, dbl, buf):
        raise RuntimeError("readInput failed")
    raw = buf.raw
    strs = [raw[512 * i: 512 * (i + 1)].split(b"\0")[0].decode() for i in range(6)]
    return dict(npix=int(ints[0]), seedcenter=int(ints[1]), seedface=int(ints[2]), seedsign=int(ints[3]), partinplanes=bool(ints[4]),
                snopt=int(ints[5]), physical=bool(ints[6]), rgrid=int(ints[7]), zs=dbl[0], fov=dbl[1], w=dbl[2], filredshiftlist=strs[0],
                pathsnap=strs[1], simulation=strs[2], directory=strs[3], suffix=strs[4], snpix=strs[5])


def read_subfile(path, hydro, cap):
    npart = np.zeros(6, np.int32)
    massarr, sc = np.zeros(6), np.zeros(6)
    nf = C.c_int()
    pos = np.zeros((cap, 3), np.float32)
    mass = np.zeros(cap, np.float32)
    rc = lib().shost_read_subfile(path.encode(), int(hydro), npart, massarr, sc, C.byref(nf), pos.ctypes.data, mass.ctypes.data, cap)
    if rc:
        raise RuntimeError(f"readSubFile rc={rc}")
    n = int(npart.sum())
    return dict(npart=npart, massarr=massarr, time=sc[0], redshift=sc[1], boxsize=sc[2], om0=sc[3], oml=sc[4], h=sc[5], numfiles=nf.value,
                pos=pos[:n], mass=mass[:n])


def write_fits(path, image, dkeys, ikeys):
    image = np.ascontiguousarray(image, np.float32)
    dn = (C.c_char_p * len(dkeys))(*[k.encode() for k, _ in dkeys])
    dv = np.array([v for _, v in dkeys], np.float64)
    in_ = (C.c_char_p * len(ikeys))(*[k.encode() for k, _ in ikeys])
    iv = np.array([v for _, v in ikeys], np.int64)
    return lib().shost_write_fits(path.encode(), image.reshape(-1), image.shape[0], len(dkeys), dn, dv, len(ikeys), in_, iv)


def run_light_cone(ini, devices=(0,), replication=False, fixed_vertex=False, ngp=False, deposit_mode=0):
    dev = np.ascontiguousarray(devices, np.int32)
    return lib().shost_run_light_cone(ini.encode(), dev, len(dev), int(replication), int(fixed_vertex), int(ngp), int(deposit_mode))


def run_light_cones(inis, devices=(0,), replication=False, fixed_vertex=False, ngp=False, deposit_mode=0, max_slots=0, rank=0, nranks=1,
                    master=None):
    """One light cone per ini (realisations of one plan: other seeds, other outputs), every snapshot read once for all (once per
    group of planes that fits `max_slots` accumulators per GPU, when given).  Returns 0 on success; inis that disagree on the
    plan are refused before anything is written.
    rank / nranks / master ("host:port", where rank 0 listens): this process is one rank of a job of `nranks` processes that
    all make this call with the same arguments but `rank` and `devices`; rank 0 writes the files.  The launcher's environment
    is not read."""
    dev = np.ascontiguousarray(devices, np.int32)
    arr = (C.c_char_p * len(inis))(*[str(i).encode() for i in inis])
    addr, port = (master.rsplit(":", 1) if master else ("", 0))
    return lib().shost_run_light_cones(arr, len(inis), dev, len(dev), int(replication), int(fixed_vertex), int(ngp), int(deposit_mode),
                                       int(max_slots), int(rank), int(nranks), addr.encode(), int(port))


def launch_from_env(env, ndev=1):
    """What SLICER_b200 makes of a launcher's environment `env` (a dict): rank, world size, local rank, meeting point and default
    GPU among `ndev`.  Raises ValueError with the driver's message when it would refuse to start."""
    kv = [f"{k}={v}".encode() for k, v in env.items()]
    arr = (C.c_char_p * max(1, len(kv)))(*kv)
    out = np.zeros(5, np.int32)
    addr, err = C.create_string_buffer(256), C.create_string_buffer(1024)
    if lib().shost_launch_from_env(arr, len(kv), ndev, out, addr, 256, err, 1024):
        raise ValueError(err.value.decode())
    return dict(rank=int(out[0]), nranks=int(out[1]), local_rank=int(out[2]), master_addr=addr.value.decode(), master_port=int(out[3]),
                device=int(out[4]))


def subfile_owners(ngpus, ffmin, ffmax):
    """The job's sub-file assignment for ranks that drive ngpus[r] GPUs: -> (rank, local GPU) of each of ffmin .. ffmax-1."""
    ng = np.ascontiguousarray(ngpus, np.int32)
    rank_of, gpu_of = np.zeros(ffmax - ffmin, np.int32), np.zeros(ffmax - ffmin, np.int32)
    if lib().shost_subfile_owners(len(ng), ng, ffmin, ffmax, rank_of, gpu_of):
        raise RuntimeError("a sub-file has two owners")
    return list(zip(rank_of.tolist(), gpu_of.tolist()))


class Group:
    """The driver's control channel between the processes of a job (tests): rank 0 listens on addr:port."""

    OPS = {"min": 0, "max": 1, "sum": 2}

    def __init__(self, rank, nranks, addr, port, timeout_s=60.0):
        rc = C.c_int()
        self.g = lib().shost_group_open(rank, nranks, addr.encode(), port, timeout_s, C.byref(rc))
        self.ok = rc.value == 0

    def close(self):
        if self.g:
            lib().shost_group_close(self.g)
            self.g = None

    def bcast(self, blob=b"", cap=1 << 20):
        buf = C.create_string_buffer(blob, max(cap, len(blob)))
        n = C.c_longlong(len(blob))
        if lib().shost_group_bcast(self.g, buf, C.byref(n), cap):
            raise RuntimeError("bcast failed")
        return buf.raw[: n.value]

    def allgather(self, blob, nranks, cap=1 << 20):
        out = C.create_string_buffer(cap)
        lens = (C.c_longlong * nranks)()
        if lib().shost_group_allgather(self.g, blob, len(blob), out, lens, cap):
            raise RuntimeError("allgather failed")
        res, off = [], 0
        for n in lens:
            res.append(out.raw[off: off + n])
            off += n
        return res

    def allreduce(self, values, op):
        v = (C.c_longlong * len(values))(*values)
        if lib().shost_group_allreduce(self.g, v, len(values), self.OPS[op]):
            raise RuntimeError("allreduce failed")
        return list(v)

    def agree(self, status=0):
        return lib().shost_group_agree(self.g, status)


def read_fits(path):
    """Minimal FITS primary-image reader (tests): -> (header dict, float32 image [NAXIS2, NAXIS1])."""
    raw = open(path, "rb").read()
    hdr = {}
    off = 0
    done = False
    while not done:
        block = raw[off: off + 2880]
        off += 2880
        for i in range(36):
            card = block[80 * i: 80 * (i + 1)].decode("ascii")
            if card.startswith("END"):
                done = True
                break
            if card.startswith("HIERARCH"):
                k, v = card[9:].split("=", 1)
            elif card[8:10] == "= ":
                k, v = card[:8], card[10:]
            else:
                continue
            v = v.split("/")[0].strip()
            k = k.strip()
            if v in ("T", "F"):
                hdr[k] = v == "T"
            else:
                try:
                    hdr[k] = int(v)
                except ValueError:
                    hdr[k] = float(v)
    n1, n2 = hdr["NAXIS1"], hdr["NAXIS2"]
    img = np.frombuffer(raw, dtype=">f4", count=n1 * n2, offset=off).astype(np.float32).reshape(n2, n1)
    return hdr, img
