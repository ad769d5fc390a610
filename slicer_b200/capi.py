"""ctypes binding of the C ABI in include/slicer_b200.h (slicer_b200/_build/libslicer_b200.so).

This is plumbing for tests, bench.py and the Python front-end: every call goes straight to the CUDA library.
There is no CPU implementation behind it — if the library or a CUDA device is missing, calls raise.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
from typing import Optional, Sequence

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
# SLICER_B200_LIB: another build of the same CUDA library, e.g. the checked one (`make -C slicer_b200/csrc checked`)
LIB_PATH = os.environ.get("SLICER_B200_LIB") or os.path.join(HERE, "_build", "libslicer_b200.so")

MAX_PLANES = 16  # planes per pass
MAX_SLOTS = 64  # plane accumulators per handle (Config.max_planes)
MAX_XFORMS = 8
NTYPES = 6
MAS_TSC, MAS_NGP = 0, 1
LAYOUT_AOS, LAYOUT_SOA = 0, 1
KERNEL_AUTO, KERNEL_SIMPLE, KERNEL_PIPELINED = 0, 1, 2
DEPOSIT_AUTO, DEPOSIT_DIRECT, DEPOSIT_BINNED = 0, 1, 2
KAPPA_MAX_SOURCES = 8
SHEAR_MAX_FFT = 32768


class SlicerError(RuntimeError):
    pass


class Config(C.Structure):
    _fields_ = [
        ("device", C.c_int),
        ("mas", C.c_int),
        ("max_m", C.c_double),
        ("frac_bits", C.c_int),
        ("max_planes", C.c_int),
        ("npix_max", C.c_int),
        ("per_type_maps", C.c_int),
        ("particle_capacity", C.c_size_t),
        ("mass_capacity", C.c_size_t),
        ("kernel", C.c_int),
        ("staging_buffers", C.c_int),
        ("deposit_mode", C.c_int),
        ("record_capacity", C.c_size_t),
        ("guard_eta", C.c_double),
    ]


class PlaneDesc(C.Structure):
    """slicer_plane_desc: what createDensityMaps receives per lens plane (densitymaps.h:161-165)."""

    _fields_ = [
        ("sgn", C.c_int * 3),
        ("face", C.c_int),
        ("centre", C.c_double * 3),
        ("rcase", C.c_float),
        ("ld", C.c_double),
        ("ld2", C.c_double),
        ("nrepperp", C.c_int),
        ("fovradiants", C.c_double),
        ("npix", C.c_int),
    ]


class Stats(C.Structure):
    _fields_ = [
        ("last_deposit_ms", C.c_double),
        ("launches", C.c_ulonglong),
        ("particles_streamed", C.c_ulonglong),
        ("resident_particles", C.c_size_t),
        ("device_bytes", C.c_size_t),
        ("sm_count", C.c_int),
        ("deposit_ms_sum", C.c_double),
        ("deposit_passes", C.c_ulonglong),
        ("deposit_launches", C.c_ulonglong),
        ("flagged_pairs", C.c_ulonglong),
        ("flagged_void", C.c_ulonglong),
    ]


EXPORTS = [
    "slicer_last_error", "slicer_device_count", "slicer_create", "slicer_destroy", "slicer_alloc_pinned",
    "slicer_free_pinned", "slicer_begin_snapshot", "slicer_next_batch", "slicer_stage_particles", "slicer_stage_device",
    "slicer_stage_synthetic", "slicer_download_segment", "slicer_deposit", "slicer_deposit_accumulate",
    "slicer_reduce", "slicer_fetch", "slicer_fetch_fixed", "slicer_synchronize", "slicer_get_stats",
    "slicer_frac_bits", "slicer_comm_unique_id", "slicer_comm_init_rank", "slicer_comm_init_all",
    "slicer_reduce_all", "slicer_wait_staging", "slicer_count_accepted", "slicer_deposit_degraded", "slicer_reset_stats", "slicer_timer_begin", "slicer_timer_end",
    "slicer_selftest_arith", "slicer_selftest_packed", "slicer_deposit_slots", "slicer_reduce_slots", "slicer_reduce_all_slots",
    "slicer_stage_synthetic_window", "slicer_settle_slots", "slicer_device_memory", "slicer_comm_init_ranks",
    "slicer_kernels_run", "slicer_kappa_maps", "slicer_kappa_add", "slicer_kappa_fetch", "slicer_kappa_load",
    "slicer_shear", "slicer_shear_fetch",
]


def build(force: bool = False) -> str:
    """Compile the CUDA library for sm_100a (slicer_b200/csrc/Makefile); no-op when it is up to date."""
    args = ["make", "-s", "-C", os.path.join(HERE, "csrc")]
    if force:
        args.append("-B")
    subprocess.check_call(args)
    return LIB_PATH


_lib = None


def lib() -> C.CDLL:
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise SlicerError(f"{LIB_PATH} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                          "(there is no CPU fallback)")
    L = C.CDLL(LIB_PATH)
    L.slicer_last_error.restype = C.c_char_p
    L.slicer_device_count.argtypes = [C.POINTER(C.c_int)]
    L.slicer_device_memory.argtypes = [C.c_int, C.POINTER(C.c_size_t), C.POINTER(C.c_size_t)]
    L.slicer_create.argtypes = [C.POINTER(Config), C.POINTER(C.c_void_p)]
    L.slicer_destroy.argtypes = [C.c_void_p]
    L.slicer_destroy.restype = None
    L.slicer_alloc_pinned.argtypes = [C.c_size_t, C.POINTER(C.c_void_p)]
    L.slicer_free_pinned.argtypes = [C.c_void_p]
    L.slicer_begin_snapshot.argtypes = [C.c_void_p, C.c_double, C.POINTER(C.c_double), C.c_int]
    L.slicer_next_batch.argtypes = [C.c_void_p]
    L.slicer_reset_stats.argtypes = [C.c_void_p]
    L.slicer_kernels_run.argtypes = [C.c_void_p, C.POINTER(C.c_ulonglong)]
    L.slicer_timer_begin.argtypes = [C.c_void_p]
    L.slicer_selftest_arith.argtypes = [C.c_void_p, C.c_ulonglong, C.c_ulonglong, C.POINTER(C.c_ulonglong)]
    L.slicer_selftest_packed.argtypes = [C.c_void_p, C.c_ulonglong, C.c_ulonglong, C.POINTER(C.c_ulonglong)]
    L.slicer_timer_end.argtypes = [C.c_void_p, C.POINTER(C.c_double)]
    L.slicer_stage_particles.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_size_t]
    L.slicer_stage_device.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_size_t]
    L.slicer_stage_synthetic.argtypes = [C.c_void_p, C.c_int, C.c_size_t, C.c_uint64, C.c_int]
    L.slicer_stage_synthetic_window.argtypes = [C.c_void_p, C.c_int, C.c_ulonglong, C.c_size_t, C.c_uint64, C.c_int]
    L.slicer_download_segment.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]
    L.slicer_deposit.argtypes = [C.c_void_p, C.POINTER(PlaneDesc), C.c_int]
    L.slicer_deposit_accumulate.argtypes = [C.c_void_p, C.POINTER(PlaneDesc), C.c_int]
    L.slicer_reduce.argtypes = [C.c_void_p, C.c_int, C.c_int]
    L.slicer_deposit_slots.argtypes = [C.c_void_p, C.POINTER(PlaneDesc), C.c_int, C.c_int, C.c_int]
    L.slicer_reduce_slots.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int]
    L.slicer_settle_slots.argtypes = [C.c_void_p, C.c_int, C.c_int]
    L.slicer_reduce_all_slots.argtypes = [C.POINTER(C.c_void_p), C.c_int, C.c_int, C.c_int, C.c_int]
    L.slicer_count_accepted.argtypes = [C.c_void_p, C.POINTER(PlaneDesc), C.c_int, C.c_void_p]
    L.slicer_deposit_degraded.argtypes = [C.c_void_p, C.POINTER(PlaneDesc), C.c_int, C.c_int, C.POINTER(C.c_void_p), C.c_int]
    L.slicer_fetch.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]
    L.slicer_fetch_fixed.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p]
    L.slicer_synchronize.argtypes = [C.c_void_p]
    L.slicer_wait_staging.argtypes = [C.c_void_p]
    L.slicer_get_stats.argtypes = [C.c_void_p, C.POINTER(Stats)]
    L.slicer_frac_bits.argtypes = [C.c_void_p]
    L.slicer_comm_unique_id.argtypes = [C.c_char_p]
    L.slicer_comm_init_rank.argtypes = [C.c_void_p, C.c_char_p, C.c_int, C.c_int]
    L.slicer_comm_init_all.argtypes = [C.POINTER(C.c_void_p), C.c_int]
    L.slicer_comm_init_ranks.argtypes = [C.POINTER(C.c_void_p), C.c_int, C.c_char_p, C.c_int, C.c_int]
    L.slicer_reduce_all.argtypes = [C.POINTER(C.c_void_p), C.c_int, C.c_int, C.c_int]
    L.slicer_kappa_maps.argtypes = [C.c_void_p, C.c_int, C.c_int]
    L.slicer_kappa_add.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]
    L.slicer_kappa_fetch.argtypes = [C.c_void_p, C.c_int, C.c_void_p]
    L.slicer_kappa_load.argtypes = [C.c_void_p, C.c_int, C.c_void_p]
    L.slicer_shear.argtypes = [C.c_void_p, C.c_int, C.c_int]
    L.slicer_shear_fetch.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
    _lib = L
    return L


def _check(rc: int) -> None:
    if rc != 0:
        raise SlicerError(lib().slicer_last_error().decode(errors="replace"))


def device_count() -> int:
    n = C.c_int(0)
    _check(lib().slicer_device_count(C.byref(n)))
    return n.value


def device_memory(device: int = 0):
    """-> (free, total) bytes of CUDA device `device`."""
    free, total = C.c_size_t(0), C.c_size_t(0)
    _check(lib().slicer_device_memory(int(device), C.byref(free), C.byref(total)))
    return free.value, total.value


def plane_desc(sgn, face, centre, rcase, ld, ld2, fovradiants, npix, nrepperp=0) -> PlaneDesc:
    d = PlaneDesc()
    d.sgn[:] = [int(v) for v in sgn]
    d.face = int(face)
    d.centre[:] = [float(v) for v in centre]
    d.rcase = float(np.float32(rcase))
    d.ld = float(ld)
    d.ld2 = float(ld2)
    d.nrepperp = int(nrepperp)
    d.fovradiants = float(fovradiants)
    d.npix = int(npix)
    return d


class PinnedBuffer:
    """Page-locked host memory (cudaHostAlloc) exposed as a numpy array."""

    def __init__(self, nbytes: int):
        p = C.c_void_p()
        _check(lib().slicer_alloc_pinned(int(nbytes), C.byref(p)))
        self.ptr = p.value
        self.nbytes = int(nbytes)
        self._raw = (C.c_ubyte * self.nbytes).from_address(self.ptr)

    def view(self, dtype, count: Optional[int] = None, offset: int = 0) -> np.ndarray:
        a = np.frombuffer(self._raw, dtype=dtype, count=-1 if count is None else count, offset=offset)
        return a

    def free(self):
        if self.ptr:
            lib().slicer_free_pinned(C.c_void_p(self.ptr))
            self.ptr = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


class Slicer:
    """One handle = one GPU: staging, the fused deposit pass, reduce, read-back."""

    def __init__(self, npix_max: int, max_planes: int = 4, mas: int = MAS_TSC, particle_capacity: int = 0,
                 mass_capacity: int = 0, per_type_maps: bool = False, device: int = 0, kernel: int = KERNEL_AUTO,
                 frac_bits: int = 0, max_m: float = 1e3, staging_buffers: int = 1, deposit_mode: int = DEPOSIT_AUTO,
                 record_capacity: int = 0, guard_eta: float = 0.0):
        cfg = Config(device=device, mas=mas, max_m=max_m, frac_bits=frac_bits, max_planes=max_planes,
                     npix_max=npix_max, per_type_maps=int(per_type_maps), particle_capacity=particle_capacity,
                     mass_capacity=mass_capacity, kernel=kernel, staging_buffers=staging_buffers, deposit_mode=deposit_mode,
                     record_capacity=record_capacity, guard_eta=guard_eta)
        h = C.c_void_p()
        _check(lib().slicer_create(C.byref(cfg), C.byref(h)))
        self.h = h
        self.cfg = cfg
        self._keep = []  # host buffers that must outlive the async copies

    # -- lifetime ---------------------------------------------------------------------------------
    def close(self):
        if getattr(self, "h", None):
            lib().slicer_destroy(self.h)
            self.h = None

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def frac_bits(self) -> int:
        return lib().slicer_frac_bits(self.h)

    # -- staging ----------------------------------------------------------------------------------
    def begin_snapshot(self, boxsize: float, massarr: Sequence[float] = (0,) * 6, hydro: bool = False):
        arr = (C.c_double * 6)(*[float(v) for v in massarr])
        _check(lib().slicer_begin_snapshot(self.h, float(boxsize), arr, int(hydro)))
        self._keep.clear()

    def next_batch(self):
        _check(lib().slicer_next_batch(self.h))

    def stage(self, ptype: int, pos: np.ndarray, mass: Optional[np.ndarray] = None, layout: int = LAYOUT_AOS):
        """pos: float32 [n,3] (AoS) or [3,n] (SoA); mass: float32 [n] or None."""
        pos = np.ascontiguousarray(pos, np.float32)
        n = pos.shape[0] if layout == LAYOUT_AOS else pos.shape[1]
        if pos.size != 3 * n:
            raise ValueError("positions must be [n,3] (AoS) or [3,n] (SoA)")
        mptr = None
        if mass is not None:
            mass = np.ascontiguousarray(mass, np.float32)
            if mass.size != n:
                raise ValueError("mass must have one entry per particle")
            mptr = mass.ctypes.data
        self._keep.append((pos, mass))
        _check(lib().slicer_stage_particles(self.h, int(ptype), pos.ctypes.data, int(layout), mptr, n))

    def stage_ptr(self, ptype: int, pos_ptr: int, n: int, mass_ptr: int = 0, layout: int = LAYOUT_AOS):
        """Stage from raw host pointers (e.g. a PinnedBuffer): asynchronous when pinned."""
        _check(lib().slicer_stage_particles(self.h, int(ptype), C.c_void_p(pos_ptr), int(layout),
                                            C.c_void_p(mass_ptr) if mass_ptr else None, int(n)))

    def stage_device(self, ptype: int, dev_pos_ptr: int, n: int, dev_mass_ptr: int = 0, layout: int = LAYOUT_AOS):
        _check(lib().slicer_stage_device(self.h, int(ptype), C.c_void_p(dev_pos_ptr), int(layout),
                                         C.c_void_p(dev_mass_ptr) if dev_mass_ptr else None, int(n)))

    def stage_synthetic(self, ptype: int, n: int, seed: int, layout: int = LAYOUT_AOS, start: int = 0):
        _check(lib().slicer_stage_synthetic_window(self.h, int(ptype), int(start), int(n), int(seed), int(layout)))

    def download_segment(self, segment: int, n: int, layout: int = LAYOUT_AOS, with_mass: bool = False):
        pos = np.empty((n, 3) if layout == LAYOUT_AOS else (3, n), np.float32)
        mass = np.empty(n, np.float32) if with_mass else None
        _check(lib().slicer_download_segment(self.h, segment, pos.ctypes.data, mass.ctypes.data if with_mass else None))
        return (pos, mass) if with_mass else pos

    # -- the pass ---------------------------------------------------------------------------------
    @staticmethod
    def _array(planes: Sequence[PlaneDesc]):
        arr = (PlaneDesc * len(planes))()
        for i, p in enumerate(planes):
            C.memmove(C.byref(arr[i]), C.byref(p), C.sizeof(PlaneDesc))
        return arr

    def deposit(self, planes: Sequence[PlaneDesc], accumulate: bool = False):
        arr = planes if isinstance(planes, C.Array) else self._array(planes)
        fn = lib().slicer_deposit_accumulate if accumulate else lib().slicer_deposit
        _check(fn(self.h, arr, len(arr)))

    def deposit_slots(self, planes: Sequence[PlaneDesc], first_slot: int, accumulate: bool = False):
        arr = planes if isinstance(planes, C.Array) else self._array(planes)
        _check(lib().slicer_deposit_slots(self.h, arr, len(arr), int(first_slot), int(accumulate)))

    def reduce_slots(self, first_slot: int, nplanes: int, root: int = 0):
        _check(lib().slicer_reduce_slots(self.h, int(first_slot), int(nplanes), int(root)))

    def selftest_arith(self, n: int, seed: int):
        """(reserved, reserved, mismatches): how many float quotients raw / box of the lean box transform's unchecked division differ
        from __fdiv_rn."""
        out = (C.c_ulonglong * 3)()
        _check(lib().slicer_selftest_arith(self.h, int(n), int(seed), out))
        return tuple(int(v) for v in out)

    def selftest_packed(self, n: int, seed: int):
        """(fma2, add2, sub2, mul2): how many lanes of the kernels' packed FP32 operations differ from the scalar ones."""
        out = (C.c_ulonglong * 4)()
        _check(lib().slicer_selftest_packed(self.h, int(n), int(seed), out))
        return tuple(int(v) for v in out)

    def count_accepted(self, planes: Sequence[PlaneDesc]) -> np.ndarray:
        """-> int64 [nplanes, 6]: accepted (particle, replica) pairs of the resident batch per plane and type."""
        arr = planes if isinstance(planes, C.Array) else self._array(planes)
        out = np.zeros((len(arr), 6), np.int64)
        _check(lib().slicer_count_accepted(self.h, arr, len(arr), out.ctypes.data))
        return out

    def deposit_degraded(self, planes: Sequence[PlaneDesc], snopt: int, keep: Sequence[np.ndarray], accumulate: bool = False):
        """keep[q]: uint8, one entry per accepted pair of plane q in the reference's order (after count_accepted)."""
        arr = planes if isinstance(planes, C.Array) else self._array(planes)
        keep = [np.ascontiguousarray(k, np.uint8) for k in keep]
        ptrs = (C.c_void_p * len(arr))(*[k.ctypes.data if k.size else None for k in keep])
        _check(lib().slicer_deposit_degraded(self.h, arr, len(arr), int(snopt), ptrs, int(accumulate)))

    def reduce(self, nplanes: int, root: int = 0):
        _check(lib().slicer_reduce(self.h, nplanes, root))

    def synchronize(self):
        _check(lib().slicer_synchronize(self.h))

    def settle_slots(self, first_slot: int, nplanes: int):
        """Settle the pairs the passes into these accumulator slots left to the host's libm, without waiting for passes into
        other slots submitted since."""
        _check(lib().slicer_settle_slots(self.h, int(first_slot), int(nplanes)))

    def wait_staging(self):
        _check(lib().slicer_wait_staging(self.h))

    def fetch(self, plane: int, ptype: int = -1, npix: Optional[int] = None, want_map: bool = True):
        """-> (map float32 [npix, npix] indexed [gy, gx] or None, counts int64[6], ingrid int64[6])"""
        npix = npix or self.cfg.npix_max
        out = np.empty(npix * npix, np.float32) if want_map else None
        counts = np.zeros(6, np.int64)
        ingrid = np.zeros(6, np.int64)
        _check(lib().slicer_fetch(self.h, plane, ptype, out.ctypes.data if want_map else None, counts.ctypes.data,
                                  ingrid.ctypes.data))
        return (out.reshape(npix, npix) if want_map else None), counts, ingrid

    def fetch_fixed(self, plane: int, ptype: int = -1, npix: Optional[int] = None) -> np.ndarray:
        npix = npix or self.cfg.npix_max
        out = np.empty(npix * npix, np.int64)
        _check(lib().slicer_fetch_fixed(self.h, plane, ptype, out.ctypes.data))
        return out.reshape(npix, npix)

    # -- convergence maps -------------------------------------------------------------------------
    def kappa_maps(self, nmaps: int, npix: int = 0):
        """Allocate and zero `nmaps` float64 maps of npix^2 on the device (0 frees them)."""
        self._kappa_npix = int(npix or self.cfg.npix_max)
        _check(lib().slicer_kappa_maps(self.h, int(nmaps), self._kappa_npix))

    def kappa_add(self, first_slot: int, maps: Sequence[int], scale, offset):
        """Slots first_slot .. first_slot + len(maps) - 1 in order: map maps[j] + k += scale[j, k] * plane_j + offset[j, k]
        (scale, offset: float64 [nplanes, nsrc]).  Asynchronous."""
        m = np.ascontiguousarray(maps, np.int32)
        sc = np.ascontiguousarray(scale, np.float64).reshape(len(m), -1)
        of = np.ascontiguousarray(offset, np.float64).reshape(sc.shape)
        _check(lib().slicer_kappa_add(self.h, int(first_slot), len(m), m.ctypes.data, sc.shape[1], sc.ctypes.data, of.ctypes.data))

    def kappa_fetch(self, m: int) -> np.ndarray:
        """-> float64 [npix, npix] indexed [gy, gx]"""
        n = getattr(self, "_kappa_npix", self.cfg.npix_max)
        out = np.empty(n * n, np.float64)
        _check(lib().slicer_kappa_fetch(self.h, int(m), out.ctypes.data))
        return out.reshape(n, n)

    def kappa_load(self, m: int, values: np.ndarray):
        v = np.ascontiguousarray(values, np.float64).reshape(-1)
        n = getattr(self, "_kappa_npix", self.cfg.npix_max)
        if v.size != n * n:
            raise ValueError("one value per pixel")
        _check(lib().slicer_kappa_load(self.h, int(m), v.ctypes.data))

    # -- shear maps -------------------------------------------------------------------------------
    def shear(self, m: int, fft_size: int):
        """Enqueue the Kaiser–Squires shear of convergence map `m` on an fft_size^2 grid (a power of two >= npix).  Asynchronous."""
        _check(lib().slicer_shear(self.h, int(m), int(fft_size)))

    def shear_fetch(self):
        """-> (g1, g2) of the last shear(): float64 [npix, npix] indexed [gy, gx]"""
        n = getattr(self, "_kappa_npix", self.cfg.npix_max)
        g1, g2 = np.empty(n * n, np.float64), np.empty(n * n, np.float64)
        _check(lib().slicer_shear_fetch(self.h, g1.ctypes.data, g2.ctypes.data))
        return g1.reshape(n, n), g2.reshape(n, n)

    def reset_stats(self):
        _check(lib().slicer_reset_stats(self.h))

    def kernels_run(self) -> int:
        """Mask of the deposit kernels launched since creation or reset_stats(): bit i = pipelined variant i, bit 40 + mas = the
        simple kernel (include/slicer_b200.h: slicer_kernels_run)."""
        m = C.c_ulonglong(0)
        _check(lib().slicer_kernels_run(self.h, C.byref(m)))
        return m.value

    def timer_begin(self):
        _check(lib().slicer_timer_begin(self.h))

    def timer_end(self) -> float:
        ms = C.c_double()
        _check(lib().slicer_timer_end(self.h, C.byref(ms)))
        return ms.value

    def stats(self) -> Stats:
        st = Stats()
        _check(lib().slicer_get_stats(self.h, C.byref(st)))
        return st

    # -- multi-GPU --------------------------------------------------------------------------------
    @staticmethod
    def comm_unique_id() -> bytes:
        buf = C.create_string_buffer(128)
        _check(lib().slicer_comm_unique_id(buf))
        return buf.raw

    def comm_init_rank(self, uid: bytes, nranks: int, rank: int):
        _check(lib().slicer_comm_init_rank(self.h, uid, nranks, rank))
