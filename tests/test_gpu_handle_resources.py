"""Lifetime of a handle's CUDA resources (slicer_capi.cu): a refused allocation leaves the thread and the handle usable, and
`device_bytes` counts what the handle holds across re-allocations.

Allocations are made to fail only with requests larger than any B200 holds: the runtime refuses them with an ordinary error
return, and no memory is taken from other work on the device."""
import numpy as np
import pytest

from slicer_b200 import capi

pytestmark = pytest.mark.gpu

BOX, NPIX, N = 128000.0, 64, 1 << 16
PLANE = capi.plane_desc([1, -1, 1], 3, [0.904897332, 0.377652943, 0.164757043], 1.0, 160.0, 192.0, 0.35, NPIX)


def handle():
    return capi.Slicer(npix_max=NPIX, max_planes=1, particle_capacity=N + 64)


def deposit_and_fetch(s):
    s.begin_snapshot(BOX, [0, 1.0375, 0, 0, 0, 0], False)
    s.stage_synthetic(1, N, 11)
    s.deposit([PLANE])
    return s.fetch_fixed(0, -1, NPIX)


def kappa_and_shear(s):
    """κ maps, a deposit, κ of it, its shear -> every array read back"""
    s.kappa_maps(2, NPIX)
    plane = deposit_and_fetch(s)
    s.kappa_add(0, [0], [[1e-3, 2e-3]], [[-1e-4, -2e-4]])
    kappa = [s.kappa_fetch(m) for m in range(2)]
    s.shear(0, 128)
    return [plane, *kappa, *s.shear_fetch()]


def same_bits(a, b):
    return len(a) == len(b) and all(x.dtype == y.dtype and x.tobytes() == y.tobytes() for x, y in zip(a, b))


def test_a_refused_create_leaves_the_thread_usable():
    """A staging pool of about 400 TB is refused; the next launches on this thread, on an old handle and on a new one, run."""
    with handle() as a:
        first = deposit_and_fetch(a)
        assert first.sum() > 0
        with pytest.raises(capi.SlicerError, match="cudaMalloc"):
            capi.Slicer(npix_max=NPIX, particle_capacity=1 << 45)
        assert same_bits([deposit_and_fetch(a)], [first])
        with handle() as b:
            assert same_bits([deposit_and_fetch(b)], [first])


def test_a_refused_kappa_allocation_leaves_the_handle_usable_and_counted():
    with handle() as s, handle() as fresh:
        bare = s.stats().device_bytes
        s.kappa_maps(3, NPIX)
        assert s.stats().device_bytes > bare
        with pytest.raises(capi.SlicerError, match="cudaMalloc"):
            s.kappa_maps(2**31 - 1, NPIX)  # 70 TB of maps
        assert s.stats().device_bytes == bare == fresh.stats().device_bytes
        got = kappa_and_shear(s)
        want = kappa_and_shear(fresh)
    assert np.std(got[1]) > 0 and np.std(got[3]) > 0
    assert same_bits(got, want)


def test_device_bytes_across_reallocation():
    with handle() as s, handle() as fresh:
        before = s.stats().device_bytes
        s.kappa_maps(3, NPIX)
        assert s.stats().device_bytes > before
        s.kappa_maps(0)
        assert s.stats().device_bytes == before
        for h in (s, fresh):
            h.kappa_maps(1, NPIX)
        s.shear(0, 256)
        s.shear(0, 128)
        fresh.shear(0, 128)
        assert s.stats().device_bytes == fresh.stats().device_bytes
