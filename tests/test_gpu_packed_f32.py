"""The packed FP32 operations of the record kernel (csrc/packed_f32.cuh: FFMA2 / FADD2 / FMUL2 in the float screen and the lean
box transform) round every lane exactly like the scalar __fmaf_rn / __fadd_rn / __fsub_rn / __fmul_rn they stand for: bit
comparison on the device over random operands of every float class (normals, denormals, +-0, +-inf, NaN, and the exponent range
of the box transform)."""
import pytest

from slicer_b200 import capi

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("seed", [1, 2, 3])
def test_packed_f32_lanes_equal_scalar_operations(seed):
    with capi.Slicer(npix_max=64, max_planes=1, mas=capi.MAS_TSC, particle_capacity=1024) as s:
        assert s.selftest_packed(200_000_000, 104729 * seed) == (0, 0, 0, 0)
