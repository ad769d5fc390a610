// aux_kernels.cuh — small helper kernels around the deposit: accumulator read-out and synthetic inputs.
#pragma once
#include <stdint.h>
#include "device_chain.cuh"
#include "packed_f32.cuh"

// int64 fixed point -> float32 map, summing `ntypes` per-type accumulators first (exact integer sum).
// Replaces the float adds of densitymaps.cpp:511-513 and the float MPI_Reduce of slicer-v2.cpp:214-217:
// one rounding per pixel instead of one per particle.
// Masses are non-negative, so an accumulator (or a sum over types) with the sign bit set has run past 2^63 — 8.4e6 mass units per
// pixel at the default 40 fraction bits: `overflow` is raised and the read-out fails instead of returning a wrapped map.
__global__ void finalize_map_kernel(const unsigned long long *__restrict__ acc, unsigned long long type_stride, int ntypes,
                                    unsigned long long npix2, double inv_scale, float *__restrict__ out, unsigned *__restrict__ overflow)
{
  const unsigned long long stride = (unsigned long long)gridDim.x * blockDim.x;
  bool bad = false;
  for (unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; i < npix2; i += stride)
  {
    long long s = 0;
    for (int t = 0; t < ntypes; t++)
    {
      const long long a = (long long)acc[(unsigned long long)t * type_stride + i];
      bad = bad || a < 0;
      s += a;
    }
    bad = bad || s < 0;
    out[i] = __double2float_rn(__dmul_rn((double)s, inv_scale));
  }
  if (bad)
    atomicOr(overflow, 1u);
}

__global__ void sum_types_kernel(const unsigned long long *__restrict__ acc, unsigned long long type_stride, int ntypes,
                                 unsigned long long npix2, long long *__restrict__ out, unsigned *__restrict__ overflow)
{
  const unsigned long long stride = (unsigned long long)gridDim.x * blockDim.x;
  bool bad = false;
  for (unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; i < npix2; i += stride)
  {
    long long s = 0;
    for (int t = 0; t < ntypes; t++)
    {
      const long long a = (long long)acc[(unsigned long long)t * type_stride + i];
      bad = bad || a < 0;
      s += a;
    }
    bad = bad || s < 0;
    out[i] = s;
  }
  if (bad)
    atomicOr(overflow, 1u);
}

// Counter-based generator: 24-bit uniform from splitmix64(seed, 3*i+k), scaled by the box (float multiply).
// slicer_b200/synth_hash.py restates it in numpy so hosts can regenerate any chunk.
__host__ __device__ inline uint64_t synth_mix(uint64_t seed, uint64_t idx)
{
  uint64_t z = seed + (idx + 1ull) * 0x9E3779B97F4A7C15ull;
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
  return z ^ (z >> 31);
}

// `start`: index of the segment's first particle in the realisation (a shard is a window of one realisation)
__global__ void synth_positions_kernel(float *__restrict__ pos, unsigned long long n, unsigned long long soa_stride,
                                       int layout_soa, uint64_t seed, float boxf, unsigned long long start)
{
  const unsigned long long total = 3ull * n;
  const unsigned long long stride = (unsigned long long)gridDim.x * blockDim.x;
  for (unsigned long long j = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; j < total; j += stride)
  {
    unsigned long long i, k;
    if (layout_soa)
    {
      k = j / n;
      i = j - k * n;
    }
    else
    {
      i = j / 3ull;
      k = j - 3ull * i;
    }
    const float u = (float)(synth_mix(seed, 3ull * (start + i) + k) >> 40) * (1.0f / 16777216.0f);
    const float v = __fmul_rn(u, boxf);
    if (layout_soa)
      pos[k * soa_stride + i] = v;
    else
      pos[j] = v;
  }
}


// ---- arithmetic self-check -------------------------------------------------------------------------------------------------
__device__ __forceinline__ unsigned long long selftest_mix(unsigned long long z)
{
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
  return z ^ (z >> 31);
}

// The unchecked float division of the lean box transform (deposit_pipelined.cuh: lean_div_box) against __fdiv_rn:
// n random (raw coordinate, box size) pairs, box in [2^-40, 2^40), raw in [2^-40, box].  out[2] += quotients that differ.
__device__ __forceinline__ float selftest_box_rcp(float boxf)
{
  const float y0 = lean_rcp_seed(boxf);
  return __fmaf_rn(y0, __fmaf_rn(y0, -boxf, 1.0f), y0);
}
__global__ void selftest_fdiv_kernel(unsigned long long n, unsigned long long seed, unsigned long long *out)
{
  unsigned long long bad = 0;
  const unsigned long long stride = (unsigned long long)gridDim.x * blockDim.x;
  for (unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride)
  {
    const unsigned long long h1 = selftest_mix(seed + 2 * i), h2 = selftest_mix(seed + 2 * i + 1);
    // a few boxes per warp iteration would hide nothing: every sample draws its own box (random mantissa and exponent)
    const float b = __uint_as_float((unsigned)(h1 & 0x007fffffu) | ((unsigned)(127 - 40 + (h1 >> 32) % 80) << 23));
    // raw = box * U(0,1] with a random mantissa, sometimes the box itself or a tiny value
    float u = __uint_as_float((unsigned)(h2 & 0x007fffffu) | ((unsigned)(127 - 40 + (h2 >> 32) % 80) << 23));
    if (u > b)
      u = __fmul_rn(b, __uint_as_float((unsigned)(h2 & 0x007fffffu) | (126u << 23))); // b * [0.5, 1)
    if ((h2 >> 60) == 0)
      u = b;
    if (!(u >= 0x1p-40f))
      u = 0x1p-40f;
    const float yb = selftest_box_rcp(b);
    const float q0 = __fmul_rn(u, yb);
    const float r = __fmaf_rn(q0, -b, u);
    const float q = __fmaf_rn(yb, r, q0);
    bad += __float_as_uint(q) != __float_as_uint(__fdiv_rn(u, b));
  }
  if (bad)
    atomicAdd(out + 2, bad);
}

// The packed FP32 helpers (packed_f32.cuh) against their scalar counterparts, lane by lane: n random operand sets, each operand
// drawn from every class (any bit pattern: normals, denormals, +-0, +-inf, NaN; denormals; special values; normals of the box
// transform's exponent range).  out[0..3] += fma2 / add2 / sub2 / mul2 lanes whose bits differ (two NaNs count as equal).
__device__ __forceinline__ float selftest_operand(unsigned long long h)
{
  const unsigned m = (unsigned)h;
  switch ((unsigned)(h >> 61))
  {
  case 0:
  case 1:
    return __uint_as_float(m);
  case 2:
    return __uint_as_float(m & 0x807fffffu); // denormal or +-0
  case 3:
  {
    const unsigned sp[8] = {0x00000000u, 0x7f800000u, 0x7fc00000u, 0x3f800000u, 0x3f000000u, 0x00800000u, 0x7f7fffffu, 0x00000001u};
    return __uint_as_float(sp[m & 7u] | (m & 0x80000000u));
  }
  default:
    return __uint_as_float((m & 0x807fffffu) | ((unsigned)(127 - 45 + (h >> 32) % 91) << 23));
  }
}
__device__ __forceinline__ unsigned long long selftest_differs(float2 p, float a, float b)
{
  const bool dx = __float_as_uint(p.x) != __float_as_uint(a) && !(isnan(p.x) && isnan(a));
  const bool dy = __float_as_uint(p.y) != __float_as_uint(b) && !(isnan(p.y) && isnan(b));
  return (unsigned long long)dx + (unsigned long long)dy;
}
__global__ void selftest_packed_kernel(unsigned long long n, unsigned long long seed, unsigned long long *out)
{
  unsigned long long bad[4] = {0, 0, 0, 0};
  const unsigned long long stride = (unsigned long long)gridDim.x * blockDim.x;
  for (unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride)
  {
    float v[6];
#pragma unroll
    for (int k = 0; k < 6; k++)
      v[k] = selftest_operand(selftest_mix(seed + 6 * i + k));
    const float2 a = make_float2(v[0], v[1]), b = make_float2(v[2], v[3]), c = make_float2(v[4], v[5]);
    bad[0] += selftest_differs(fma2_rn(a, b, c), __fmaf_rn(a.x, b.x, c.x), __fmaf_rn(a.y, b.y, c.y));
    bad[1] += selftest_differs(add2_rn(a, b), __fadd_rn(a.x, b.x), __fadd_rn(a.y, b.y));
    bad[2] += selftest_differs(sub2_rn(a, b), __fsub_rn(a.x, b.x), __fsub_rn(a.y, b.y));
    bad[3] += selftest_differs(mul2_rn(a, b), __fmul_rn(a.x, b.x), __fmul_rn(a.y, b.y));
  }
#pragma unroll
  for (int k = 0; k < 4; k++)
    if (bad[k])
      atomicAdd(out + k, bad[k]);
}
