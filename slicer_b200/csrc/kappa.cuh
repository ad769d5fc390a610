// kappa.cuh — convergence maps: the Born sum of the lens planes of one light cone, formed where the planes are.
//
// For every map m = run_map[r] + k of a run r of consecutive planes (one realisation's planes of a call), per pixel p:
//   kappa_m[p] = kappa_m[p] + (scale[j][k] * (double(acc_j[p]) * 2^-frac_bits) + offset[j][k])      for j in the run, in order
// with acc_j[p] the int64 accumulator summed over the particle types.  Every operation is a round-to-nearest double
// operation in exactly this order (no contraction), and every pixel is owned by one thread, so the result does not depend on
// how the planes of a light cone are split over calls, GPUs or processes: it is a function of the integer planes alone.
// A thread loads each kappa value of a run once, applies all planes of the run and stores it once: the traffic of a call is
// 8 B x npix^2 x (planes x types) of plane reads plus one read and one write of each map touched.
#pragma once
#include "pass_params.h"

#define KAPPA_MAX_PLANES SLICER_MAX_SLOTS

// Everything a call needs, passed by value (kernel parameters: uniform loads through the constant cache).  The host builds it
// in slicer_kappa_add: planes [0, nplanes) are the call's slots in order; run r covers planes [run_begin[r], run_begin[r+1]).
struct KappaArgs
{
  const unsigned long long *acc; // accumulator of the call's first slot
  double *maps;                  // map m starts at maps + m * map_stride
  unsigned *map_ovf;             // one flag per map: a summed accumulator had its sign bit set
  unsigned long long slot_stride, type_stride, map_stride, npix2;
  double inv_scale; // 2^-frac_bits
  int ntypes, nsrc, nruns, nmaps;
  int run_begin[KAPPA_MAX_PLANES + 1];
  int run_map[KAPPA_MAX_PLANES];
  unsigned run_mask[KAPPA_MAX_PLANES];   // sources some plane of the run contributes to (bit k)
  unsigned plane_mask[KAPPA_MAX_PLANES]; // sources plane j contributes to: (scale, offset) != (0, 0)
  double scale[KAPPA_MAX_PLANES * SLICER_KAPPA_MAX_SOURCES], offset[KAPPA_MAX_PLANES * SLICER_KAPPA_MAX_SOURCES];
};

// one plane term of one source, in the contract's order: scale * (double(acc) * 2^-frac_bits) + offset
__device__ __forceinline__ double kappa_term(double scale, long long s, double inv_scale, double offset)
{
  return __dadd_rn(__dmul_rn(scale, __dmul_rn((double)s, inv_scale)), offset);
}

// VEC: two pixels per thread and iteration with 16-byte loads and stores (every slot, type and map starts on a 16-byte boundary,
// npix2 pairs); otherwise one pixel.  Grid-stride loop over pixel groups, sized like finalize_map_kernel.
template <bool VEC>
__global__ void __launch_bounds__(256) kappa_add_kernel(const KappaArgs A)
{
  constexpr int W = VEC ? 2 : 1;
  const unsigned long long ngroups = A.npix2 / W;
  const unsigned long long stride = (unsigned long long)gridDim.x * blockDim.x;
  for (unsigned long long g = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; g < ngroups; g += stride)
  {
    const unsigned long long i = g * W;
    for (int r = 0; r < A.nruns; r++)
    {
      const unsigned rmask = A.run_mask[r];
      if (!rmask)
        continue;
      double kv[SLICER_KAPPA_MAX_SOURCES][W];
#pragma unroll
      for (int k = 0; k < SLICER_KAPPA_MAX_SOURCES; k++)
        if (rmask >> k & 1u)
        {
          const unsigned long long m = (unsigned long long)(A.run_map[r] + k);
          SLICER_CHECK(i + W <= A.npix2 && m < (unsigned long long)A.nmaps && (!VEC || ((A.map_stride & 1ull) == 0)));
          const double *src = A.maps + m * A.map_stride + i;
          if (VEC)
          {
            const double2 v = *reinterpret_cast<const double2 *>(src);
            kv[k][0] = v.x;
            kv[k][W - 1] = v.y;
          }
          else
            kv[k][0] = src[0];
        }
      bool bad = false;
      for (int j = A.run_begin[r]; j < A.run_begin[r + 1]; j++)
      {
        SLICER_CHECK(j >= 0 && j < KAPPA_MAX_PLANES);
        const unsigned pmask = A.plane_mask[j];
        if (!pmask)
          continue;
        long long s[W];
#pragma unroll
        for (int w = 0; w < W; w++)
          s[w] = 0;
        for (int t = 0; t < A.ntypes; t++)
        {
          const unsigned long long *src = A.acc + (unsigned long long)j * A.slot_stride + (unsigned long long)t * A.type_stride + i;
          long long a[W];
          if (VEC)
          {
            const longlong2 v = *reinterpret_cast<const longlong2 *>(src);
            a[0] = v.x;
            a[W - 1] = v.y;
          }
          else
            a[0] = (long long)src[0];
#pragma unroll
          for (int w = 0; w < W; w++)
          {
            bad = bad || a[w] < 0;
            s[w] += a[w];
          }
        }
#pragma unroll
        for (int w = 0; w < W; w++)
          bad = bad || s[w] < 0;
#pragma unroll
        for (int k = 0; k < SLICER_KAPPA_MAX_SOURCES; k++)
          if (pmask >> k & 1u)
          {
            const double sc = A.scale[j * SLICER_KAPPA_MAX_SOURCES + k], of = A.offset[j * SLICER_KAPPA_MAX_SOURCES + k];
#pragma unroll
            for (int w = 0; w < W; w++)
              kv[k][w] = __dadd_rn(kv[k][w], kappa_term(sc, s[w], A.inv_scale, of));
          }
      }
#pragma unroll
      for (int k = 0; k < SLICER_KAPPA_MAX_SOURCES; k++)
        if (rmask >> k & 1u)
        {
          const unsigned long long m = (unsigned long long)(A.run_map[r] + k);
          double *dst = A.maps + m * A.map_stride + i;
          if (VEC)
            *reinterpret_cast<double2 *>(dst) = make_double2(kv[k][0], kv[k][W - 1]);
          else
            dst[0] = kv[k][0];
          if (bad)
            atomicOr(A.map_ovf + m, 1u);
        }
    }
  }
}
