// shear.cuh — shear maps: Kaiser–Squires γ1, γ2 of a convergence map through a deterministic, zero-padded FFT.
//
// κ is the double map of slicer_kappa_* (element k[gx + npix*gy]); axis 1 is gx, axis 2 is gy; pixels are square in angle.
//   1. Embed: K[x, y] = k[x, y] for x, y < npix, 0 elsewhere on a P x P grid (P a power of two >= npix; the driver takes the
//      smallest >= 2 npix, so that mass near one edge does not wrap onto the opposite one: κ is taken as 0 outside the field).
//   2. Forward: K^ = DFT2(K), kernel e^(-2 pi i (f1 x + f2 y) / P).
//   3. Multiply: s = f for f < P/2, f - P otherwise; d = s1^2 + s2^2 (exact); D1 = (s1^2 - s2^2) / d, D2 = (2 s1 s2) / d;
//      D1 = D2 = 0 at (0, 0); D2 = 0 where s1 or s2 is -P/2 (the odd factor breaks the Hermitian pairing there; zeroing it keeps
//      γ2 real).  Γ^ = (D1 + i D2) K^ in real operations: re = D1 Kr - D2 Ki, im = D1 Ki + D2 Kr.
//   4. Inverse: Γ = DFT2^-1(Γ^) * (1/P^2) (an exact power of two); γ1 = Re Γ, γ2 = Im Γ on x, y < npix.
//      Equivalently γ1 = (∂1² - ∂2²)ψ / 2, γ2 = ∂1∂2ψ with ∇²ψ = 2κ, in the map's own axes.
//
// The transform along one axis is a fixed sequence of Stockham stages: radix 4 while at least 4 points remain per sub-transform,
// then one radix 2.  A stage of radix R on sub-transforms of n points (m = P / (n R)) takes x[q m n + g n + j] (q < R, g < m,
// j < n), multiplies x_q for q >= 1 by the table's w^(q j m) (forward: (a c + b s, b c - a s), inverse: (a c - b s, b c + a s),
// (c, s) = (cos, sin)(2 pi k / P)), and writes the exact radix-R DFT of the R values (±1, ±i only; radix 4 as
// a0 = t0 + t2, a1 = t0 - t2, a2 = t1 + t3, a3 = t1 - t3, y0 = a0 + a2, y2 = a0 - a2, and y1, y3 = a1 ∓ i a3 forward, a1 ± i a3
// inverse) to y[g R n + r n + j].  The table holds cos(2.0*M_PI*k/P), sin(2.0*M_PI*k/P) for k < P, from the host's libm.
// Order: forward rows (y < npix only: the other rows are zero and stay +0), forward columns (all P), multiply, inverse columns
// (all P), inverse rows (y < npix only: the window).  Every operation is an IEEE double round-to-nearest operation
// (__dmul_rn / __dadd_rn / __dsub_rn / __ddiv_rn), every output element is written by one thread, nothing is atomic: the maps are
// a function of κ and P alone.  tests/test_gpu_shear.py restates the sequence in numpy and matches it bit for bit.
//
// A kernel launch runs two consecutive stages (RA then RB; RB = 1: one) in registers: the RA x RB values a thread loads are
// exactly the inputs of RB butterflies of the second stage's RA groups, so the arithmetic is that of the two stages one after the
// other and the data cross memory once per pair.  The first forward pass reads κ itself (zero outside the window), the first
// forward column pass reads +0 for the rows the row passes skipped, the last forward pass applies the multiplier, and the last
// inverse pass scales and writes γ1 and γ2.
#pragma once
#include "pass_params.h"

#define SHEAR_MAX_FFT SLICER_SHEAR_MAX_FFT

enum
{
  SHEAR_IN_KAPPA = 1,  // read κ (double, npix^2) instead of src; 0 for x >= npix
  SHEAR_IN_ZERO = 2,   // elements along the axis at or beyond npix are +0, not read
  SHEAR_OUT_MULT = 4,  // multiply the output by D1 + i D2 (columns: the line is f1, the output index f2)
  SHEAR_OUT_GAMMA = 8, // write scale * (re, im) of x < npix to g1, g2 (rows)
};

struct ShearArgs
{
  const double2 *src; // P x P, element [x + P y]
  double2 *dst;
  const double *kappa; // SHEAR_IN_KAPPA
  const double2 *tw;   // P entries: (cos, sin)(2 pi k / P)
  double *g1, *g2;     // SHEAR_OUT_GAMMA: npix^2 each, element [x + npix y]
  double scale;        // 1 / P^2
  int P, npix, n, nlines, flags;
};

__device__ __forceinline__ double2 shear_cadd(double2 a, double2 b) { return make_double2(__dadd_rn(a.x, b.x), __dadd_rn(a.y, b.y)); }
__device__ __forceinline__ double2 shear_csub(double2 a, double2 b) { return make_double2(__dsub_rn(a.x, b.x), __dsub_rn(a.y, b.y)); }

// x * w^k, w = e^(-+2 pi i / P)
template <bool INV>
__device__ __forceinline__ double2 shear_twiddle(double2 x, double2 w)
{
  if (INV)
    return make_double2(__dsub_rn(__dmul_rn(x.x, w.x), __dmul_rn(x.y, w.y)), __dadd_rn(__dmul_rn(x.y, w.x), __dmul_rn(x.x, w.y)));
  return make_double2(__dadd_rn(__dmul_rn(x.x, w.x), __dmul_rn(x.y, w.y)), __dsub_rn(__dmul_rn(x.y, w.x), __dmul_rn(x.x, w.y)));
}

// one stage on v[0], v[S], .., v[(R-1) S] in place: twiddles w^(q j m) for q >= 1, then the exact radix-R DFT
template <int R, bool INV, int S>
__device__ __forceinline__ void shear_stage(double2 *v, const double2 *tw, int j, int m, int P)
{
#pragma unroll
  for (int q = 1; q < R; q++)
  {
    const int k = q * j * m;
    SLICER_CHECK(k >= 0 && k < P);
    v[q * S] = shear_twiddle<INV>(v[q * S], __ldg(tw + k));
  }
  if (R == 2)
  {
    const double2 a = v[0], b = v[S];
    v[0] = shear_cadd(a, b);
    v[S] = shear_csub(a, b);
  }
  else
  {
    const double2 a0 = shear_cadd(v[0], v[2 * S]), a1 = shear_csub(v[0], v[2 * S]);
    const double2 a2 = shear_cadd(v[S], v[3 * S]), a3 = shear_csub(v[S], v[3 * S]);
    const double2 p = make_double2(__dadd_rn(a1.x, a3.y), __dsub_rn(a1.y, a3.x)); // a1 - i a3
    const double2 mi = make_double2(__dsub_rn(a1.x, a3.y), __dadd_rn(a1.y, a3.x)); // a1 + i a3
    v[0] = shear_cadd(a0, a2);
    v[2 * S] = shear_csub(a0, a2);
    v[S] = INV ? mi : p;
    v[3 * S] = INV ? p : mi;
  }
}

// D1 + i D2 at signed frequencies (s1, s2), times z
__device__ __forceinline__ double2 shear_multiply(double2 z, int f1, int f2, int P)
{
  const int s1 = f1 < P / 2 ? f1 : f1 - P, s2 = f2 < P / 2 ? f2 : f2 - P;
  double D1 = 0.0, D2 = 0.0;
  if (s1 != 0 || s2 != 0)
  {
    const double a = (double)s1, b = (double)s2;
    const double d = __dadd_rn(__dmul_rn(a, a), __dmul_rn(b, b));
    D1 = __ddiv_rn(__dsub_rn(__dmul_rn(a, a), __dmul_rn(b, b)), d);
    D2 = (s1 == -P / 2 || s2 == -P / 2) ? 0.0 : __ddiv_rn(__dmul_rn(__dmul_rn(2.0, a), b), d);
  }
  return make_double2(__dsub_rn(__dmul_rn(D1, z.x), __dmul_rn(D2, z.y)), __dadd_rn(__dmul_rn(D1, z.y), __dmul_rn(D2, z.x)));
}

// Stages (RA on sub-transforms of n points, then RB on RA n points) along AXIS (0: rows, x; 1: columns, y) of A.nlines lines.
// One thread per (line, g', j): AXIS 1 puts consecutive columns on consecutive threads, AXIS 0 consecutive j (or g' when n = 1):
// both load and store consecutive 16-byte elements across a warp.
template <int RA, int RB, bool INV, int AXIS>
__global__ void __launch_bounds__(256) shear_fft_pass(const ShearArgs A)
{
  const int P = A.P, n = A.n;
  const int B = P / (RA * RB); // threads per line
  const size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= (size_t)A.nlines * B)
    return;
  const int line = AXIS ? (int)(t % P) : (int)(t / B);
  const int b = AXIS ? (int)(t / P) : (int)(t % B);
  const int j = b % n, gp = b / n;
  const int m = P / (RA * n), mb = m / RB;
  SLICER_CHECK(line < A.nlines && gp < mb && RA * RB * n * mb == P);
  const size_t es = AXIS ? (size_t)P : 1, base = AXIS ? (size_t)line : (size_t)line * P;
  double2 v[RA * RB]; // v[qb * RA + q]: input q of stage A in its group g = qb mb + gp
#pragma unroll
  for (int qb = 0; qb < RB; qb++)
#pragma unroll
    for (int q = 0; q < RA; q++)
    {
      const int e = q * m * n + (qb * mb + gp) * n + j;
      SLICER_CHECK(e < P);
      double2 x;
      if (A.flags & SHEAR_IN_KAPPA)
        x = e < A.npix ? make_double2(A.kappa[(size_t)line * A.npix + e], 0.0) : make_double2(0.0, 0.0);
      else if ((A.flags & SHEAR_IN_ZERO) && e >= A.npix)
        x = make_double2(0.0, 0.0);
      else
        x = A.src[base + e * es];
      v[qb * RA + q] = x;
    }
#pragma unroll
  for (int qb = 0; qb < RB; qb++)
    shear_stage<RA, INV, 1>(v + qb * RA, A.tw, j, m, P); // output r of group qb*mb + gp -> v[qb * RA + r]
  const int n2 = RA * n;
  if (RB > 1)
#pragma unroll
    for (int r = 0; r < RA; r++)
      shear_stage<RB, INV, RA>(v + r, A.tw, r * n + j, mb, P); // output rb of (gp, r n + j) -> v[rb * RA + r]
#pragma unroll
  for (int rb = 0; rb < RB; rb++)
#pragma unroll
    for (int r = 0; r < RA; r++)
    {
      const int o = gp * RB * n2 + rb * n2 + r * n + j;
      SLICER_CHECK(o < P);
      double2 y = v[rb * RA + r];
      if (A.flags & SHEAR_OUT_MULT)
        y = shear_multiply(y, line, o, P);
      if (A.flags & SHEAR_OUT_GAMMA)
      {
        if (o < A.npix)
        {
          SLICER_CHECK(line < A.npix);
          A.g1[(size_t)line * A.npix + o] = __dmul_rn(y.x, A.scale);
          A.g2[(size_t)line * A.npix + o] = __dmul_rn(y.y, A.scale);
        }
      }
      else
        A.dst[base + o * es] = y;
    }
}
