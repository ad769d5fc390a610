// lean_math.h — the projection of an accepted-candidate particle in ~55 double-precision instructions, with a rigorous
// ambiguity guard.  Shared verbatim by the CUDA kernels (deposit_pipelined.cuh) and by the host-side error-budget check
// (tools/lean_math_check.c, tests/test_lean_math.py), so the formulas that run on the GPU are the ones checked on the CPU.
//
// What the reference computes (densitymaps.cpp:382-386, utilities.cpp:23-25), all in double, no FMA:
//     X = x - 0.5, Y = y - 0.5, Z = z          (x, y, z are floats)
//     d = sqrt(X*X + Y*Y + Z*Z);  dec = asin(X/d);  ra = atan2(Y, Z)           [glibc libm]
//     accept <=> fabs(ra) <= T && fabs(dec) <= T
//     xs = float(dec/fov + 0.5),  ys = float(ra/fov + 0.5)
// What only matters downstream: the accept decision and the two FLOATS xs, ys.
//
// The lean evaluation computes w = dec/fov and v = w + 0.5 directly (1/fov folded into the series coefficients) from
// X * rsqrt(d^2) and Y * rcp(Z) (float MUFU seeds refined by one third-order Newton step in double), with the odd
// Maclaurin series of asin / atan (narrow fields: |arg| <= arg_lim <= 0.385).  Error budget, relative to |w|, in units of
// u = 2^-53:
//     reference:  d 2u, X/d 1u, glibc asin / atan2 <= 1u (documented bound), dec/fov 1u              -> <= 5.5u
//     lean:       d^2 1.5u, rsqrt 2u (Newton residual 2^-64 + three roundings), X*r 1u, series (truncation <= 1u by the
//                 choice of K, coefficient rounding 1u, Horner roundings scaled by arg^2 <= 0.15), final fma 1u  -> <= 8u
//   so |w_lean - w_ref| <= 13.5u * |w| <= 2^-49.2 * 0.51 and, with the two roundings of v (<= 2^-54 each),
//   |v_lean - v_ref| < 2^-49.9.  The guard uses ETA = 2^-47: 7.5x the bound.
// A particle is FLAGGED when a decision could differ within ETA: |w| within ETA of the field threshold T/fov, or v within ETA of
// a float rounding boundary (float(v - ETA) != float(v + ETA)).  Flagged particles (a few per million) are recomputed with
// the host's libm exactly as the reference does (slicer_capi.cu: resolve_deferred); everything else provably yields the
// reference's bits.
#pragma once
#include <math.h>

#if defined(__CUDACC__)
#define LEAN_HD __host__ __device__ __forceinline__
#else
#define LEAN_HD static inline
#endif

#define LEAN_MAX_TERMS 20
#define LEAN_ETA 0x1p-47

// Per-pass constants of the lean projection (uniform over the pass: every plane shares field and map size).
struct LeanDev
{
  int enabled;   // the pass qualifies (slicer_capi.cu: build_pass) and the box is in the fast transform's range
  int K;         // series terms beyond the linear one: asin(s) ~ s + s^3 (a_1 + a_2 s^2 + ... + a_K s^(2K-2))
  double A;      // 1 / fovradiants
  double w_in;   // |w| <= w_in   => inside the field for sure        (T/fov - ETA)
  double w_out;  // |w| >  w_out  => outside for sure                  (T/fov + ETA)
  double eta;    // the guard: LEAN_ETA, or wider (slicer_config::guard_eta: more particles take the host's libm path)
  double arg_lim; // series validity: |X/d|, |Y/Z| beyond it cannot be accepted (> tan T / cos T)
  double cs[LEAN_MAX_TERMS + 1]; // A * asin coefficients a_k, k = 1..K  (index 0 unused)
  double ct[LEAN_MAX_TERMS + 1]; // A * atan coefficients
  float umin;    // raw coordinates in (umin, raw_hi) take the fast box transform (no wrap at the first site, normal quotient)
};

#if defined(__CUDA_ARCH__)
#define LEAN_FMA(a, b, c) __fma_rn((a), (b), (c))
LEAN_HD float lean_rsqrt_seed(float x)
{
  float r;
  asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
  return r;
}
LEAN_HD float lean_rcp_seed(float x)
{
  float r;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
  return r;
}
#else
#define LEAN_FMA(a, b, c) fma((a), (b), (c))
// host stand-ins for the MUFU seeds: correctly rounded value times (1 + LEAN_SEED_ERR), |err| up to 2^-21.5 (worse than the
// documented 2^-22.9 / 1 ulp of rsqrt.approx.f32 / rcp.approx.f32); the check sweeps the perturbation
#ifndef LEAN_SEED_ERR
#define LEAN_SEED_ERR 0.0f
#endif
LEAN_HD float lean_rsqrt_seed(float x) { return (1.0f / sqrtf(x)) * (1.0f + (LEAN_SEED_ERR)); }
LEAN_HD float lean_rcp_seed(float x) { return (1.0f / x) * (1.0f + (LEAN_SEED_ERR)); }
#endif

// s = X / sqrt(X^2 + Y^2 + Z^2) and t = Y / Z to ~1.5 ulp, without division or square root instructions
LEAN_HD void lean_ratios(float x, float y, float z, double *s, double *t)
{
  const double X = (double)x - 0.5, Y = (double)y - 0.5, Z = (double)z; // exact: x, y are floats in [0, 1]
  const double d2 = LEAN_FMA(Z, Z, LEAN_FMA(Y, Y, X * X));
  double r = (double)lean_rsqrt_seed((float)d2);
  {
    const double g = d2 * r;                 // ~ sqrt(d2)
    const double e = LEAN_FMA(-g, r, 1.0);   // 1 - d2 r^2  (|e| <~ 2^-21)
    const double c = LEAN_FMA(e, 0.375, 0.5);
    r = LEAN_FMA(c, r * e, r);               // r (1 + e/2 + 3 e^2 / 8): third order
  }
  *s = X * r;
  double iz = (double)lean_rcp_seed(z);
  {
    double e = LEAN_FMA(-Z, iz, 1.0); // |e| <= 2^-22
    e = LEAN_FMA(e, e, e);
    iz = LEAN_FMA(iz, e, iz); // iz (1 + e + e^2): third order
  }
  *t = Y * iz;
}

// w = (1/fov) * f(a) for the odd series f with pre-scaled coefficients c[1..K]; a*A is the linear term
LEAN_HD double lean_series(double a, const double *c, int K, double A)
{
  const double z = a * a;
  double p = c[K];
  for (int k = K - 1; k >= 1; k--)
    p = LEAN_FMA(p, z, c[k]);
  return LEAN_FMA(a * z, p, a * A);
}

enum { LEAN_REJECT = 0, LEAN_ACCEPT = 1, LEAN_FLAGGED = 2 };

// Decision and map coordinates from w (= angle / fov) of both axes.  ACCEPT: xs, ys are the reference's floats.
LEAN_HD int lean_classify(double wx, double wy, const LeanDev &L, float *xs, float *ys)
{
  const double ax = fabs(wx), ay = fabs(wy);
  if (!(ax <= L.w_out && ay <= L.w_out))
  { // outside for sure — unless a NaN got here (z == 0, a degenerate particle at the observer): let the host decide
    return (ax > L.w_out || ay > L.w_out) ? LEAN_REJECT : LEAN_FLAGGED;
  }
  const double vx = wx + 0.5, vy = wy + 0.5;
  const float x_lo = (float)(vx - L.eta), x_hi = (float)(vx + L.eta);
  const float y_lo = (float)(vy - L.eta), y_hi = (float)(vy + L.eta);
  *xs = x_lo;
  *ys = y_lo;
  const bool sure = ax <= L.w_in && ay <= L.w_in && x_lo == x_hi && y_lo == y_hi;
  return sure ? LEAN_ACCEPT : LEAN_FLAGGED;
}

// the whole lean projection of one particle (the kernels interleave two of these per lane)
LEAN_HD int lean_project(float x, float y, float z, const LeanDev &L, float *xs, float *ys)
{
  double s, t;
  lean_ratios(x, y, z, &s, &t);
  if (fabs(s) > L.arg_lim || fabs(t) > L.arg_lim)
    return LEAN_REJECT; // |dec| or |ra| > T for sure (arg_lim > tan T / cos T); also keeps the series inside its range
  return lean_classify(lean_series(s, L.cs, L.K, L.A), lean_series(t, L.ct, L.K, L.A), L, xs, ys);
}

// Host: fill the constants for a field (T = fov*(1+2/npix)*0.5, densitymaps.cpp:383).  Returns 0 when the field is too wide
// for the series (the kernels then use the libdevice path).
static inline int lean_setup(LeanDev *L, double fovrad, double T, double eta = LEAN_ETA)
{
  if (!(eta >= LEAN_ETA))
    eta = LEAN_ETA;
  L->enabled = 0;
  L->K = 0;
  if (!(T < 1.5) || !(fovrad > 0))
    return 0;
  const double arg_lim = tan(T) * (1.0 + 1e-5) / cos(T) * 1.01;
  if (!(arg_lim <= 0.385))
    return 0;
  // Maclaurin coefficients: asin a_k = a_{k-1} (2k-1)^2 / (2k (2k+1)), a_0 = 1; atan (-1)^k / (2k+1)
  long double as[LEAN_MAX_TERMS + 2];
  as[0] = 1.0L;
  for (int k = 1; k <= LEAN_MAX_TERMS + 1; k++)
    as[k] = as[k - 1] * (long double)((2 * k - 1) * (2 * k - 1)) / (long double)(2 * k * (2 * k + 1));
  // smallest K whose truncation stays below 2^-53 relative to the function value:
  //   asin: sum_{k>K} a_k z^k <= a_{K+1} z^{K+1} / (1 - z)   (a_k decreasing);   atan (alternating): <= z^{K+1} / (2K+3)
  const double z = arg_lim * arg_lim;
  int K = 0;
  for (int k = 2; k <= LEAN_MAX_TERMS && !K; k++)
  {
    const double tail_s = (double)as[k + 1] * pow(z, k + 1) / (1.0 - z), tail_t = pow(z, k + 1) / (2.0 * k + 3.0);
    if (tail_s <= 0x1p-53 && tail_t <= 0x1p-53)
      K = k;
  }
  if (K == 0)
    return 0;
  L->K = K;
  L->A = 1.0 / fovrad;
  L->arg_lim = arg_lim;
  const double tv = T / fovrad;
  L->eta = eta;
  L->w_in = tv - eta;
  L->w_out = tv + eta;
  for (int k = 0; k <= LEAN_MAX_TERMS; k++)
  {
    L->cs[k] = k <= K ? (double)((long double)L->A * as[k]) : 0.0;
    L->ct[k] = k <= K ? L->A * ((k & 1) ? -1.0 : 1.0) / (double)(2 * k + 1) : 0.0;
  }
  L->umin = 0x1p-40f;
  L->enabled = 1;
  return 1;
}
