// pass_params.h — host/device structures describing one pass (one kernel launch).
//
// A pass streams the resident particles of a snapshot once and deposits them into every lens plane that
// uses this snapshot.  Planes that share a randomisation (Random.*[isnap], rcase — data.h:126-131,
// slicer-v2.cpp:184-185) share an XformDev, so the box transform of gadget2io.cpp:204-270 is evaluated
// once per particle and only the slab test (densitymaps.cpp:374) is per plane.
#pragma once
#include <stddef.h>
#include <stdint.h>
#include "../../include/slicer_b200.h"
#include "lean_math.h"

// Device-side bounds checks of the checked build (`make checked` -> libslicer_b200_chk.so, loaded when SLICER_B200_LIB points
// to it): a violated condition traps, the next API call then fails with the CUDA error.  compute-sanitizer is not always
// available on shared GPU pools; these cover every computed index of the queues, record regions, sort and tiles.
#ifdef SLICER_CHECKS
#define SLICER_CHECK(cond) \
  do                       \
  {                        \
    if (!(cond))           \
      __trap();            \
  } while (0)
#else
#define SLICER_CHECK(cond) ((void)0)
#endif

// The float arrays cf, sgn, sinv, offs and wadd start at multiples of 8 bytes: the kernels read their x and y entries as one
// register pair (one 64-bit constant load) for the packed FP32 operations (deposit_pipelined.cuh: screen2, lean_axis2).
struct XformDev
{
  double box;    // Header.boxsize (data.h:70)
  double c[3];   // Random.x0,y0,z0 (data.h:128)
  float cf[3];   // == c[] when exact_f32
  float boxf;    // == box when exact_f32
  float sgn[3];  // sign applied to output axis k (already permuted): Random.sgn of the raw axis feeding it
  float rcase;   // slicer-v2.cpp:137,185
  int perm[3];   // raw axis (0,1,2) feeding output axis k (x,y,z): Random.face, gadget2io.cpp:223-252
  int exact_f32; // box and centre are float-representable: float ops reproduce the double chain bit for bit
  int first_plane, nplanes; // planes [first_plane, first_plane+nplanes) of PassParams::pl use this transform
  float zmin, zmax;         // union of those planes' slabs: cheap early-out
  // --- conservative float screen of the pipelined kernel (deposit_pipelined.cuh) ---
  // a_k = fma(raw[perm k], sinv[k], offs[k]) approximates (sgn*raw/box [+1 if sgn<0]) - centre_k to ~4e-7;
  // one wrap (a<0 -> a+1) gives the box coordinate.  Particles the screen cannot decide are sent to the
  // exact chain, never dropped.
  float sinv[3];
  float tmax;       // max over this transform's planes of pre_tx (>= pre_ty)
  float offs[3];
  float thr_m;      // additive slack of the lateral test: screen error + tmax * (z error)
  float zlo_m, zhi_m; // zmin/zmax widened by the screen's error margin
  float zamb;       // z-wrap ambiguity: |w - 0.5| > zamb  => undecidable
  float raw_hi;     // raw coordinates outside the open interval (0, raw_hi) may wrap in the exact chain => undecidable
  // --- fast box transform of the lean exact phase (deposit_pipelined.cuh: lean_axis), valid for raw in (LeanDev::umin, raw_hi) ---
  float wadd[3];    // 1 when sgn[k] < 0 (the wrap 1 + q of gadget2io.cpp:213-214 always fires), else 0 (no wrap can fire)
  float nboxf;      // -boxf: residual r = fma(q0, -box, u) of the division u / box
};
static_assert(offsetof(XformDev, cf) % 8 == 0 && offsetof(XformDev, sgn) % 8 == 0 && offsetof(XformDev, sinv) % 8 == 0 &&
                  offsetof(XformDev, offs) % 8 == 0 && offsetof(XformDev, wadd) % 8 == 0,
              "packed pairs of XformDev are 8-byte aligned");

struct PlaneDev
{
  // slab (densitymaps.cpp:346-347,374): double(z) >= minDist && double(z) < maxDist, restated on floats:
  // zlo = smallest float >= minDist, zhi = smallest float >= maxDist  =>  z >= zlo && z < zhi
  float zlo, zhi;
  // conservative float prefilter: an accepted replica satisfies |Y| <= Z*pre_ty and |X| <= Z*pre_tx (+ slack)
  float pre_tx, pre_ty;
  float npixf;
  int npix;
  int nrep;  // Lens.nrepperp (data.h:116)
  int pow2;  // npix is a power of two: dl is exact, divisions by dl become exact multiplications
  double T;          // fovradiants*(1.+2./npix)*0.5     densitymaps.cpp:383
  double fovrad;     // densitymaps.cpp:385-386
  double dl;         // 1./double(nn)                   utilities.cpp:50
  double half_dl;    // 0.5*dx                          utilities.cpp:9
  double onehalf_dl; // 0.5*3.0*dx                      utilities.cpp:11
  double scale;      // 2^frac_bits
  float scalef;      // the same as a float (exact)
  float dlf, half_dlf, onehalf_dlf; // float copies of dl, 0.5*dl, 1.5*dl: exact when npix is a power of two
  double guard_eta;  // rounding guard on dec/fov + 0.5 (slicer_config::guard_eta, default 2^-47) ...
  double guard_T;    // ... and on |ra|, |dec| against T: decisions inside the guard are settled with the host's libm
  double arg_lim;    // small-angle series: valid (and sufficient) for |X/d|, |Y/Z| <= arg_lim
  int nt;            // terms of the small-angle series, 0 => use libdevice asin/atan2 (wide fields)
  unsigned long long *acc;    // this plane's accumulators: [ntypes_alloc][npix*npix] int64 fixed point
  unsigned long long *counts; // [SLICER_NTYPES][2]: accepted pairs, in-grid pairs
  unsigned long long type_stride; // npix*npix when per-type maps are kept, else 0
  int slot;                       // the caller's plane index (device slots are grouped by randomisation)
};

struct PassParams
{
  int nxform;
  int nplanes;
  int fast;  // every plane: npix a power of two, no perpendicular replication, disjoint slabs per randomisation
  LeanDev lean; // lean projection + ambiguity guard (lean_math.h); enabled for fast passes whose planes share one narrow field
  XformDev xf[SLICER_MAX_XFORMS];
  PlaneDev pl[SLICER_MAX_PLANES];
};

// Particles whose accept decision or float map coordinates lie within the lean projection's error bound of a boundary: the
// kernels append them here (exact box coordinates, mass, plane) and the host recomputes them with libm exactly as the reference
// does (slicer_capi.cu: resolve_deferred) before any accumulator is read.
struct DeferEntry
{
  float x, y, z, m;      // box coordinates after gadget2io.cpp:204-270 (exact floats), particle mass after the MAX_M cut
  unsigned pass;         // which pass of the handle (host-side table of the plane parameters)
  unsigned short plane;  // device plane slot within that pass
  unsigned short type;   // particle type
};
struct DeferDev
{
  DeferEntry *buf;
  unsigned *count;    // entries appended so far (may exceed cap: the excess is lost and the pass is reported as failed)
  unsigned cap;
  unsigned pass;
};

struct SegmentDev
{
  const float *pos;  // AoS: n*3 floats; SoA: x[n_pad] y[n_pad] z[n_pad] with stride soa_stride
  const float *mass; // n floats or nullptr
  unsigned long long n;
  unsigned long long soa_stride;
  float const_mass; // float(massarr[type])            densitymaps.cpp:372
  float max_m;      // MAX_M cut for per-particle mass  densitymaps.cpp:368
  int type;
  int layout;
};
