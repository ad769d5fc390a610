// deposit_binned.cuh — the privatised (shared-memory tile) deposit for passes with many accepted particles.
//
// With tens of per cent of the snapshot inside the field of view, 9 global red.u64 per particle into maps that do
// not fit the L2 (4 planes x 32 MiB at 2048^2) run at ~9 G particles/s — 20x below the particle stream.  This path
// splits the pass into
//   K1  deposit_pipelined_kernel<..., EMIT>  stream + screen + exact chain up to the map coordinates (xs, ys);
//       every accepted particle becomes an 8-byte record, appended to its CTA's region (one shared-memory atomic per warp
//       and emit, no global atomics)
//   K2a bin_histogram_kernel                 records per (region, bin); K2b/K2c scans -> offset of every region in
//                                            every bin (no global atomics, deterministic bin layout)
//   K2d bin_scatter_kernel                   counting sort of the records by (plane, map tile) bin
//   K3  tile_deposit_kernel                  one CTA per bin: the TSC 3x3 stencil (same float arithmetic as
//                                            chain::deposit_pow2) is accumulated with 32-bit shared-memory atomics
//                                            into a (TILE+2)^2 tile of 64-bit fixed-point cells kept as two
//                                            32-bit limbs (carry from the returned old value), then flushed once
//                                            with red.global.add.u64.
// The int64 sums are exact and order independent, so the result is bit-identical to the direct path.
// K2/K3 sort and deposit at most MAX_BINS bins at a time: maps with more (plane, tile) pairs (8192^2) sort by groups of 2 or 4
// tiles adjacent in x (EmitDev::gshift; the tile kernel runs one CTA per tile and skips its neighbours' records), and beyond
// that in windows of the bin range over the SAME records (SortDev::bin_lo), i.e. K1 still runs once.
// With at most HIST_BINS bins K2a is folded into K1 (EmitDev::region_hist).
// Requirements (PassParams::fast): power-of-two npix equal for all planes, no perpendicular replication, <= 65536 bins.
#pragma once
#include <cuda_runtime.h>
#include "device_chain.cuh"

namespace binned
{

constexpr int TILE = 166;          // interior cells per tile side: one 1024-thread CTA per SM owns 226 KB
constexpr int TW = TILE + 2;       // + 1-cell halo for the 3x3 stencil
constexpr int TCELLS = TW * TW;    // 28,224 cells x 8 B = 225,792 B of shared memory
constexpr int MAX_BINS = 5120; // bins per sort window: 3 tables of MAX_BINS words + the 16K-record batch fill the scatter kernel's shared memory
constexpr int SCATTER_THREADS = 1024;
constexpr int DEPOSIT_THREADS = 1024;

struct EmitDev
{
  float2 *rec;              // [regions][region_cap]  (xs, ys)
  unsigned short *key;      // [regions][region_cap]  bin
  float *mass;              // [regions][region_cap]  or nullptr (constant-mass segment)
  unsigned *region_count;   // [regions]
  unsigned long long region_cap;
  int ntile;                // tiles per map side
  // Maps with more (plane, tile) pairs than one sort handles (8192^2: 4 x 2500) sort by GROUPS of 2^gshift tiles adjacent in x:
  // a bin then holds the records of the whole group, and the tile kernel runs one CTA per tile that skips its neighbours' records
  // (a second read of an 8-byte record is far cheaper than a second sort window over all records).
  int ntx;                  // tile groups per map row: ceil(ntile / 2^gshift)
  int gshift;
  // Passes with at most HIST_BINS bins: the record kernel counts its region's records per bin in shared memory and writes the
  // column of SortDev::region_hist itself (no bin_histogram_kernel: no second pass over the keys).  nullptr otherwise.
  unsigned *region_hist;    // [nbins][nregions]
  int nregions, nbins;
};
constexpr int HIST_BINS = 1024; // 4 KB per record-kernel CTA: 2048^2 maps in up to 6 planes (169 tiles each)

struct SortDev
{
  const float2 *rec_u;
  const unsigned short *key_u;
  const float *mass_u;
  const unsigned *region_count;
  unsigned long long region_cap;
  int nregions;
  int nbins;  // bins sorted by this round of K2/K3: global bins [bin_lo, bin_lo + nbins); records of other bins are skipped
  int bin_lo; // (maps whose planes x tiles exceed MAX_BINS are deposited window by window from ONE set of records)
  unsigned *region_hist; // [nbins][nregions]: records of region r in bin b, then (after the scan) their offset within the bin
  unsigned *bin_count;   // [nbins]
  unsigned *bin_start;   // [nbins + 1]
  float2 *rec_s;
  float *mass_s;
  unsigned long long capacity; // records rec_u/rec_s/key_u can hold (bounds checks of the checked build)
};

__device__ __forceinline__ int bin_of(int q, int gx, int gy, int nn, int ntile, int ntx, int gshift)
{
  const int cx = min(max(gx, 0), nn - 1) / TILE;
  const int cy = min(max(gy, 0), nn - 1) / TILE;
  return (q * ntile + cy) * ntx + (cx >> gshift);
}

// keys of a region, four at a time (region offsets are multiples of 1024 records, so the 8-byte loads are aligned)
template <typename F>
__device__ __forceinline__ void for_each_key(const unsigned short *key, unsigned n, int tid, int nthreads, F f)
{
  const uint2 *k4 = reinterpret_cast<const uint2 *>(key);
  const unsigned n4 = n >> 2;
  for (unsigned i = tid; i < n4; i += nthreads)
  {
    const uint2 v = k4[i];
    f(4 * i + 0, v.x & 0xffffu);
    f(4 * i + 1, v.x >> 16);
    f(4 * i + 2, v.y & 0xffffu);
    f(4 * i + 3, v.y >> 16);
  }
  for (unsigned i = 4 * n4 + tid; i < n; i += nthreads)
    f(i, (unsigned)key[i]);
}


// K2a: one CTA per region: shared-memory histogram of its keys -> region_hist[bin][region]
__global__ void __launch_bounds__(SCATTER_THREADS) bin_histogram_kernel(const __grid_constant__ SortDev D)
{
  __shared__ unsigned hist[MAX_BINS];
  for (int i = threadIdx.x; i < D.nbins; i += SCATTER_THREADS)
    hist[i] = 0;
  __syncthreads();
  const int r = blockIdx.x;
  const unsigned n = D.region_count[r];
  for_each_key(D.key_u + (unsigned long long)r * D.region_cap, n, threadIdx.x, SCATTER_THREADS,
               [&](unsigned, unsigned k) {
                 k -= (unsigned)D.bin_lo;
                 if (k < (unsigned)D.nbins)
                   atomicAdd(&hist[k], 1u);
               });
  __syncthreads();
  for (int i = threadIdx.x; i < D.nbins; i += SCATTER_THREADS)
    D.region_hist[(size_t)i * D.nregions + r] = hist[i];
}

__device__ __forceinline__ unsigned block_exclusive_scan_1024(unsigned x, unsigned *wsum, unsigned *total)
{
  const int t = threadIdx.x, lane = t & 31, w = t >> 5;
  unsigned incl = x;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1)
  {
    const unsigned y = __shfl_up_sync(0xffffffffu, incl, d);
    if (lane >= d)
      incl += y;
  }
  if (lane == 31)
    wsum[w] = incl;
  __syncthreads();
  if (w == 0)
  {
    const unsigned s = wsum[lane];
    unsigned si = s;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1)
    {
      const unsigned y = __shfl_up_sync(0xffffffffu, si, d);
      if (lane >= d)
        si += y;
    }
    wsum[lane] = si - s;
    if (lane == 31)
      *total = si;
  }
  __syncthreads();
  const unsigned excl = wsum[w] + incl - x;
  __syncthreads();
  return excl;
}

// K2b: one CTA per bin: exclusive scan of that bin's counts over the regions (in place) + the bin total
__global__ void __launch_bounds__(1024) bin_region_scan_kernel(const __grid_constant__ SortDev D)
{
  __shared__ unsigned wsum[32];
  __shared__ unsigned total;
  unsigned *h = D.region_hist + (size_t)blockIdx.x * D.nregions;
  unsigned carry = 0;
  for (int base = 0; base < D.nregions; base += 1024)
  {
    const int i = base + threadIdx.x;
    const unsigned x = i < D.nregions ? h[i] : 0u;
    const unsigned e = block_exclusive_scan_1024(x, wsum, &total);
    if (i < D.nregions)
      h[i] = carry + e;
    carry += total;
    __syncthreads();
  }
  if (threadIdx.x == 0)
    D.bin_count[blockIdx.x] = carry;
}

// K2c: exclusive scan of <= MAX_BINS bin totals (one CTA; thread t owns bins [PER t, PER t + PER))
__global__ void __launch_bounds__(1024) bin_scan_kernel(const __grid_constant__ SortDev D)
{
  __shared__ unsigned wsum[32];
  __shared__ unsigned total;
  constexpr int PER = MAX_BINS / 1024;
  const int t = threadIdx.x;
  unsigned v[PER], x = 0;
#pragma unroll
  for (int j = 0; j < PER; j++)
  {
    v[j] = (PER * t + j < D.nbins) ? D.bin_count[PER * t + j] : 0u;
    x += v[j];
  }
  unsigned excl = block_exclusive_scan_1024(x, wsum, &total);
#pragma unroll
  for (int j = 0; j < PER; j++)
  {
    if (PER * t + j < D.nbins)
      D.bin_start[PER * t + j] = excl;
    excl += v[j];
  }
  if (t == 0)
    D.bin_start[D.nbins] = total;
}

// bulk prefetch of [p, p + bytes) into L2 (bytes a multiple of 16, p 16-byte aligned): one instruction, no registers, no wait
__device__ __forceinline__ void l2_prefetch(const void *p, unsigned bytes)
{
  asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(p), "r"(bytes) : "memory");
}

// K2d: one CTA per region: record -> bin_start[bin] + (offset of this region in the bin) + (rank inside the region).
// Measured on B200: a warp store whose 32 lanes hit 32 different sectors costs ~3-6 cycles per LANE per SM
// (~50-100 G sector requests/s chip-wide, whatever the instruction: st, st.cs, red), 5x more than the same bytes
// written as full sectors.  So every batch of SCATTER_BATCH records is first counting-sorted in shared memory and
// then written out in sorted order: consecutive lanes carry consecutive records of one bin, i.e. consecutive
// addresses.  No global atomics; the bin layout is deterministic up to the order inside a (batch, bin) run.
constexpr int SCATTER_BATCH = 16384;
constexpr int SCATTER_PER = SCATTER_BATCH / SCATTER_THREADS; // records per thread per batch
// NB = table size: MAX_BINS, or SMALL_BINS for the usual few-plane 2048^2 passes (a shorter scan per batch).
// (Measured and not kept: two 768-thread CTAs per SM with 6 K-record batches and 1536-bin tables, to overlap the phases between
// the barriers: 5.25 instead of 4.2 ms on the densest C3 group — the shorter runs cost more than the overlap gains.)
constexpr int SMALL_BINS = 4096;
template <int NB, int THREADS, int PER>
struct ScatterSmem
{
  float2 rec[THREADS * PER];
  unsigned short bin[THREADS * PER];
  unsigned cnt[NB];    // records of the batch per bin, then running rank
  unsigned lstart[NB]; // first sorted slot of the bin in this batch
  unsigned gcur[NB];   // next free global slot of the bin for this region
  unsigned wsum[THREADS / 32];
  unsigned ntot; // records of the batch inside the bin window
};

// WIN: the sort covers a window of the bins only (maps with more than MAX_BINS plane-tiles), other records are skipped.
// MASS: the records carry a per-particle mass (hydro segments): a second sweep applies the same permutation to the masses.
//
// Per batch of THREADS * PER records:  1. rank inside (batch, bin) by shared-memory atomics  2. exclusive scan of the batch
// histogram  3. the records go to their sorted slot in shared memory  4. write-out in sorted order.  The global loads of a
// batch are paired (one 16-byte load of two records, one 4-byte load of their two keys: half the load instructions in flight)
// and the next batch is brought into L2 by a bulk prefetch (one instruction per array) while this one is sorted, so that its
// loads do not wait for DRAM: 1.05 -> 0.83 ms per slice of the densest C3 group.  (Measured and not kept: loading the next
// batch's keys into registers before the write-out — the register allocator spills them at 64 registers, which serialises
// the loads: 1.18 ms; per-bin cursors in registers with one `slot -> global` offset table for the write-out: 1.0 ms.)
template <int NB, bool WIN, bool MASS, int THREADS, int PER, int CTAS>
__global__ void __launch_bounds__(THREADS, CTAS) bin_scatter_kernel(const __grid_constant__ SortDev D)
{
  extern __shared__ __align__(16) unsigned char scatter_raw[];
  using Sm = ScatterSmem<NB, THREADS, PER>;
  Sm &sm = *reinterpret_cast<Sm *>(scatter_raw);
  float *smass = reinterpret_cast<float *>(sm.rec); // per-particle masses reuse the record staging in a second sweep
  constexpr int BATCH = THREADS * PER;
  constexpr int PERB = NB / THREADS; // bins per thread in the scan
  static_assert(NB % THREADS == 0 && THREADS % 32 == 0 && THREADS / 32 <= 32 && PER % 2 == 0, "scan layout");
  const int r = blockIdx.x;
  const int t = threadIdx.x, lane = t & 31, w = t >> 5;
  const unsigned n = D.region_count[r];
  if (n == 0)
    return;
  for (int i = t; i < NB; i += THREADS)
    sm.cnt[i] = 0; // (entries >= nbins are never incremented: the batch scan runs over all NB entries)
  const unsigned long long off = (unsigned long long)r * D.region_cap;
  const unsigned short *key = D.key_u + off;
  const float2 *rec = D.rec_u + off;
  const float *mass = MASS ? D.mass_u + off : nullptr;
  // record j of the thread is record rec_index(j) of the batch
  auto rec_index = [&](int j) { return 2u * (unsigned)((j >> 1) * THREADS + t) + (unsigned)(j & 1); };
  for (int i = t; i < D.nbins; i += THREADS)
    sm.gcur[i] = D.bin_start[i] + D.region_hist[(size_t)i * D.nregions + r];
  for (unsigned base = 0; base < n; base += BATCH)
  {
    const unsigned nb = min(n - base, (unsigned)BATCH);
    for (int i = t; i < D.nbins; i += THREADS)
      sm.cnt[i] = 0;
    __syncthreads();
    // 1. coalesced loads, rank inside (batch, bin)
    unsigned k[PER]; // bin | rank << 16 (rank < BATCH <= 2^14)
    float2 e[PER];
    {
      // (region offsets and `base` are multiples of 1024 records: the paired loads are aligned)
      const uint32_t *key2 = reinterpret_cast<const uint32_t *>(key + base);
      const float4 *rec2 = reinterpret_cast<const float4 *>(rec + base);
#pragma unroll
      for (int jj = 0; jj < PER / 2; jj++)
      {
        const unsigned pi = (unsigned)(jj * THREADS + t), i = 2u * pi;
        k[2 * jj] = k[2 * jj + 1] = 0xffffffffu;
        if (i < nb)
        { // (the second record of the last pair of an odd batch is stale memory inside the region's capacity: loaded, ignored)
          const uint32_t kk2 = key2[pi];
          const float4 r4 = rec2[pi]; // unconditionally: a load that waits for the key compare would serialise the two latencies
          e[2 * jj] = make_float2(r4.x, r4.y);
          e[2 * jj + 1] = make_float2(r4.z, r4.w);
          const unsigned k0 = (kk2 & 0xffffu) - (WIN ? (unsigned)D.bin_lo : 0u), k1 = (kk2 >> 16) - (WIN ? (unsigned)D.bin_lo : 0u);
          if (!WIN || k0 < (unsigned)D.nbins)
            k[2 * jj] = k0;
          if ((!WIN || k1 < (unsigned)D.nbins) && i + 1 < nb)
            k[2 * jj + 1] = k1;
        }
      }
    }
    // While this batch is sorted in shared memory the memory system is idle: have the next batch brought into L2 (one bulk
    // prefetch per array, issued by one thread), so that its loads do not wait for DRAM.
    if (t == 0 && base + BATCH < n)
    {
      const unsigned nn = min(n - (base + BATCH), (unsigned)BATCH);
      l2_prefetch(rec + base + BATCH, (nn * 8u + 15u) & ~15u);
      l2_prefetch(key + base + BATCH, (nn * 2u + 15u) & ~15u);
      if (MASS)
        l2_prefetch(mass + base + BATCH, (nn * 4u + 15u) & ~15u);
    }
#pragma unroll
    for (int j = 0; j < PER; j++)
      if (k[j] != 0xffffffffu)
        k[j] |= atomicAdd(&sm.cnt[k[j]], 1u) << 16;
    __syncthreads();
    // 2. exclusive scan of the batch histogram: thread t owns bins [PERB t, PERB t + PERB)
    unsigned c[PERB], x = 0;
#pragma unroll
    for (int j = 0; j < PERB; j++)
    {
      c[j] = sm.cnt[PERB * t + j];
      x += c[j];
    }
    unsigned incl = x;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1)
    {
      const unsigned y = __shfl_up_sync(0xffffffffu, incl, d);
      if (lane >= d)
        incl += y;
    }
    if (lane == 31)
      sm.wsum[w] = incl;
    __syncthreads();
    if (w == 0)
    {
      const unsigned sv = lane < THREADS / 32 ? sm.wsum[lane] : 0u;
      unsigned si = sv;
#pragma unroll
      for (int d = 1; d < 32; d <<= 1)
      {
        const unsigned y = __shfl_up_sync(0xffffffffu, si, d);
        if (lane >= d)
          si += y;
      }
      if (lane < THREADS / 32)
        sm.wsum[lane] = si - sv;
    }
    __syncthreads();
    unsigned ex = sm.wsum[w] + incl - x;
#pragma unroll
    for (int j = 0; j < PERB; j++)
    {
      sm.lstart[PERB * t + j] = ex;
      ex += c[j];
    }
    if (WIN && t == THREADS - 1)
      sm.ntot = ex;
    __syncthreads();
    const unsigned ntot = WIN ? sm.ntot : nb;
    // 3. sorted order in shared memory
#pragma unroll
    for (int j = 0; j < PER; j++)
      if (k[j] != 0xffffffffu)
      {
        const unsigned lp = sm.lstart[k[j] & 0xffffu] + (k[j] >> 16);
        SLICER_CHECK((k[j] & 0xffffu) < (unsigned)D.nbins && lp < (unsigned)BATCH);
        sm.rec[lp] = e[j];
        sm.bin[lp] = (unsigned short)(k[j] & 0xffffu);
      }
    __syncthreads();
    // 4. write-out: slot i of the sorted batch -> gcur[bin] + (i - lstart[bin]); runs are contiguous in memory
    for (unsigned i = t; i < ntot; i += THREADS)
    {
      const unsigned b = sm.bin[i];
      const unsigned dst = sm.gcur[b] + (i - sm.lstart[b]);
      SLICER_CHECK(b < (unsigned)D.nbins && dst >= D.bin_start[b] && dst < D.bin_start[b + 1] && dst < D.capacity);
      D.rec_s[dst] = sm.rec[i];
    }
    __syncthreads();
    if (MASS)
    { // same permutation for the masses
#pragma unroll
      for (int j = 0; j < PER; j++)
        if (k[j] != 0xffffffffu)
          smass[sm.lstart[k[j] & 0xffffu] + (k[j] >> 16)] = mass[base + rec_index(j)];
      __syncthreads();
      for (unsigned i = t; i < ntot; i += THREADS)
        D.mass_s[sm.gcur[sm.bin[i]] + (i - sm.lstart[sm.bin[i]])] = smass[i];
      __syncthreads();
    }
#pragma unroll
    for (int j = 0; j < PERB; j++)
      sm.gcur[PERB * t + j] += c[j];
  }
}

using ScatterSmall = ScatterSmem<SMALL_BINS, SCATTER_THREADS, SCATTER_PER>;
using ScatterWin = ScatterSmem<MAX_BINS, SCATTER_THREADS, SCATTER_PER>;

static inline cudaError_t prepare_bin_scatter()
{
  cudaError_t e = cudaSuccess;
  auto prep = [&](auto kern, size_t bytes) {
    if (e == cudaSuccess)
      e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
  };
  prep(bin_scatter_kernel<SMALL_BINS, false, false, SCATTER_THREADS, SCATTER_PER, 1>, sizeof(ScatterSmall));
  prep(bin_scatter_kernel<SMALL_BINS, false, true, SCATTER_THREADS, SCATTER_PER, 1>, sizeof(ScatterSmall));
  prep(bin_scatter_kernel<MAX_BINS, true, false, SCATTER_THREADS, SCATTER_PER, 1>, sizeof(ScatterWin));
  prep(bin_scatter_kernel<MAX_BINS, true, true, SCATTER_THREADS, SCATTER_PER, 1>, sizeof(ScatterWin));
  return e;
}

static inline void launch_bin_scatter(const SortDev &Q, bool windowed, cudaStream_t stream)
{
  const bool small = !windowed && Q.nbins <= SMALL_BINS;
  if (small && !Q.mass_u)
    bin_scatter_kernel<SMALL_BINS, false, false, SCATTER_THREADS, SCATTER_PER, 1><<<Q.nregions, SCATTER_THREADS, sizeof(ScatterSmall), stream>>>(Q);
  else if (small)
    bin_scatter_kernel<SMALL_BINS, false, true, SCATTER_THREADS, SCATTER_PER, 1><<<Q.nregions, SCATTER_THREADS, sizeof(ScatterSmall), stream>>>(Q);
  else if (!Q.mass_u)
    bin_scatter_kernel<MAX_BINS, true, false, SCATTER_THREADS, SCATTER_PER, 1><<<Q.nregions, SCATTER_THREADS, sizeof(ScatterWin), stream>>>(Q);
  else
    bin_scatter_kernel<MAX_BINS, true, true, SCATTER_THREADS, SCATTER_PER, 1><<<Q.nregions, SCATTER_THREADS, sizeof(ScatterWin), stream>>>(Q);
}

// The TSC 3x3 stencil of one record (utilities.cpp:78-94) into the tile: 64-bit cells kept as two 32-bit limbs.
// (x0, y0) = map cell of local cell (0,0); `sm` = sqrtf(mass).
__device__ __forceinline__ void tile_tsc(unsigned *lo, unsigned *hi, int x0, int y0, int nn, const PlaneDev &L, float xs, float ys, int gx, int gy,
                                         float sm)
{
    const int lx = gx - 1 - x0, ly = gy - 1 - y0; // local index of stencil cell (0,0)
    unsigned *plo = lo + ly * TW + lx, *phi = hi + ly * TW + lx;
    // one cell: 64-bit add as two 32-bit shared-memory atomics, the carry taken from the returned old value of the low limb
    auto add_cell = [&](int off, float contribution_scaled) {
      const unsigned long long v = (unsigned long long)__float2ll_rn(contribution_scaled);
      const unsigned vl = (unsigned)v, vh = (unsigned)(v >> 32);
      const unsigned old = atomicAdd(plo + off, vl);
      atomicAdd(phi + off, vh + (unsigned)(((unsigned long long)old + vl) >> 32));
    };
    if (gx >= 1 && gx <= nn - 2 && gy >= 1 && gy <= nn - 2)
    {
      // Interior stencil (all but the map's border).  npix is a power of two (PassParams::fast), so scaling by npix or dl is
      // exact and the reference's |xs - cx_k| / dl (utilities.cpp:4-16,78-89; chain::deposit_pow2) can be evaluated on the
      // scaled coordinate: with X = xs * npix >= 1 and f = X - floor(X) (exact), X - (gx + k - 1/2) and f - (k - 1/2) are the
      // same real number, hence the same float after the one rounding of the subtraction.  Likewise the fixed-point scale
      // 2^frac_bits is folded into the x weights: fl(sm 2^b vx) fl(sm vy) rounds exactly like 2^b fl(fl(sm vx) fl(sm vy)),
      // and where the unscaled product would be denormal both forms convert to 0.
      SLICER_CHECK(lx >= 0 && lx + 2 < TW && ly >= 0 && ly + 2 < TW); // the record belongs to this tile (+ halo)
      const float fx = __fsub_rn(__fmul_rn(xs, L.npixf), (float)gx), fy = __fsub_rn(__fmul_rn(ys, L.npixf), (float)gy);
      const float ax0 = fabsf(__fadd_rn(fx, 0.5f)), ax1 = fabsf(__fsub_rn(fx, 0.5f)), ax2 = fabsf(__fsub_rn(fx, 1.5f));
      const float ay0 = fabsf(__fadd_rn(fy, 0.5f)), ay1 = fabsf(__fsub_rn(fy, 0.5f)), ay2 = fabsf(__fsub_rn(fy, 1.5f));
      const float tx0 = __fsub_rn(1.5f, ax0), tx2 = __fsub_rn(1.5f, ax2), ty0 = __fsub_rn(1.5f, ay0), ty2 = __fsub_rn(1.5f, ay2);
      const float smx = __fmul_rn(sm, L.scalef);
      float wx[3], wy[3];
      wx[0] = __fmul_rn(smx, __fmul_rn(0.5f, __fmul_rn(tx0, tx0)));
      wx[1] = __fmul_rn(smx, __fsub_rn(0.75f, __fmul_rn(ax1, ax1)));
      wx[2] = __fmul_rn(smx, __fmul_rn(0.5f, __fmul_rn(tx2, tx2)));
      wy[0] = __fmul_rn(sm, __fmul_rn(0.5f, __fmul_rn(ty0, ty0)));
      wy[1] = __fmul_rn(sm, __fsub_rn(0.75f, __fmul_rn(ay1, ay1)));
      wy[2] = __fmul_rn(sm, __fmul_rn(0.5f, __fmul_rn(ty2, ty2)));
      // nine unconditional limb pairs, no branches — adding a zero limb is harmless and cheaper than testing for it
#pragma unroll
      for (int jy = 0; jy < 3; jy++)
#pragma unroll
        for (int jx = 0; jx < 3; jx++)
          add_cell(jy * TW + jx, __fmul_rn(wx[jx], wy[jy]));
    }
    else
    {
      // border stencil: the reference's arithmetic operation for operation (xs * npix may be negative here)
      float wx[3], wy[3];
#pragma unroll
      for (int k = 0; k < 3; k++)
      {
        const float cx = __fmul_rn(__fadd_rn((float)(gx + k - 1), 0.5f), L.dlf);
        const float cy = __fmul_rn(__fadd_rn((float)(gy + k - 1), 0.5f), L.dlf);
        const float ax = __fmul_rn(fabsf(__fsub_rn(xs, cx)), L.npixf);
        const float ay = __fmul_rn(fabsf(__fsub_rn(ys, cy)), L.npixf);
        float vx, vy;
        if (k == 1)
        {
          vx = __fsub_rn(0.75f, __fmul_rn(ax, ax));
          vy = __fsub_rn(0.75f, __fmul_rn(ay, ay));
        }
        else
        {
          const float t1 = __fsub_rn(1.5f, ax), t2 = __fsub_rn(1.5f, ay);
          vx = __fmul_rn(0.5f, __fmul_rn(t1, t1));
          vy = __fmul_rn(0.5f, __fmul_rn(t2, t2));
        }
        wx[k] = __fmul_rn(sm, vx);
        wy[k] = __fmul_rn(sm, vy);
      }
      for (int jy = 0; jy < 3; jy++)
        for (int jx = 0; jx < 3; jx++)
        {
          const int cx = gx + jx - 1, cy = gy + jy - 1;
          if (cx < 0 || cx >= nn || cy < 0 || cy >= nn)
            continue; // utilities.cpp:91 drops cells outside the map
          SLICER_CHECK(lx + jx >= 0 && lx + jx < TW && ly + jy >= 0 && ly + jy < TW);
          add_cell(jy * TW + jx, __fmul_rn(__fmul_rn(wx[jx], wy[jy]), L.scalef));
        }
    }
}

// K3: one CTA per (plane, tile) bin
template <int MAS>
__global__ void __launch_bounds__(DEPOSIT_THREADS, 1)
    tile_deposit_kernel(const __grid_constant__ PassParams P, const __grid_constant__ SortDev D, int ntile, int ntx, int gshift, int type,
                        float const_mass)
{
  extern __shared__ __align__(16) unsigned tile_smem[];
  __shared__ unsigned s_ingrid, s_n;
  unsigned *lo = tile_smem;
  unsigned *hi = tile_smem + TCELLS;
  const int bl = blockIdx.x >> gshift, sub = blockIdx.x & ((1 << gshift) - 1); // bin of this launch, tile within the bin's group
  const unsigned r0 = D.bin_start[bl], r1 = D.bin_start[bl + 1];
  if (r0 == r1)
    return;
  if (threadIdx.x == 0)
  {
    s_ingrid = 0;
    s_n = 0;
  }
  const int b = bl + D.bin_lo;
  const int q = b / (ntile * ntx);
  const int tb = b - q * ntile * ntx;
  const int ty = tb / ntx, tx = ((tb - ty * ntx) << gshift) + sub;
  if (tx >= ntile)
    return; // the last group of a row may be incomplete
  const PlaneDev &L = P.pl[q];
  const int nn = L.npix;
  const int x0 = tx * TILE - 1, y0 = ty * TILE - 1; // map cell of local (0,0)
  // The records of this bin are the accepted pairs of (plane, tile): this kernel keeps mapParticles' counters for the binned
  // path (densitymaps.cpp:402-403), the record kernel does not count.  Only a border tile can hold records whose nearest
  // grid point is outside the map.
  const bool border = tx == 0 || ty == 0 || tx == ntile - 1 || ty == ntile - 1;
  unsigned my_ingrid = 0, my_n = 0; // (my_n: records of THIS tile when the bin holds a group of tiles)
  for (int i = threadIdx.x; i < 2 * TCELLS; i += DEPOSIT_THREADS)
    tile_smem[i] = 0;
  __syncthreads();
  // `sm` = sqrtf(mass) (utilities.cpp:86-89 multiplies each 1-D weight by it); for a constant-mass segment it is hoisted out
  // of the record loop (the IEEE square root is a guarded sequence of ~15 instructions)
  const float sm_const = __fsqrt_rn(const_mass);
  auto one = [&](float xs, float ys, float m, float sm) {
    const int gx = __float2int_rd(__fmul_rn(xs, L.npixf));
    const int gy = __float2int_rd(__fmul_rn(ys, L.npixf));
    if (gshift)
    { // the bin holds the records of 2^gshift tiles: this CTA deposits its own
      if (min(max(gx, 0), nn - 1) / TILE != tx)
        return;
      my_n++;
    }
    if (border)
      my_ingrid += (gx >= 0 && gx < nn && gy >= 0 && gy < nn) ? 1u : 0u;
    if constexpr (MAS == SLICER_MAS_NGP)
    { // utilities.cpp:72-76: the whole mass goes to the nearest grid point, if it is inside the map
      if (gx >= 0 && gx < nn && gy >= 0 && gy < nn)
      {
        const unsigned long long v = (unsigned long long)chain::to_fixed(m, L);
        const int c = (gy - y0) * TW + gx - x0;
        SLICER_CHECK(gx - x0 >= 1 && gx - x0 <= TILE && gy - y0 >= 1 && gy - y0 <= TILE);
        const unsigned vl = (unsigned)v, vh = (unsigned)(v >> 32);
        const unsigned old = atomicAdd(lo + c, vl);
        atomicAdd(hi + c, vh + ((old + vl < old) ? 1u : 0u));
      }
    }
    else
      tile_tsc(lo, hi, x0, y0, nn, L, xs, ys, gx, gy, sm);
  };
  {
    unsigned i = r0 + threadIdx.x;
    for (; i + 3 * DEPOSIT_THREADS < r1; i += 4 * DEPOSIT_THREADS)
    { // four records in flight per thread
      float2 e[4];
      float m[4];
#pragma unroll
      for (int j = 0; j < 4; j++)
      {
        e[j] = D.rec_s[i + j * DEPOSIT_THREADS];
        m[j] = D.mass_s ? D.mass_s[i + j * DEPOSIT_THREADS] : const_mass;
      }
#pragma unroll
      for (int j = 0; j < 4; j++)
        one(e[j].x, e[j].y, m[j], D.mass_s ? __fsqrt_rn(m[j]) : sm_const);
    }
    for (; i < r1; i += DEPOSIT_THREADS)
    {
      const float2 e0 = D.rec_s[i];
      const float m0 = D.mass_s ? D.mass_s[i] : const_mass;
      one(e0.x, e0.y, m0, D.mass_s ? __fsqrt_rn(m0) : sm_const);
    }
  }
  if (border)
  {
    const unsigned wsum = __reduce_add_sync(0xffffffffu, my_ingrid);
    if ((threadIdx.x & 31) == 0 && wsum)
      atomicAdd(&s_ingrid, wsum);
  }
  if (gshift)
  {
    const unsigned wsum = __reduce_add_sync(0xffffffffu, my_n);
    if ((threadIdx.x & 31) == 0 && wsum)
      atomicAdd(&s_n, wsum);
  }
  __syncthreads();
  if (threadIdx.x == 0)
  {
    const unsigned mine = gshift ? s_n : r1 - r0;
    atomicAdd(L.counts + 2 * type, (unsigned long long)mine);
    atomicAdd(L.counts + 2 * type + 1, (unsigned long long)(border ? s_ingrid : mine));
  }
  unsigned long long *map = L.acc + L.type_stride * (unsigned long long)type;
  for (int i = threadIdx.x; i < TCELLS; i += DEPOSIT_THREADS)
  {
    const unsigned long long v = ((unsigned long long)hi[i] << 32) | lo[i];
    if (v)
    {
      const int cy = y0 + i / TW, cx = x0 + i % TW;
      SLICER_CHECK(cx >= 0 && cx < nn && cy >= 0 && cy < nn); // halo cells outside the map never receive mass
      chain::red_add(map + (size_t)cx + (size_t)nn * cy, (long long)v);
    }
  }
}


} // namespace binned
