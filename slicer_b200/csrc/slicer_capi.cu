// slicer_capi.cu — implementation of include/slicer_b200.h: handle, device memory, streams, pass set-up,
// kernel launches, NCCL reduce.  Host-side arithmetic that feeds the kernel (minDist/maxDist, T, dl) is written
// with the reference's own expressions so the doubles are bit-identical:
//   densitymaps.cpp:346-347 (minDist,maxDist)  :383 (T)  utilities.cpp:50 (dl)  utilities.cpp:9,11 (0.5*dx, 0.5*3.0*dx)
#include <chrono>
#include <cuda_runtime.h>
#include <dlfcn.h>
#include <nccl.h>
#include <math.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <string>
#include <vector>

#include "../../include/slicer_b200.h"
#include "pass_params.h"
#include "aux_kernels.cuh"
#include "deposit_simple.cuh"
#include "deposit_pipelined.cuh"
#include "deposit_degrade.cuh"

#define POS_U 1.0 /* gadget2io.h:14 */

// ------------------------------------------------------------------------------------------------------------
// errors
// ------------------------------------------------------------------------------------------------------------
static thread_local char g_err[512] = "";

static int fail(const char *fmt, ...)
{
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return 1;
}

#define CU(expr)                                                                                   \
  do                                                                                               \
  {                                                                                                \
    cudaError_t _e = (expr);                                                                       \
    if (_e != cudaSuccess)                                                                         \
      return fail("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__);     \
  } while (0)

extern "C" const char *slicer_last_error(void) { return g_err; }

// ------------------------------------------------------------------------------------------------------------
// NCCL, loaded lazily so that single-GPU use has no dependency on it
// ------------------------------------------------------------------------------------------------------------
struct NcclApi
{
  void *lib = nullptr;
  ncclResult_t (*GetUniqueId)(ncclUniqueId *) = nullptr;
  ncclResult_t (*CommInitRank)(ncclComm_t *, int, ncclUniqueId, int) = nullptr;
  ncclResult_t (*CommInitAll)(ncclComm_t *, int, const int *) = nullptr;
  ncclResult_t (*Reduce)(const void *, void *, size_t, ncclDataType_t, ncclRedOp_t, int, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*GroupStart)() = nullptr;
  ncclResult_t (*GroupEnd)() = nullptr;
  ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
  const char *(*GetErrorString)(ncclResult_t) = nullptr;
};
static NcclApi g_nccl;

static int load_nccl()
{
  if (g_nccl.lib)
    return 0;
  const char *names[] = {"libnccl.so.2", "libnccl.so", nullptr};
  for (int i = 0; names[i] && !g_nccl.lib; i++)
    g_nccl.lib = dlopen(names[i], RTLD_NOW | RTLD_GLOBAL);
  if (!g_nccl.lib)
    return fail("cannot load NCCL (libnccl.so.2): %s", dlerror());
#define SYM(field, name)                                           \
  *(void **)(&g_nccl.field) = dlsym(g_nccl.lib, name);             \
  if (!g_nccl.field)                                               \
  return fail("NCCL symbol %s missing", name)
  SYM(GetUniqueId, "ncclGetUniqueId");
  SYM(CommInitRank, "ncclCommInitRank");
  SYM(CommInitAll, "ncclCommInitAll");
  SYM(Reduce, "ncclReduce");
  SYM(GroupStart, "ncclGroupStart");
  SYM(GroupEnd, "ncclGroupEnd");
  SYM(CommDestroy, "ncclCommDestroy");
  SYM(GetErrorString, "ncclGetErrorString");
#undef SYM
  return 0;
}

#define NC(expr)                                                                                        \
  do                                                                                                    \
  {                                                                                                     \
    ncclResult_t _r = (expr);                                                                           \
    if (_r != ncclSuccess)                                                                              \
      return fail("%s failed: %s (%s:%d)", #expr, g_nccl.GetErrorString(_r), __FILE__, __LINE__);       \
  } while (0)

// ------------------------------------------------------------------------------------------------------------
// handle
// ------------------------------------------------------------------------------------------------------------
static const size_t PASS_RING = 256; // pending (start, stop) event pairs kept per handle

struct Segment
{
  int type;
  size_t n;
  const float *dpos;
  const float *dmass;
  int layout;
  size_t soa_stride;
};

struct slicer_handle
{
  slicer_config cfg;
  int frac_bits;
  int ntypes_alloc;
  size_t npix2max;
  int sm_count;
  cudaStream_t compute = nullptr, copy = nullptr, comm_stream = nullptr;
  cudaStream_t aux = nullptr;                      // zeroing of large accumulators, concurrent with the record kernel of a binned pass
  cudaEvent_t ev_zero_start = nullptr, ev_zero_done = nullptr;
  bool zero_pending = false;                       // the compute stream has not yet waited for ev_zero_done
  cudaEvent_t ev_pass_done = nullptr;              // compute -> comm_stream: the passes a reduce sums
  cudaEvent_t ev_slot[SLICER_MAX_SLOTS];           // comm_stream -> compute: the last reduce of accumulator slot q
  bool slot_reducing[SLICER_MAX_SLOTS];            // ev_slot[q] is pending
  cudaEvent_t ev_copy = nullptr;
  cudaEvent_t ev_buf_done[2] = {nullptr, nullptr}; // last pass that read staging pool b
  cudaEvent_t ev_t0 = nullptr, ev_t1 = nullptr;    // slicer_timer_*
  std::vector<cudaEvent_t> pass_ev;                // ring of (start, stop) pairs, resolved lazily
  size_t pass_head = 0, pass_tail = 0;             // pairs [tail, head) are pending
  int nbuf = 1, cur_buf = 0;
  int debug = 0;
  bool no_series = false; // env SLICER_B200_NO_SERIES: always use libdevice asin/atan2 (A/B checks)
  bool no_lean = false;   // env SLICER_B200_NO_LEAN: general exact chain instead of the lean projection + guard (A/B checks)
  float *d_pos_pool = nullptr;  // nbuf * (particle_capacity * 3 + 64) floats
  float *d_mass_pool = nullptr; // nbuf * (mass_capacity + 64) floats
  float *d_pos = nullptr;  // current pool
  float *d_mass = nullptr;
  size_t pos_used = 0;     // in particles
  size_t mass_used = 0;
  std::vector<Segment> segs;
  unsigned long long *d_acc = nullptr;    // [max_planes][ntypes_alloc][npix2max]
  unsigned long long *d_counts = nullptr; // [max_planes][6][2]
  float *d_out = nullptr;                 // npix2max
  long long *d_sum = nullptr;             // npix2max
  double boxsize = 0;
  double massarr[SLICER_NTYPES] = {0, 0, 0, 0, 0, 0};
  int hydro = 0;
  int plane_npix[SLICER_MAX_SLOTS];
  bool copy_pending = false;
  slicer_stats stats;
  size_t device_bytes = 0;
  ncclComm_t comm = nullptr;
  int nranks = 1, rank = 0;
  PipelinedScratch pipe;
  // lean exact phase: particles it could not decide (lean_math.h), settled with the host's libm by resolve_deferred()
  struct SavedPass
  {
    PassParams P;
    unsigned long long epoch[SLICER_MAX_PLANES]; // zeroing count of the accumulator slot of device plane k when the pass was submitted
  };
  // Two banks: the passes of one set of planes (a non-accumulating pass and the accumulating ones behind it) append to one
  // bank, the next set to the other, so that a set can be settled — waiting for ITS last pass only, with the few deposits
  // on a stream of their own — while the passes of the next set run (slicer_settle_slots, slicer_reduce_slots).
  // Which bank a new set takes: run_pass.
  struct DeferBank
  {
    DeferEntry *buf = nullptr;
    unsigned *count = nullptr;      // device: entries appended since the bank was last settled
    DeferEntry *host = nullptr;     // pinned mirror
    unsigned *host_count = nullptr; // pinned: the counter as of the end of the bank's last pass (copied behind every pass)
    std::vector<SavedPass> passes;  // passes since the last settle; DeferEntry::pass indexes it
    cudaEvent_t ev_done = nullptr;  // behind the bank's last pass and the copies of its counter / list head
    uint64_t slot_mask = 0;         // accumulator slots the bank's passes deposit into (bit q: slot q)
  };
  struct
  {
    DeferBank bank[2];
    int cur = 0;
    unsigned cap = 0;
    bool failed = false;
  } defer;
  unsigned *d_ovf = nullptr;        // device flag: an accumulator ran past 2^63 (raised at read-out)
  cudaStream_t settle = nullptr;    // deposits of the pairs libm settled, beside the passes running on `compute`
  cudaEvent_t ev_settled = nullptr; // settle -> compute / comm_stream
  bool settle_pending = false;      // `compute` has not yet waited for ev_settled
  bool settle_pending_comm = false; // nor has `comm_stream`
  cudaEvent_t slot_pass_ev[SLICER_MAX_SLOTS]; // the stop event (pass_ev ring) of the last pass into accumulator slot q, or nullptr
  unsigned long long slot_epoch[SLICER_MAX_SLOTS];
  size_t pos_stride = 0, mass_stride = 0; // floats per staging pool (16-byte multiples)
  size_t pcap = 0, mcap = 0;              // particles / masses a pool holds, padding of the segments included
  // particles per slice the binned path will use (before allocation: what it would allocate)
  size_t bin_slice_hint() const
  {
    if (bin.slice)
      return bin.slice;
    size_t s = cfg.record_capacity ? cfg.record_capacity : ((size_t)1 << 28);
    return cfg.particle_capacity && s > cfg.particle_capacity ? cfg.particle_capacity : s;
  }
  // binned deposit (deposit_binned.cuh): buffers allocated on first use
  struct
  {
    float2 *rec_u = nullptr, *rec_s = nullptr;
    unsigned short *key_u = nullptr;
    float *mass_u = nullptr, *mass_s = nullptr;
    unsigned *region_count = nullptr, *region_hist = nullptr, *bin_count = nullptr, *bin_start = nullptr;
    size_t slice = 0;    // particles per slice
    size_t capacity = 0; // records the buffers hold
  } bin;
  // Part. Degradation (deposit_degrade.cuh): per-particle accepted counts and ranks of the resident batch
  struct
  {
    unsigned char *cnt = nullptr, *keep = nullptr;
    unsigned *rank = nullptr, *block_sums = nullptr;
    size_t stride = 0, nblocks = 0, keep_cap = 0;
    size_t bytes = 0; // device bytes of cnt, rank and block_sums
    int nplanes = 0;
    bool valid = false;
    unsigned long long plane_total[SLICER_MAX_PLANES];
  } deg;
};

static int set_device(slicer_handle *h)
{
  CU(cudaSetDevice(h->cfg.device));
  return 0;
}

extern "C" int slicer_device_count(int *count)
{
  CU(cudaGetDeviceCount(count));
  return 0;
}

extern "C" int slicer_device_memory(int device, size_t *free_bytes, size_t *total_bytes)
{
  if (!free_bytes || !total_bytes)
    return fail("slicer_device_memory: null argument");
  int ndev = 0;
  CU(cudaGetDeviceCount(&ndev));
  if (device < 0 || device >= ndev)
    return fail("slicer_device_memory: device %d out of range (have %d)", device, ndev);
  int prev = 0;
  CU(cudaGetDevice(&prev));
  CU(cudaSetDevice(device));
  const cudaError_t e = cudaMemGetInfo(free_bytes, total_bytes);
  cudaSetDevice(prev);
  if (e != cudaSuccess)
    return fail("cudaMemGetInfo failed: %s", cudaGetErrorString(e));
  return 0;
}

extern "C" int slicer_alloc_pinned(size_t bytes, void **out)
{
  CU(cudaHostAlloc(out, bytes, cudaHostAllocDefault));
  return 0;
}

extern "C" int slicer_free_pinned(void *p)
{
  CU(cudaFreeHost(p));
  return 0;
}

template <typename T>
static int dev_alloc(slicer_handle *h, T **p, size_t count)
{
  size_t bytes = count * sizeof(T);
  CU(cudaMalloc((void **)p, bytes));
  h->device_bytes += bytes;
  return 0;
}

extern "C" int slicer_create(const slicer_config *cfg, slicer_handle **out)
{
  if (!cfg || !out)
    return fail("slicer_create: null argument");
  if (cfg->max_planes < 1 || cfg->max_planes > SLICER_MAX_SLOTS)
    return fail("slicer_create: max_planes must be 1..%d (SLICER_MAX_SLOTS)", SLICER_MAX_SLOTS);
  if (cfg->npix_max < 1)
    return fail("slicer_create: npix_max must be positive");
  if (cfg->mas != SLICER_MAS_TSC && cfg->mas != SLICER_MAS_NGP)
    return fail("slicer_create: unknown mass-assignment scheme %d", cfg->mas);
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0)
    return fail("slicer_create: no usable CUDA device (%s); this library has no CPU path",
                e == cudaSuccess ? "device count is 0" : cudaGetErrorString(e));
  if (cfg->device < 0 || cfg->device >= ndev)
    return fail("slicer_create: device %d out of range (have %d)", cfg->device, ndev);
  slicer_handle *h = new slicer_handle;
  for (int q = 0; q < SLICER_MAX_SLOTS; q++)
  {
    h->ev_slot[q] = nullptr;
    h->slot_reducing[q] = false;
    h->slot_pass_ev[q] = nullptr;
  }
  h->cfg = *cfg;
  h->frac_bits = cfg->frac_bits > 0 ? cfg->frac_bits : 40;
  if (h->frac_bits > 60)
  {
    delete h;
    return fail("slicer_create: frac_bits must be <= 60");
  }
  if (h->cfg.max_m <= 0)
    h->cfg.max_m = 1e3; /* densitymaps.h:21 */
  h->ntypes_alloc = cfg->per_type_maps ? SLICER_NTYPES : 1;
  h->no_series = getenv("SLICER_B200_NO_SERIES") != nullptr;
  h->no_lean = getenv("SLICER_B200_NO_LEAN") != nullptr;
  if (const char *dbg = getenv("SLICER_B200_DEBUG"))
    h->debug = atoi(dbg);
  h->npix2max = (size_t)cfg->npix_max * (size_t)cfg->npix_max;
  memset(&h->stats, 0, sizeof(h->stats));
  memset(h->plane_npix, 0, sizeof(h->plane_npix));
  int rc = 0;
  // SLICER_B200_TIMING: wall-clock of the set-up phases on stderr (context, allocations, kernel set-up)
  const bool timing = getenv("SLICER_B200_TIMING") != nullptr;
  auto now = [] { return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count(); };
  const double t_start = now();
  double t_ctx = 0, t_alloc = 0;
  do
  {
    if ((rc = set_device(h)))
      break;
    if (timing)
      cudaFree(nullptr); // force the context now, so that the phases are attributed correctly
    t_ctx = now();
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, cfg->device) != cudaSuccess)
    {
      rc = fail("cudaGetDeviceProperties failed");
      break;
    }
    if (prop.major < 10)
    {
      rc = fail("slicer_create: device %d is sm_%d%d; this library is built for sm_100a (B200) only", cfg->device,
                prop.major, prop.minor);
      break;
    }
    h->sm_count = prop.multiProcessorCount;
#define TRY(expr)                                                        \
  if ((expr) != cudaSuccess)                                             \
  {                                                                      \
    rc = fail("%s failed: %s", #expr, cudaGetErrorString(cudaGetLastError())); \
    break;                                                               \
  }
    TRY(cudaStreamCreateWithFlags(&h->compute, cudaStreamNonBlocking));
    TRY(cudaStreamCreateWithFlags(&h->copy, cudaStreamNonBlocking));
    TRY(cudaStreamCreateWithFlags(&h->comm_stream, cudaStreamNonBlocking));
    TRY(cudaStreamCreateWithFlags(&h->aux, cudaStreamNonBlocking));
    TRY(cudaStreamCreateWithFlags(&h->settle, cudaStreamNonBlocking));
    TRY(cudaEventCreateWithFlags(&h->ev_settled, cudaEventDisableTiming));
    TRY(cudaEventCreateWithFlags(&h->defer.bank[0].ev_done, cudaEventDisableTiming));
    TRY(cudaEventCreateWithFlags(&h->defer.bank[1].ev_done, cudaEventDisableTiming));
    TRY(cudaEventCreateWithFlags(&h->ev_zero_start, cudaEventDisableTiming));
    TRY(cudaEventCreateWithFlags(&h->ev_zero_done, cudaEventDisableTiming));
    TRY(cudaEventCreateWithFlags(&h->ev_pass_done, cudaEventDisableTiming));
    for (int q = 0; q < cfg->max_planes; q++)
      TRY(cudaEventCreateWithFlags(&h->ev_slot[q], cudaEventDisableTiming));
    TRY(cudaEventCreateWithFlags(&h->ev_copy, cudaEventDisableTiming));
    TRY(cudaEventCreateWithFlags(&h->ev_buf_done[0], cudaEventDisableTiming));
    TRY(cudaEventCreateWithFlags(&h->ev_buf_done[1], cudaEventDisableTiming));
    TRY(cudaEventCreate(&h->ev_t0));
    TRY(cudaEventCreate(&h->ev_t1));
    h->pass_ev.resize(2 * PASS_RING, nullptr);
    {
      bool bad = false;
      for (size_t i = 0; i < h->pass_ev.size() && !bad; i++)
        bad = cudaEventCreate(&h->pass_ev[i]) != cudaSuccess;
      if (bad)
      {
        rc = fail("cudaEventCreate failed: %s", cudaGetErrorString(cudaGetLastError()));
        break;
      }
    }
#undef TRY
    h->nbuf = cfg->staging_buffers >= 2 ? 2 : 1;
    // +64 floats of slack so 16-byte bulk copies may over-read the tail of the last chunk; every pool starts on a 16-byte
    // boundary whatever the capacity (cp.async.bulk needs 16-byte aligned sources)
    // (internal capacities: the caller's, rounded up to a multiple of 4, plus room for the 16-byte padding of up to 8 segments)
    h->pcap = cfg->particle_capacity ? ((cfg->particle_capacity + 3) & ~(size_t)3) + 32 : 0;
    h->mcap = cfg->mass_capacity ? ((cfg->mass_capacity + 3) & ~(size_t)3) + 32 : 0;
    h->pos_stride = h->pcap * 3 + 64;
    h->mass_stride = h->mcap + 64;
    if (cfg->particle_capacity && (rc = dev_alloc(h, &h->d_pos_pool, h->nbuf * h->pos_stride)))
      break;
    if (cfg->mass_capacity && (rc = dev_alloc(h, &h->d_mass_pool, h->nbuf * h->mass_stride)))
      break;
    // 2^19 entries (12 MiB) per bank and per 16 slots: one bank may hold the passes of every slot range (run_pass), and the
    // flagged pairs (about 8 per million accepted pairs at the default guard) grow with the planes deposited between settles
    h->defer.cap = (1u << 19) * (unsigned)((cfg->max_planes + SLICER_MAX_PLANES - 1) / SLICER_MAX_PLANES);
    if ((rc = dev_alloc(h, &h->d_ovf, 1)))
      break;
    for (int b = 0; b < 2 && !rc; b++)
    {
      slicer_handle::DeferBank &B = h->defer.bank[b];
      if ((rc = dev_alloc(h, &B.buf, (size_t)h->defer.cap)) || (rc = dev_alloc(h, &B.count, 1)))
        break;
      if (cudaHostAlloc((void **)&B.host, (size_t)h->defer.cap * sizeof(DeferEntry), cudaHostAllocDefault) != cudaSuccess ||
          cudaHostAlloc((void **)&B.host_count, 2 * sizeof(unsigned), cudaHostAllocDefault) != cudaSuccess)
      {
        rc = fail("cudaHostAlloc failed: %s", cudaGetErrorString(cudaGetLastError()));
        break;
      }
      B.host_count[0] = 0;
    }
    if (rc)
      break;
    memset(h->slot_epoch, 0, sizeof(h->slot_epoch));
    h->d_pos = h->d_pos_pool;
    h->d_mass = h->d_mass_pool;
    if ((rc = dev_alloc(h, &h->d_acc, (size_t)cfg->max_planes * h->ntypes_alloc * h->npix2max)))
      break;
    if ((rc = dev_alloc(h, &h->d_counts, (size_t)cfg->max_planes * SLICER_NTYPES * 2)))
      break;
    if ((rc = dev_alloc(h, &h->d_out, h->npix2max)))
      break;
    if ((rc = dev_alloc(h, &h->d_sum, h->npix2max)))
      break;
    t_alloc = now();
    if ((rc = pipelined_init(&h->pipe, h->sm_count)))
    {
      rc = fail("pipelined kernel set-up failed: %s", cudaGetErrorString(cudaGetLastError()));
      break;
    }
    if (cudaMemsetAsync(h->d_acc, 0, (size_t)cfg->max_planes * h->ntypes_alloc * h->npix2max * 8, h->compute) != cudaSuccess ||
        cudaMemsetAsync(h->d_counts, 0, (size_t)cfg->max_planes * SLICER_NTYPES * 2 * 8, h->compute) != cudaSuccess ||
        cudaMemsetAsync(h->defer.bank[0].count, 0, sizeof(unsigned), h->compute) != cudaSuccess ||
        cudaMemsetAsync(h->defer.bank[1].count, 0, sizeof(unsigned), h->compute) != cudaSuccess ||
        cudaMemsetAsync(h->d_ovf, 0, sizeof(unsigned), h->compute) != cudaSuccess ||
        cudaStreamSynchronize(h->compute) != cudaSuccess)
    {
      rc = fail("initial memset failed: %s", cudaGetErrorString(cudaGetLastError()));
      break;
    }
    if (timing)
      fprintf(stderr, "[timing] slicer_create(device %d): context %.3f s, streams + device allocations %.3f s, kernel set-up %.3f s\n", cfg->device,
              t_ctx - t_start, t_alloc - t_ctx, now() - t_alloc);
  } while (0);
  if (rc)
  {
    slicer_destroy(h);
    return rc;
  }
  *out = h;
  return 0;
}

extern "C" void slicer_destroy(slicer_handle *h)
{
  if (!h)
    return;
  cudaSetDevice(h->cfg.device);
  if (h->compute)
    cudaStreamSynchronize(h->compute);
  if (h->copy)
    cudaStreamSynchronize(h->copy);
  if (h->comm_stream)
    cudaStreamSynchronize(h->comm_stream);
  if (h->comm && g_nccl.CommDestroy)
    g_nccl.CommDestroy(h->comm);
  pipelined_destroy(&h->pipe);
  cudaFree(h->deg.cnt);
  cudaFree(h->deg.keep);
  cudaFree(h->deg.rank);
  cudaFree(h->deg.block_sums);
  cudaFree(h->bin.rec_u);
  cudaFree(h->bin.rec_s);
  cudaFree(h->bin.key_u);
  cudaFree(h->bin.mass_u);
  cudaFree(h->bin.mass_s);
  cudaFree(h->bin.region_count);
  cudaFree(h->bin.bin_count);
  cudaFree(h->bin.bin_start);
  cudaFree(h->bin.region_hist);
  if (h->settle)
  {
    cudaStreamSynchronize(h->settle);
    cudaStreamDestroy(h->settle);
  }
  if (h->ev_settled)
    cudaEventDestroy(h->ev_settled);
  cudaFree(h->d_ovf);
  for (int b = 0; b < 2; b++)
  {
    slicer_handle::DeferBank &B = h->defer.bank[b];
    cudaFree(B.buf);
    cudaFree(B.count);
    if (B.host)
      cudaFreeHost(B.host);
    if (B.host_count)
      cudaFreeHost(B.host_count);
    if (B.ev_done)
      cudaEventDestroy(B.ev_done);
  }
  cudaFree(h->d_pos_pool);
  cudaFree(h->d_mass_pool);
  cudaFree(h->d_acc);
  cudaFree(h->d_counts);
  cudaFree(h->d_out);
  cudaFree(h->d_sum);
  if (h->ev_copy)
    cudaEventDestroy(h->ev_copy);
  for (int b = 0; b < 2; b++)
    if (h->ev_buf_done[b])
      cudaEventDestroy(h->ev_buf_done[b]);
  if (h->ev_t0)
    cudaEventDestroy(h->ev_t0);
  if (h->ev_t1)
    cudaEventDestroy(h->ev_t1);
  for (size_t i = 0; i < h->pass_ev.size(); i++)
    if (h->pass_ev[i])
      cudaEventDestroy(h->pass_ev[i]);
  if (h->aux)
  {
    cudaStreamSynchronize(h->aux);
    cudaStreamDestroy(h->aux);
  }
  if (h->ev_zero_start)
    cudaEventDestroy(h->ev_zero_start);
  if (h->ev_zero_done)
    cudaEventDestroy(h->ev_zero_done);
  if (h->ev_pass_done)
    cudaEventDestroy(h->ev_pass_done);
  for (int q = 0; q < SLICER_MAX_SLOTS; q++)
    if (h->ev_slot[q])
      cudaEventDestroy(h->ev_slot[q]);
  if (h->compute)
    cudaStreamDestroy(h->compute);
  if (h->copy)
    cudaStreamDestroy(h->copy);
  if (h->comm_stream)
    cudaStreamDestroy(h->comm_stream);
  delete h;
}

extern "C" int slicer_frac_bits(slicer_handle *h) { return h ? h->frac_bits : -1; }

// ------------------------------------------------------------------------------------------------------------
// staging
// ------------------------------------------------------------------------------------------------------------
extern "C" int slicer_begin_snapshot(slicer_handle *h, double boxsize, const double massarr[SLICER_NTYPES], int hydro)
{
  if (!h)
    return fail("null handle");
  if (!(boxsize > 0))
    return fail("slicer_begin_snapshot: boxsize must be positive");
  if (set_device(h))
    return 1;
  h->boxsize = boxsize;
  for (int i = 0; i < SLICER_NTYPES; i++)
    h->massarr[i] = massarr ? massarr[i] : 0.0;
  h->hydro = hydro;
  return slicer_next_batch(h);
}

extern "C" int slicer_next_batch(slicer_handle *h)
{
  if (!h)
    return fail("null handle");
  if (!(h->boxsize > 0))
    return fail("slicer_begin_snapshot must be called before slicer_next_batch");
  if (set_device(h))
    return 1;
  h->cur_buf = (h->cur_buf + 1) % h->nbuf;
  // this pool is about to be overwritten: copies must wait for the pass that last read it
  CU(cudaStreamWaitEvent(h->copy, h->ev_buf_done[h->cur_buf], 0));
  h->d_pos = h->d_pos_pool ? h->d_pos_pool + (size_t)h->cur_buf * h->pos_stride : nullptr;
  h->d_mass = h->d_mass_pool ? h->d_mass_pool + (size_t)h->cur_buf * h->mass_stride : nullptr;
  h->segs.clear();
  h->pos_used = 0;
  h->mass_used = 0;
  h->deg.valid = false;
  return 0;
}

static bool uses_particle_mass(const slicer_handle *h, int type)
{
  return h->hydro && h->massarr[type] == 0; /* densitymaps.cpp:358 */
}

static int check_stage(slicer_handle *h, int type, int layout)
{
  if (!h)
    return fail("null handle");
  if (type < 0 || type >= SLICER_NTYPES)
    return fail("particle type %d out of range", type);
  if (layout != SLICER_LAYOUT_AOS && layout != SLICER_LAYOUT_SOA)
    return fail("unknown layout %d", layout);
  if (!(h->boxsize > 0))
    return fail("slicer_begin_snapshot must be called before staging");
  return set_device(h);
}

// particles are placed at multiples of 4 so every segment starts 16-byte aligned in both layouts
static size_t pad4(size_t n) { return (n + 3) & ~(size_t)3; }

extern "C" int slicer_stage_particles(slicer_handle *h, int type, const float *pos, int layout, const float *mass, size_t n)
{
  if (check_stage(h, type, layout))
    return 1;
  if (n == 0)
    return 0;
  if (!pos)
    return fail("slicer_stage_particles: null positions");
  const bool pm = uses_particle_mass(h, type);
  if (pm && !mass)
    return fail("slicer_stage_particles: type %d has massarr==0 in a hydro snapshot: per-particle masses required", type);
  const size_t npad = pad4(n);
  if (h->pos_used + npad > h->pcap)
    return fail("slicer_stage_particles: %zu particles exceed particle_capacity %zu", h->pos_used + n, h->cfg.particle_capacity);
  if (pm && h->mass_used + npad > h->mcap)
    return fail("slicer_stage_particles: %zu masses exceed mass_capacity %zu", h->mass_used + n, h->cfg.mass_capacity);
  Segment s;
  s.type = type;
  s.n = n;
  s.layout = layout;
  s.soa_stride = npad;
  float *dst = h->d_pos + 3 * h->pos_used;
  if (layout == SLICER_LAYOUT_AOS)
    CU(cudaMemcpyAsync(dst, pos, n * 3 * sizeof(float), cudaMemcpyHostToDevice, h->copy));
  else
    for (int k = 0; k < 3; k++)
      CU(cudaMemcpyAsync(dst + k * npad, pos + (size_t)k * n, n * sizeof(float), cudaMemcpyHostToDevice, h->copy));
  s.dpos = dst;
  s.dmass = nullptr;
  if (pm)
  {
    float *md = h->d_mass + h->mass_used;
    CU(cudaMemcpyAsync(md, mass, n * sizeof(float), cudaMemcpyHostToDevice, h->copy));
    s.dmass = md;
    h->mass_used += npad;
  }
  h->pos_used += npad;
  h->segs.push_back(s);
  h->copy_pending = true;
  return 0;
}

extern "C" int slicer_stage_device(slicer_handle *h, int type, const void *dev_pos, int layout, const void *dev_mass, size_t n)
{
  if (check_stage(h, type, layout))
    return 1;
  if (n == 0)
    return 0;
  if (!dev_pos)
    return fail("slicer_stage_device: null positions");
  if (((uintptr_t)dev_pos & 15) || ((uintptr_t)dev_mass & 15))
    return fail("slicer_stage_device: device pointers must be 16-byte aligned");
  if (layout == SLICER_LAYOUT_SOA && (n & 3))
    return fail("slicer_stage_device: SoA segments need n %% 4 == 0 (rows must stay 16-byte aligned)");
  const bool pm = uses_particle_mass(h, type);
  if (pm && !dev_mass)
    return fail("slicer_stage_device: per-particle masses required for type %d", type);
  Segment s;
  s.type = type;
  s.n = n;
  s.layout = layout;
  s.soa_stride = n;
  s.dpos = (const float *)dev_pos;
  s.dmass = pm ? (const float *)dev_mass : nullptr;
  h->segs.push_back(s);
  return 0;
}

extern "C" int slicer_stage_synthetic(slicer_handle *h, int type, size_t n, uint64_t seed, int layout)
{
  return slicer_stage_synthetic_window(h, type, 0, n, seed, layout);
}

extern "C" int slicer_stage_synthetic_window(slicer_handle *h, int type, unsigned long long start, size_t n, uint64_t seed, int layout)
{
  if (check_stage(h, type, layout))
    return 1;
  if (n == 0)
    return 0;
  if (uses_particle_mass(h, type))
    return fail("slicer_stage_synthetic: synthetic segments carry no per-particle mass");
  const size_t npad = pad4(n);
  if (h->pos_used + npad > h->pcap)
    return fail("slicer_stage_synthetic: %zu particles exceed particle_capacity %zu", h->pos_used + n, h->cfg.particle_capacity);
  Segment s;
  s.type = type;
  s.n = n;
  s.layout = layout;
  s.soa_stride = npad;
  float *dst = h->d_pos + 3 * h->pos_used;
  s.dpos = dst;
  s.dmass = nullptr;
  const int blocks = (int)((3 * n + 255) / 256 < (size_t)h->sm_count * 16 ? (3 * n + 255) / 256 : (size_t)h->sm_count * 16);
  // generated on the copy stream so it orders with other staging work
  synth_positions_kernel<<<blocks, 256, 0, h->copy>>>(dst, n, npad, layout == SLICER_LAYOUT_SOA, seed, (float)h->boxsize, start);
  CU(cudaGetLastError());
  h->stats.launches++;
  h->pos_used += npad;
  h->segs.push_back(s);
  h->copy_pending = true;
  return 0;
}

extern "C" int slicer_download_segment(slicer_handle *h, int segment, float *pos_out, float *mass_out)
{
  if (!h)
    return fail("null handle");
  if (segment < 0 || segment >= (int)h->segs.size())
    return fail("segment %d out of range", segment);
  if (set_device(h))
    return 1;
  const Segment &s = h->segs[segment];
  CU(cudaStreamSynchronize(h->copy));
  if (pos_out)
  {
    if (s.layout == SLICER_LAYOUT_AOS)
      CU(cudaMemcpy(pos_out, s.dpos, s.n * 3 * sizeof(float), cudaMemcpyDeviceToHost));
    else
      for (int k = 0; k < 3; k++)
        CU(cudaMemcpy(pos_out + (size_t)k * s.n, s.dpos + k * s.soa_stride, s.n * sizeof(float), cudaMemcpyDeviceToHost));
  }
  if (mass_out && s.dmass)
    CU(cudaMemcpy(mass_out, s.dmass, s.n * sizeof(float), cudaMemcpyDeviceToHost));
  return 0;
}

// ------------------------------------------------------------------------------------------------------------
// pass set-up
// ------------------------------------------------------------------------------------------------------------
static float float_ceil(double d)
{ // smallest float >= d
  float f = (float)d;
  if ((double)f < d)
    f = nextafterf(f, INFINITY);
  return f;
}
static float float_floor(double d)
{ // largest float <= d
  float f = (float)d;
  if ((double)f > d)
    f = nextafterf(f, -INFINITY);
  return f;
}
static bool is_f32(double d) { return (double)(float)d == d; }

// planes[i] deposits into accumulator slot first_slot + i
static int build_pass(slicer_handle *h, const slicer_plane_desc *planes, int nplanes, PassParams *P, int first_slot = 0)
{
  if (nplanes < 1 || nplanes > h->cfg.max_planes)
    return fail("slicer_deposit: nplanes %d outside 1..%d (max_planes)", nplanes, h->cfg.max_planes);
  if (nplanes > SLICER_MAX_PLANES) // (a handle may have more slots than one pass can fill)
    return fail("slicer_deposit: %d planes in one pass, more than SLICER_MAX_PLANES (%d)", nplanes, SLICER_MAX_PLANES);
  memset(P, 0, sizeof(*P));
  // group planes by randomisation
  int xf_of[SLICER_MAX_PLANES];
  int nx = 0;
  int rep[SLICER_MAX_XFORMS];
  for (int i = 0; i < nplanes; i++)
  {
    const slicer_plane_desc &d = planes[i];
    if (d.face < 1 || d.face > 6)
      return fail("plane %d: face %d outside 1..6", i, d.face);
    for (int k = 0; k < 3; k++)
      if (d.sgn[k] != 1 && d.sgn[k] != -1)
        return fail("plane %d: sgn[%d]=%d must be +1 or -1", i, k, d.sgn[k]);
    if (d.npix < 1 || d.npix > h->cfg.npix_max)
      return fail("plane %d: npix %d outside 1..%d (npix_max)", i, d.npix, h->cfg.npix_max);
    if (d.nrepperp < 0)
      return fail("plane %d: negative nrepperp", i);
    if (!(d.ld2 > d.ld) || d.ld < 0)
      return fail("plane %d: need 0 <= ld < ld2", i);
    if (!(d.fovradiants > 0))
      return fail("plane %d: fovradiants must be positive", i);
    int t = -1;
    for (int j = 0; j < nx && t < 0; j++)
    {
      const slicer_plane_desc &r = planes[rep[j]];
      if (memcmp(r.sgn, d.sgn, sizeof(d.sgn)) == 0 && r.face == d.face && r.centre[0] == d.centre[0] &&
          r.centre[1] == d.centre[1] && r.centre[2] == d.centre[2] && r.rcase == d.rcase)
        t = j;
    }
    if (t < 0)
    {
      if (nx == SLICER_MAX_XFORMS)
        return fail("slicer_deposit: more than %d distinct randomisations in one pass", SLICER_MAX_XFORMS);
      rep[nx] = i;
      t = nx++;
    }
    xf_of[i] = t;
  }
  P->nxform = nx;
  P->nplanes = nplanes;
  P->debug = h->debug;
  P->fast = 1;
  P->est_accept = 0;
  P->pair = 0;
  static const int perm_of_face[7][3] = {{0, 1, 2}, {0, 1, 2}, {0, 2, 1}, {1, 2, 0}, {1, 0, 2}, {2, 0, 1}, {2, 1, 0}}; /* gadget2io.cpp:223-252 */
  int slot = 0;
  for (int t = 0; t < nx; t++)
  {
    const slicer_plane_desc &r = planes[rep[t]];
    XformDev &X = P->xf[t];
    X.box = h->boxsize;
    X.boxf = (float)h->boxsize;
    X.exact_f32 = is_f32(h->boxsize);
    for (int k = 0; k < 3; k++)
    {
      X.c[k] = r.centre[k];
      X.cf[k] = (float)r.centre[k];
      X.exact_f32 = X.exact_f32 && is_f32(r.centre[k]);
      X.perm[k] = perm_of_face[r.face][k];
      X.sgn[k] = (float)r.sgn[X.perm[k]];
    }
    X.rcase = r.rcase;
    X.first_plane = slot;
    X.nplanes = 0;
    X.zmin = INFINITY;
    X.zmax = -INFINITY;
    for (int i = 0; i < nplanes; i++)
    {
      if (xf_of[i] != t)
        continue;
      const slicer_plane_desc &d = planes[i];
      // NOTE: device slot != caller's plane index; acc/counts pointers keep the caller's index i
      PlaneDev &L = P->pl[slot++];
      X.nplanes++;
      const double minDist = d.ld / h->boxsize * 1.e+3 / POS_U;  /* densitymaps.cpp:346 */
      const double maxDist = d.ld2 / h->boxsize * 1.e+3 / POS_U; /* densitymaps.cpp:347 */
      L.zlo = float_ceil(minDist);
      L.zhi = float_ceil(maxDist);
      if (L.zlo < X.zmin)
        X.zmin = L.zlo;
      if (L.zhi > X.zmax)
        X.zmax = L.zhi;
      L.npix = d.npix;
      L.npixf = (float)d.npix;
      L.nrep = d.nrepperp;
      L.pow2 = (d.npix & (d.npix - 1)) == 0;
      L.T = d.fovradiants * (1. + 2. / d.npix) * 0.5; /* densitymaps.cpp:383 */
      L.fovrad = d.fovradiants;
      L.dl = 1. / double(d.npix);  /* utilities.cpp:50 */
      L.half_dl = 0.5 * L.dl;      /* utilities.cpp:9  */
      L.onehalf_dl = 0.5 * 3.0 * L.dl; /* utilities.cpp:11 */
      L.scale = ldexp(1.0, h->frac_bits);
      L.scalef = (float)L.scale;
      L.dlf = (float)L.dl;
      L.half_dlf = (float)L.half_dl;
      L.onehalf_dlf = (float)L.onehalf_dl;
      if (L.T < 1.5)
      {
        const double tt = tan(L.T) * (1.0 + 1e-5);
        L.pre_ty = float_ceil(tt);
        L.pre_tx = float_ceil(tt / cos(L.T));
      }
      else
      {
        L.pre_tx = INFINITY;
        L.pre_ty = INFINITY;
      }
      // small-angle series for asin/atan (device_chain.cuh): enough terms that arg_lim^(2 nt) < 2^-55
      L.nt = 0;
      L.arg_lim = 0;
      L.guard_eta = h->cfg.guard_eta >= LEAN_ETA ? h->cfg.guard_eta : LEAN_ETA;
      L.guard_T = 2.0 * L.guard_eta * L.T; // an angle is (map coordinate - 0.5) * fov: the same guard, in radians
      if (!h->no_series && isfinite(L.pre_tx) && (double)L.pre_tx * 1.01 <= 0.385)
      {
        L.arg_lim = (double)L.pre_tx * 1.01;
        L.nt = (int)ceil(55.0 * log(2.0) / (2.0 * log(1.0 / L.arg_lim)));
        if (L.nt < 2)
          L.nt = 2;
        if (L.nt > 20)
          L.nt = 0;
      }
      const int slot = first_slot + i;
      L.acc = h->d_acc + (size_t)slot * h->ntypes_alloc * h->npix2max;
      L.counts = h->d_counts + (size_t)slot * SLICER_NTYPES * 2;
      L.type_stride = h->cfg.per_type_maps ? h->npix2max : 0;
      L.slot = slot;
      h->plane_npix[slot] = d.npix;
      {
        // fraction of a uniform snapshot this plane accepts: slab thickness x (field width / box)^2 at mid-distance
        const double w = L.T < 1.5 ? 2.0 * tan(L.T) * 0.5 * (minDist + maxDist) : 1.0;
        P->est_accept += (maxDist - minDist) * (w < 1.0 ? w * w : 1.0);
      }
    }
    for (int a = X.first_plane; a < X.first_plane + X.nplanes; a++)
    {
      if (!P->pl[a].pow2 || P->pl[a].nrep != 0)
        P->fast = 0;
      for (int b = a + 1; b < X.first_plane + X.nplanes; b++)
        if (P->pl[a].zlo < P->pl[b].zhi && P->pl[b].zlo < P->pl[a].zhi)
          P->fast = 0; // overlapping slabs: a particle can belong to two planes
    }
    // float screen of the pipelined kernel (deposit_pipelined.cuh: screen()); all margins are >= 5x the
    // worst-case difference between the screen's coordinates and the exact chain's
    X.tmax = 0.f;
    for (int q = X.first_plane; q < X.first_plane + X.nplanes; q++)
      if (P->pl[q].pre_tx > X.tmax)
        X.tmax = P->pl[q].pre_tx;
    for (int k = 0; k < 3; k++)
    {
      X.sinv[k] = (float)((double)X.sgn[k] / h->boxsize);
      X.offs[k] = (float)((X.sgn[k] < 0.f ? 1.0 : 0.0) - X.c[k]);
    }
    const float zulp = nextafterf(X.zmax, INFINITY) - X.zmax;
    const float mz = 2e-6f + 4.f * zulp;
    X.zlo_m = X.zmin - mz;
    X.zhi_m = X.zmax + mz;
    X.zamb = 0.5f - 2e-6f;
    X.thr_m = isinf(X.tmax) ? 0.f : 4e-6f + X.tmax * mz * 1.01f;
    X.raw_hi = float_floor(h->boxsize * (1.0 - 1e-6)); // 0 < raw < raw_hi  =>  raw/box in (0,1): no wrap at the first site
    X.nboxf = -X.boxf;
    for (int k = 0; k < 3; k++)
      X.wadd[k] = X.sgn[k] < 0.f ? 1.f : 0.f;
  }
  P->pair = P->fast && P->pl[0].nt > 0;
  for (int t = 0; t < P->nxform; t++)
    if (!P->xf[t].exact_f32)
      P->pair = 0; // the lean exact phase assumes a float-exact box and centre
  for (int q = 1; q < P->nplanes; q++)
    if (P->pl[q].T != P->pl[0].T || P->pl[q].fovrad != P->pl[0].fovrad || P->pl[q].npix != P->pl[0].npix)
      P->pair = 0;
  // lean exact phase (lean_math.h, deposit_pipelined.cuh: drain_lean): one narrow field and map size for all planes, float-exact
  // box and centres, and a box size for which the unchecked float division cannot leave the normal range
  P->lean.enabled = 0;
  if (P->pair && h->boxsize >= 0x1p-40 && h->boxsize <= 0x1p40 && !h->no_lean)
  {
    lean_setup(&P->lean, P->pl[0].fovrad, P->pl[0].T, h->cfg.guard_eta);
    if (!(P->xf[0].raw_hi > P->lean.umin))
      P->lean.enabled = 0;
    for (int t = 0; t < P->nxform; t++)
      for (int k = 0; k < 3; k++)
        if (!(P->xf[t].cf[k] >= 0.f && P->xf[t].cf[k] <= 1.f))
          P->lean.enabled = 0; // lean_axis assumes a centre inside the box (randomizeBox draws it in [0, 1])
  }
  return 0;
}

static void fill_segment(const slicer_handle *h, const Segment &s, SegmentDev *D)
{
  D->pos = s.dpos;
  D->mass = s.dmass;
  D->n = s.n;
  D->soa_stride = s.soa_stride;
  D->const_mass = (float)h->massarr[s.type]; /* densitymaps.cpp:372: num_float1 = data.massarr[i] */
  D->max_m = float_floor(h->cfg.max_m);      /* float m > double MAX_M  <=>  m > largest float <= MAX_M */
  D->type = s.type;
  D->layout = s.layout;
}

// ------------------------------------------------------------------------------------------------------------
// binned deposit: K1 (records) -> histogram -> scan -> scatter -> tile deposit, slice by slice
// ------------------------------------------------------------------------------------------------------------
static int binned_tiles(const PassParams &P) { return (P.pl[0].npix + binned::TILE - 1) / binned::TILE; }
// Sort bins = (plane, tile row, group of 2^gshift tiles along x).  Groups are as small as possible for the bins of the pass to
// fit one sort (MAX_BINS); beyond groups of four tiles the sort runs in windows of the bins.
static int binned_gshift(const PassParams &P)
{
  const int nt = binned_tiles(P);
  int g = 0;
  while (g < 2 && (long long)P.nplanes * nt * ((nt + (1 << g) - 1) >> g) > binned::MAX_BINS)
    g++;
  return g;
}

// 0: direct map atomics; 1: binned.  When the planes' tiles exceed MAX_BINS even in groups of four (8192^2 maps from 8 planes
// up, 16384^2 from 3) the records are still produced once; the sort and the tile deposit then run window by window over the
// bins (binned_pass).
static int use_binned(const slicer_handle *h, const PassParams &P, const SegmentDev &D)
{
  if (!P.fast || h->cfg.deposit_mode == SLICER_DEPOSIT_DIRECT)
    return 0;
  for (int q = 1; q < P.nplanes; q++)
    if (P.pl[q].npix != P.pl[0].npix)
      return 0;
  const int nt = binned_tiles(P), gs = binned_gshift(P);
  if ((long long)P.nplanes * nt * ((nt + (1 << gs) - 1) >> gs) > 65536)
    return 0; // record keys are 16 bits (16 planes of 21248^2 pixels still fit)
  if (h->cfg.deposit_mode == SLICER_DEPOSIT_BINNED)
    return 1;
  // the sort + tile kernels cost ~65 us per segment before the first record; a record then costs ~50 ps against ~105 ps of
  // direct atomics (measured on 2^24- and 2^27-particle segments): worth it from ~1.2 million expected records
  if (P.est_accept * (double)D.n < 1.2e6)
    return 0;
  // measured break-even (DESIGN.md §5): 3 % of the snapshot accepted; 1.5 % when one slice holds the whole batch, or when
  // the planes' accumulators are several times the L2 (> 256 MiB, e.g. 4096^2 and 8192^2 maps: the direct path's atomics go to HBM)
  const bool big_maps = (size_t)P.nplanes * P.pl[0].npix * P.pl[0].npix * sizeof(unsigned long long) > ((size_t)256 << 20);
  return P.est_accept > (h->bin_slice_hint() >= D.n || big_maps ? 0.015 : 0.03) ? 1 : 0;
}

static int binned_alloc(slicer_handle *h, bool need_mass)
{
  if (h->bin.rec_u && need_mass && !h->bin.mass_u)
  { // first segment with per-particle masses on this handle (e.g. staged from device memory without a mass_capacity)
    if (dev_alloc(h, &h->bin.mass_u, h->bin.capacity) || dev_alloc(h, &h->bin.mass_s, h->bin.capacity))
      return 1;
  }
  if (h->bin.rec_u)
    return 0;
  size_t slice = h->cfg.record_capacity ? h->cfg.record_capacity : ((size_t)1 << 28);
  if (slice > ((size_t)1 << 31))
    slice = (size_t)1 << 31; // record offsets are 32-bit
  size_t cap_particles = h->cfg.particle_capacity ? h->cfg.particle_capacity : slice;
  if (slice > cap_particles)
    slice = cap_particles;
  slice = (slice + pipe::CHUNK - 1) / pipe::CHUNK * pipe::CHUNK;
  // every CTA region is rounded up to whole chunks, times the randomisations of a pass (one record per particle and randomisation)
  const size_t cap = slice + ((size_t)h->pipe.grid_max + 1) * pipe::CHUNK * SLICER_MAX_XFORMS;
  if (dev_alloc(h, &h->bin.rec_u, cap) || dev_alloc(h, &h->bin.rec_s, cap) || dev_alloc(h, &h->bin.key_u, cap))
    return 1;
  if ((h->cfg.mass_capacity || need_mass) && (dev_alloc(h, &h->bin.mass_u, cap) || dev_alloc(h, &h->bin.mass_s, cap)))
    return 1;
  if (dev_alloc(h, &h->bin.region_count, (size_t)h->pipe.grid_max) ||
      dev_alloc(h, &h->bin.region_hist, (size_t)binned::MAX_BINS * h->pipe.grid_max) ||
      dev_alloc(h, &h->bin.bin_count, (size_t)binned::MAX_BINS) || dev_alloc(h, &h->bin.bin_start, (size_t)binned::MAX_BINS + 1))
    return 1;
  h->bin.slice = slice;
  h->bin.capacity = cap;
  return 0;
}

// Large accumulators are zeroed on a side stream (run_pass) so that the write overlaps the record kernel of a binned pass, which
// does not touch the maps; whatever does touch them calls this first.
static int maps_ready(slicer_handle *h)
{
  if (h->zero_pending)
  {
    CU(cudaStreamWaitEvent(h->compute, h->ev_zero_done, 0));
    h->zero_pending = false;
  }
  return 0;
}

static int binned_pass(slicer_handle *h, const PassParams &P, const SegmentDev &D, const DeferDev &F)
{
  if (binned_alloc(h, D.mass != nullptr))
    return 1;
  const int nt = binned_tiles(P), gshift = binned_gshift(P), ntx = (nt + (1 << gshift) - 1) >> gshift;
  const int nbins = P.nplanes * nt * ntx;
  // one slice as large as the record buffers allow: the per-slice fixed costs (tile zero + flush, sort set-up, kernel tails) fall
  // with the number of slices (round 2, with the prefetching scatter: 15.2 -> 14.75 ms on the densest C3 group between 2^28- and
  // 2^30-particle slices; round 1's scatter had its optimum at 2^28)
  size_t slice = h->bin.slice;
  // a particle yields up to one record per randomisation of the pass: the slice shrinks so that the regions still fit
  if (P.nxform > 1)
  {
    slice = slice / P.nxform / pipe::CHUNK * pipe::CHUNK;
    if (slice < (size_t)pipe::CHUNK)
      slice = pipe::CHUNK;
  }
  for (unsigned long long off = 0; off < D.n; off += slice)
  {
    SegmentDev S = D;
    S.n = D.n - off < slice ? D.n - off : slice;
    S.pos = D.layout == SLICER_LAYOUT_AOS ? D.pos + 3ull * off : D.pos + off;
    S.mass = D.mass ? D.mass + off : nullptr;
    const int grid = pipelined_grid(&h->pipe, S.n);
    const unsigned long long nchunks = (S.n + pipe::CHUNK - 1) / pipe::CHUNK;
    const unsigned long long cmax = (nchunks + grid - 1) / grid;
    binned::EmitDev E;
    E.rec = h->bin.rec_u;
    E.key = h->bin.key_u;
    E.mass = D.mass ? h->bin.mass_u : nullptr;
    E.region_count = h->bin.region_count;
    E.region_cap = cmax * pipe::CHUNK * (unsigned long long)P.nxform; // one region per K1 CTA: every (particle, randomisation) pair of its chunks could be accepted
    E.ntile = nt;
    E.ntx = ntx;
    E.gshift = gshift;
    const int nregions = grid;
    // few bins (one sort window of at most HIST_BINS): the record kernel counts its region's records per bin itself
    const bool k1_hist = nbins <= binned::HIST_BINS && nbins <= binned::MAX_BINS;
    E.region_hist = k1_hist ? h->bin.region_hist : nullptr;
    E.nregions = nregions;
    E.nbins = nbins;
    if ((unsigned long long)nregions * E.region_cap > h->bin.capacity)
      return fail("binned deposit: record buffer too small (internal error)");
    binned::SortDev Q;
    Q.rec_u = h->bin.rec_u;
    Q.key_u = h->bin.key_u;
    Q.mass_u = E.mass;
    Q.region_count = h->bin.region_count;
    Q.region_cap = E.region_cap;
    Q.nregions = nregions;
    Q.nbins = nbins;
    Q.bin_lo = 0;
    Q.region_hist = h->bin.region_hist;
    Q.bin_count = h->bin.bin_count;
    Q.bin_start = h->bin.bin_start;
    Q.rec_s = h->bin.rec_s;
    Q.mass_s = D.mass ? h->bin.mass_s : nullptr;
    Q.capacity = h->bin.capacity;
    if (pipelined_launch_emit(grid, P, S, E, F, h->compute))
      return fail("record kernel launch failed: %s", cudaGetErrorString(cudaGetLastError()));
    const int nwin = (nbins + binned::MAX_BINS - 1) / binned::MAX_BINS;
    const int wbins = (nbins + nwin - 1) / nwin;
    for (int lo = 0; lo < nbins; lo += wbins)
    {
      Q.bin_lo = lo;
      Q.nbins = nbins - lo < wbins ? nbins - lo : wbins;
      if (!k1_hist)
        binned::bin_histogram_kernel<<<nregions, binned::SCATTER_THREADS, 0, h->compute>>>(Q);
      binned::bin_region_scan_kernel<<<Q.nbins, 1024, 0, h->compute>>>(Q);
      binned::bin_scan_kernel<<<1, 1024, 0, h->compute>>>(Q);
      binned::launch_bin_scatter(Q, nwin > 1, h->compute);
      if (maps_ready(h))
        return 1;
      if (!(h->debug & 4)) // measurement aid: SLICER_B200_DEBUG bit 2 skips the tile deposit
      {
        if (h->cfg.mas == SLICER_MAS_NGP)
          binned::tile_deposit_kernel<SLICER_MAS_NGP><<<Q.nbins << gshift, binned::DEPOSIT_THREADS, binned::TCELLS * 8, h->compute>>>(P, Q, nt, ntx, gshift, D.type, D.const_mass);
        else
          binned::tile_deposit_kernel<SLICER_MAS_TSC><<<Q.nbins << gshift, binned::DEPOSIT_THREADS, binned::TCELLS * 8, h->compute>>>(P, Q, nt, ntx, gshift, D.type, D.const_mass);
      }
      h->stats.launches += k1_hist ? 3 : 4;
    }
    CU(cudaGetLastError());
    h->stats.launches += 1;
  }
  return 0;
}

// fold the device time of the oldest `n` pending passes (all if n == 0) into the stats; blocks until they finished
static int resolve_passes(slicer_handle *h, size_t n)
{
  size_t upto = n ? h->pass_tail + n : h->pass_head;
  if (upto > h->pass_head)
    upto = h->pass_head;
  for (; h->pass_tail < upto; h->pass_tail++)
  {
    cudaEvent_t e0 = h->pass_ev[2 * (h->pass_tail % PASS_RING)], e1 = h->pass_ev[2 * (h->pass_tail % PASS_RING) + 1];
    CU(cudaEventSynchronize(e1));
    float ms = 0;
    CU(cudaEventElapsedTime(&ms, e0, e1));
    h->stats.last_deposit_ms = ms;
    h->stats.deposit_ms_sum += ms;
    h->stats.deposit_passes++;
  }
  return 0;
}

// ------------------------------------------------------------------------------------------------------------
// deferred particles of the lean exact phase (lean_math.h): the reference's own arithmetic with this host's libm
// ------------------------------------------------------------------------------------------------------------
static const unsigned DEFER_HEAD = 16384; // entries copied to the host behind every pass

struct ResolvedRec
{
  float xs, ys, m;
  unsigned short plane, type;
};
static_assert(sizeof(ResolvedRec) <= sizeof(DeferEntry), "resolved records are uploaded into the deferred buffer");

template <int MAS>
__global__ void resolved_deposit_kernel(const __grid_constant__ PassParams P, const ResolvedRec *__restrict__ r, unsigned n)
{
  const unsigned i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n)
    return;
  const ResolvedRec e = r[i];
  const PlaneDev &L = P.pl[e.plane];
  atomicAdd(L.counts + 2 * e.type, 1ull);
  if (P.debug & 1)
    return;
  if (chain::deposit<MAS>(e.xs, e.ys, e.m, L, L.acc + L.type_stride * (unsigned long long)e.type))
    atomicAdd(L.counts + 2 * e.type + 1, 1ull);
}

// densitymaps.cpp:382-386 + utilities.cpp:23-25 for one particle (ni = nj = 0), evaluated on the host like the reference
// (same libm; this translation unit is compiled without FMA contraction)
static bool host_project(const DeferEntry &e, const PlaneDev &L, float *xs, float *ys)
{
  volatile double X = (double)e.x - 0.5, Y = (double)e.y - 0.5, Z = (double)e.z;
  volatile double xx = X * X, yy = Y * Y, zz = Z * Z;
  volatile double sum = xx + yy;
  sum = sum + zz;
  const double d = sqrt(sum);
  volatile double sd = X / d;
  const double dec = asin(sd);
  const double ra = atan2(Y, Z);
  if (!(fabs(ra) <= L.T && fabs(dec) <= L.T))
    return false;
  volatile double vx = dec / L.fovrad, vy = ra / L.fovrad;
  vx = vx + 0.5;
  vy = vy + 0.5;
  *xs = (float)vx;
  *ys = (float)vy;
  return true;
}

// Settle the particles the passes of one bank deferred: waits for the bank's last pass (not for what was submitted to the
// compute stream after it), evaluates them with libm and deposits the accepted ones on the settle stream.
static int resolve_bank(slicer_handle *h, int bi)
{
  slicer_handle::DeferBank &B = h->defer.bank[bi];
  if (B.passes.empty())
    return 0;
  if (set_device(h))
    return 1;
  // run_pass copies the counter and the head of the list to pinned memory behind every pass: one wait settles the usual
  // case (a few thousand entries), without further round trips
  CU(cudaEventSynchronize(B.ev_done));
  const unsigned n = B.host_count[0];
  if (n > h->defer.cap)
  {
    h->defer.failed = true;
    B.passes.clear();
    B.slot_mask = 0;
    CU(cudaMemsetAsync(B.count, 0, sizeof(unsigned), h->compute));
    B.host_count[0] = 0;
    return fail("%u particles within the rounding guard of a decision boundary exceed the deferred buffer (%u): the planes deposited since the "
                "last fetch are incomplete; deposit and fetch in smaller batches",
                n, h->defer.cap);
  }
  if (n)
  {
    if (n > DEFER_HEAD)
    {
      CU(cudaMemcpyAsync(B.host + DEFER_HEAD, B.buf + DEFER_HEAD, (size_t)(n - DEFER_HEAD) * sizeof(DeferEntry), cudaMemcpyDeviceToHost, h->settle));
      CU(cudaStreamSynchronize(h->settle));
    }
    const size_t np = B.passes.size();
    std::vector<std::vector<ResolvedRec>> out(np);
    for (unsigned i = 0; i < n; i++)
    {
      const DeferEntry &e = B.host[i];
      if (e.pass >= np || e.plane >= SLICER_MAX_PLANES)
        return fail("corrupt deferred entry (internal error)");
      const slicer_handle::SavedPass &sp = B.passes[e.pass];
      const PlaneDev &L = sp.P.pl[e.plane];
      if (sp.epoch[e.plane] != h->slot_epoch[L.slot])
      {
        h->stats.flagged_void++;
        continue; // the accumulator was zeroed after that pass
      }
      ResolvedRec r;
      h->stats.flagged_pairs++;
      if (!host_project(e, L, &r.xs, &r.ys))
        continue;
      r.m = e.m;
      r.plane = e.plane;
      r.type = e.type;
      out[e.pass].push_back(r);
    }
    // (the list itself is the staging area of the settled pairs: the bank's passes are over, nothing appends to it)
    ResolvedRec *dev = reinterpret_cast<ResolvedRec *>(B.buf);
    ResolvedRec *stage = reinterpret_cast<ResolvedRec *>(B.host);
    size_t off = 0;
    for (size_t k = 0; k < np; k++)
    {
      const unsigned m = (unsigned)out[k].size();
      if (!m)
        continue;
      memcpy(stage + off, out[k].data(), (size_t)m * sizeof(ResolvedRec));
      CU(cudaMemcpyAsync(dev + off, stage + off, (size_t)m * sizeof(ResolvedRec), cudaMemcpyHostToDevice, h->settle));
      if (h->cfg.mas == SLICER_MAS_NGP)
        resolved_deposit_kernel<SLICER_MAS_NGP><<<(m + 127) / 128, 128, 0, h->settle>>>(B.passes[k].P, dev + off, m);
      else
        resolved_deposit_kernel<SLICER_MAS_TSC><<<(m + 127) / 128, 128, 0, h->settle>>>(B.passes[k].P, dev + off, m);
      CU(cudaGetLastError());
      h->stats.launches++;
      off += m;
    }
    CU(cudaMemsetAsync(B.count, 0, sizeof(unsigned), h->settle));
    B.host_count[0] = 0;
    // whatever touches the accumulators or this bank next (a pass, a read-out, a reduce) waits for these on the device;
    // the next use of the pinned mirror is behind the next cudaEventSynchronize(B.ev_done), which these precede in stream order
    CU(cudaEventRecord(h->ev_settled, h->settle));
    h->settle_pending = h->settle_pending_comm = true;
  }
  B.passes.clear();
  B.slot_mask = 0;
  return 0;
}

// Settle what the passes into accumulator slots [lo, lo + n) deferred (n < 0: every pass submitted so far): the older bank first.
static int resolve_deferred(slicer_handle *h, int lo = 0, int n = -1)
{
  uint64_t mask = ~(uint64_t)0;
  if (n >= 0)
  {
    mask = 0;
    for (int q = lo; q < lo + n && q < SLICER_MAX_SLOTS; q++)
      mask |= (uint64_t)1 << q;
  }
  for (int k = 1; k <= 2; k++)
  {
    const int bi = (h->defer.cur + k) & 1;
    if ((h->defer.bank[bi].slot_mask & mask) && resolve_bank(h, bi))
      return 1;
  }
  return 0;
}

// the compute stream (or the communication stream) must see the deposits of the settled pairs before it touches accumulators
static int wait_settled(slicer_handle *h, bool comm)
{
  if (!comm && h->settle_pending)
  {
    CU(cudaStreamWaitEvent(h->compute, h->ev_settled, 0));
    h->settle_pending = false;
  }
  if (comm && h->settle_pending_comm)
  {
    CU(cudaStreamWaitEvent(h->comm_stream, h->ev_settled, 0));
    h->settle_pending_comm = false;
  }
  return 0;
}

// compute-stream work on accumulator slots [lo, lo + n) must follow the reduces still running on them
static int wait_slot_reduces(slicer_handle *h, int lo, int n)
{
  for (int q = lo; q < lo + n && q < SLICER_MAX_SLOTS; q++)
    if (h->slot_reducing[q])
    {
      CU(cudaStreamWaitEvent(h->compute, h->ev_slot[q], 0));
      h->slot_reducing[q] = false;
    }
  return 0;
}

// staged particles must be on the device before the compute stream reads them
static int staging_fence(slicer_handle *h)
{
  if (h->copy_pending)
  {
    CU(cudaEventRecord(h->ev_copy, h->copy));
    CU(cudaStreamWaitEvent(h->compute, h->ev_copy, 0));
    h->copy_pending = false;
  }
  return 0;
}

// Every write into accumulator slots [lo, lo + n) on the compute stream claims them first: it follows the reduces still reading
// them and the deposits of the pairs libm settled.  A write that does not accumulate also zeroes them and voids the pairs earlier
// passes into them deferred; large accumulators are zeroed on `aux`, so the writer calls maps_ready before it touches them.
static int claim_slots(slicer_handle *h, int lo, int n, bool accumulate)
{
  if (wait_slot_reduces(h, lo, n) || wait_settled(h, false))
    return 1;
  if (accumulate)
    return 0;
  const size_t zbytes = (size_t)n * h->ntypes_alloc * h->npix2max * sizeof(unsigned long long);
  unsigned long long *zptr = h->d_acc + (size_t)lo * h->ntypes_alloc * h->npix2max;
  if (zbytes >= ((size_t)64 << 20))
  { // (8192^2 planes: 2 GiB per pass, 0.7 ms on the compute stream) after everything queued so far, beside what comes next
    if (maps_ready(h))
      return 1;
    CU(cudaEventRecord(h->ev_zero_start, h->compute));
    CU(cudaStreamWaitEvent(h->aux, h->ev_zero_start, 0));
    CU(cudaMemsetAsync(zptr, 0, zbytes, h->aux));
    CU(cudaEventRecord(h->ev_zero_done, h->aux));
    h->zero_pending = true;
  }
  else
    CU(cudaMemsetAsync(zptr, 0, zbytes, h->compute));
  CU(cudaMemsetAsync(h->d_counts + (size_t)lo * SLICER_NTYPES * 2, 0, (size_t)n * SLICER_NTYPES * 2 * sizeof(unsigned long long), h->compute));
  for (int q = lo; q < lo + n; q++)
    h->slot_epoch[q]++; // deferred particles of earlier passes into these accumulators are void
  return 0;
}

// After a write into slots [lo, lo + n) on the compute stream: a reduce of them waits for `done`, or for the whole compute stream
// when `done` is nullptr; the staging pool the write read may be overwritten behind it.
static int slots_written(slicer_handle *h, int lo, int n, cudaEvent_t done)
{
  for (int q = lo; q < lo + n; q++)
    h->slot_pass_ev[q] = done;
  CU(cudaEventRecord(h->ev_buf_done[h->cur_buf], h->compute));
  return 0;
}

static int run_pass(slicer_handle *h, const slicer_plane_desc *planes, int nplanes, bool accumulate, int first_slot = 0)
{
  if (!h || !planes)
    return fail("slicer_deposit: null argument");
  if (set_device(h))
    return 1;
  if (first_slot < 0 || nplanes < 1 || first_slot + nplanes > h->cfg.max_planes)
    return fail("slicer_deposit: slots %d..%d outside 0..%d (max_planes)", first_slot, first_slot + nplanes - 1, h->cfg.max_planes - 1);
  PassParams P;
  if (build_pass(h, planes, nplanes, &P, first_slot) || staging_fence(h))
    return 1;
  // A new set of planes takes the other bank when that bank is settled (a caller that alternates between two slot ranges and
  // settles or reduces one range behind the next pass finds it so every time), or when it zeroes slots the current bank holds
  // (the other bank is then settled first: its passes are two sets back).  A set into other slots, submitted while both banks
  // hold passes, joins the current bank: several sets deposited before any is settled (the first passes of several light cones
  // over one sub-file: A, B, C non-accumulating, then A, B, C accumulating) so never make the host wait for a running pass.
  // Every pass sits in one bank with the epochs of its slots; resolve_deferred settles each bank that holds a pass into the
  // slots it is asked for.
  if (!accumulate)
  {
    uint64_t mine = 0;
    for (int q = first_slot; q < first_slot + nplanes; q++)
      mine |= (uint64_t)1 << q;
    if (h->defer.bank[h->defer.cur ^ 1].passes.empty() || (h->defer.bank[h->defer.cur].slot_mask & mine))
    {
      h->defer.cur ^= 1;
      if (resolve_bank(h, h->defer.cur))
        return 1;
    }
  }
  if (h->defer.bank[h->defer.cur].passes.size() >= 4096 && resolve_bank(h, h->defer.cur))
    return 1;
  if (claim_slots(h, first_slot, nplanes, accumulate))
    return 1;
  slicer_handle::DeferBank &B = h->defer.bank[h->defer.cur];
  DeferDev F;
  F.buf = B.buf;
  F.count = B.count;
  F.cap = h->defer.cap;
  F.pass = (unsigned)B.passes.size();
  { // (any path can defer pairs: the lean projection and the general chain's guard)
    slicer_handle::SavedPass sp;
    sp.P = P;
    for (int k = 0; k < P.nplanes; k++)
    {
      sp.epoch[k] = h->slot_epoch[P.pl[k].slot];
      B.slot_mask |= (uint64_t)1 << P.pl[k].slot;
    }
    B.passes.push_back(sp);
  }
  int kernel = h->cfg.kernel;
  if (kernel == SLICER_KERNEL_AUTO)
    kernel = SLICER_KERNEL_PIPELINED;
  if (h->pass_head - h->pass_tail == PASS_RING && resolve_passes(h, 1))
    return 1;
  cudaEvent_t e0 = h->pass_ev[2 * (h->pass_head % PASS_RING)], e1 = h->pass_ev[2 * (h->pass_head % PASS_RING) + 1];
  CU(cudaEventRecord(e0, h->compute));
  for (size_t si = 0; si < h->segs.size(); si++)
  {
    SegmentDev D;
    fill_segment(h, h->segs[si], &D);
    if (D.n == 0)
      continue;
    if (D.mass && D.n >> 32) // (the kernels carry a particle's index to its mass in 32 bits)
      return fail("slicer_deposit: a segment with per-particle masses holds %llu particles; stage it in batches of fewer than 2^32", D.n);
    if (kernel == SLICER_KERNEL_PIPELINED)
    {
      const int ub = use_binned(h, P, D);
      if (ub == 1)
      {
        if (binned_pass(h, P, D, F))
          return 1;
      }
      else if (maps_ready(h) || pipelined_launch(&h->pipe, h->cfg.mas, P, D, F, h->compute))
        return fail("pipelined launch failed: %s", cudaGetErrorString(cudaGetLastError()));
    }
    else
    {
      size_t want = (D.n + 255) / 256;
      size_t cap = (size_t)h->sm_count * 8;
      int blocks = (int)(want < cap ? want : cap);
      if (maps_ready(h))
        return 1;
      if (h->cfg.mas == SLICER_MAS_NGP)
        deposit_simple_kernel<SLICER_MAS_NGP><<<blocks, 256, 0, h->compute>>>(P, D, F);
      else
        deposit_simple_kernel<SLICER_MAS_TSC><<<blocks, 256, 0, h->compute>>>(P, D, F);
      CU(cudaGetLastError());
    }
    h->stats.launches++;
    h->stats.deposit_launches++;
    h->stats.particles_streamed += D.n;
  }
  if (maps_ready(h)) // (a pass without particles still leaves zeroed planes behind it in stream order)
    return 1;
  CU(cudaEventRecord(e1, h->compute));
  // the bank's deferred list as of now, for resolve_bank
  CU(cudaMemcpyAsync(B.host_count, B.count, sizeof(unsigned), cudaMemcpyDeviceToHost, h->compute));
  CU(cudaMemcpyAsync(B.host, B.buf, (size_t)DEFER_HEAD * sizeof(DeferEntry), cudaMemcpyDeviceToHost, h->compute));
  CU(cudaEventRecord(B.ev_done, h->compute));
  if (slots_written(h, first_slot, nplanes, e1)) // (a recycled ring entry stands for a later pass: waiting for it is still sufficient)
    return 1;
  h->pass_head++;
  return 0;
}

extern "C" int slicer_selftest_arith(slicer_handle *h, unsigned long long n, unsigned long long seed, unsigned long long out[3])
{
  if (!h || !out)
    return fail("null argument");
  if (set_device(h))
    return 1;
  unsigned long long *d = (unsigned long long *)h->d_out; // npix_max^2 floats of scratch
  if (h->npix2max * sizeof(float) < 3 * sizeof(unsigned long long))
    return fail("slicer_selftest_arith needs npix_max >= 3");
  CU(cudaStreamSynchronize(h->compute));
  CU(cudaMemset(d, 0, 3 * sizeof(unsigned long long)));
  selftest_fdiv_kernel<<<h->sm_count * 8, 256, 0, h->compute>>>(n, seed, d);
  CU(cudaGetLastError());
  CU(cudaStreamSynchronize(h->compute));
  CU(cudaMemcpy(out, d, 3 * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
  return 0;
}

extern "C" int slicer_deposit(slicer_handle *h, const slicer_plane_desc *planes, int nplanes)
{
  return run_pass(h, planes, nplanes, false);
}

extern "C" int slicer_deposit_accumulate(slicer_handle *h, const slicer_plane_desc *planes, int nplanes)
{
  return run_pass(h, planes, nplanes, true);
}

extern "C" int slicer_deposit_slots(slicer_handle *h, const slicer_plane_desc *planes, int nplanes, int first_slot, int accumulate)
{
  return run_pass(h, planes, nplanes, accumulate != 0, first_slot);
}

// ------------------------------------------------------------------------------------------------------------
// Part. Degradation
// ------------------------------------------------------------------------------------------------------------
static int degrade_prepare(slicer_handle *h, const slicer_plane_desc *planes, int nplanes, PassParams *P, size_t *total)
{
  if (!h || !planes)
    return fail("null argument");
  if (set_device(h) || build_pass(h, planes, nplanes, P))
    return 1;
  for (int q = 0; q < nplanes; q++)
    if ((2 * planes[q].nrepperp + 1) * (2 * planes[q].nrepperp + 1) > 255)
      return fail("Part. Degradation supports nrepperp <= 7");
  size_t n = 0;
  for (size_t i = 0; i < h->segs.size(); i++)
    n += h->segs[i].n;
  *total = n;
  return 0;
}

// one degrade_kernel launch per resident segment with particles; G.seg_base: the segment's first particle in the batch
template <int MODE>
static int degrade_launch(slicer_handle *h, const PassParams &P, degrade::Dev G)
{
  G.seg_base = 0;
  for (size_t si = 0; si < h->segs.size(); si++)
  {
    SegmentDev D;
    fill_segment(h, h->segs[si], &D);
    if (D.n)
    {
      const size_t want = (D.n + 255) / 256, cap = (size_t)h->sm_count * 16;
      const int blocks = (int)(want < cap ? want : cap);
      if (h->cfg.mas == SLICER_MAS_NGP)
        degrade::degrade_kernel<SLICER_MAS_NGP, MODE><<<blocks, 256, 0, h->compute>>>(P, D, G);
      else
        degrade::degrade_kernel<SLICER_MAS_TSC, MODE><<<blocks, 256, 0, h->compute>>>(P, D, G);
      CU(cudaGetLastError());
      h->stats.launches++;
      if (MODE == degrade::DEPOSIT)
        h->stats.particles_streamed += D.n;
    }
    G.seg_base += D.n;
  }
  return 0;
}

extern "C" int slicer_count_accepted(slicer_handle *h, const slicer_plane_desc *planes, int nplanes, long long *counts)
{
  PassParams P;
  size_t total = 0;
  if (degrade_prepare(h, planes, nplanes, &P, &total) || staging_fence(h))
    return 1;
  if (!counts)
    return fail("slicer_count_accepted: null output");
  for (int i = 0; i < nplanes * SLICER_NTYPES; i++)
    counts[i] = 0;
  h->deg.valid = false;
  if (total == 0)
  {
    for (int q = 0; q < nplanes; q++)
      h->deg.plane_total[q] = 0;
    h->deg.nplanes = nplanes;
    h->deg.stride = 0;
    h->deg.valid = true;
    return 0;
  }
  if (h->deg.stride < total || h->deg.nplanes < nplanes)
  {
    CU(cudaStreamSynchronize(h->compute));
    cudaFree(h->deg.cnt);
    cudaFree(h->deg.rank);
    cudaFree(h->deg.block_sums);
    h->device_bytes -= h->deg.bytes;
    h->deg.cnt = nullptr;
    h->deg.rank = nullptr;
    h->deg.block_sums = nullptr;
    const size_t stride = total + total / 8 + 1024;
    const size_t nblocks = (stride + 1 + degrade::SCAN_BLOCK * degrade::SCAN_PER - 1) / (degrade::SCAN_BLOCK * degrade::SCAN_PER);
    const int np = nplanes > h->deg.nplanes ? nplanes : h->deg.nplanes;
    const size_t before = h->device_bytes;
    const int rc = dev_alloc(h, &h->deg.cnt, (size_t)np * stride) || dev_alloc(h, &h->deg.rank, (size_t)np * (stride + 1)) ||
                   dev_alloc(h, &h->deg.block_sums, (size_t)np * nblocks);
    h->deg.bytes = h->device_bytes - before;
    if (rc)
      return 1;
    h->deg.stride = stride;
    h->deg.nblocks = nblocks;
    h->deg.nplanes = np;
  }
  const size_t stride = h->deg.stride;
  CU(cudaMemsetAsync(h->deg.cnt, 0, (size_t)nplanes * stride, h->compute));
  degrade::Dev G;
  memset(&G, 0, sizeof(G));
  G.cnt = h->deg.cnt;
  G.rank = h->deg.rank;
  G.stride = stride;
  if (degrade_launch<degrade::MARK>(h, P, G))
    return 1;
  std::vector<size_t> seg_start(1, 0); // first particle of each segment in the batch, then the total
  for (const Segment &sg : h->segs)
    seg_start.push_back(seg_start.back() + sg.n);
  const size_t nb = (total + 1 + degrade::SCAN_BLOCK * degrade::SCAN_PER - 1) / (degrade::SCAN_BLOCK * degrade::SCAN_PER);
  const dim3 grid((unsigned)nb, (unsigned)nplanes);
  degrade::scan_block_sums<<<grid, degrade::SCAN_BLOCK, 0, h->compute>>>(h->deg.cnt, stride, total, h->deg.block_sums, h->deg.nblocks);
  degrade::scan_of_block_sums<<<dim3(1, nplanes), 1024, 0, h->compute>>>(h->deg.block_sums, h->deg.nblocks);
  degrade::scan_finish<<<grid, degrade::SCAN_BLOCK, 0, h->compute>>>(h->deg.cnt, stride, total, h->deg.block_sums, h->deg.nblocks, h->deg.rank);
  CU(cudaGetLastError());
  h->stats.launches += 3;
  // accepted pairs per (plane, segment) = differences of the ranks at the segment boundaries
  std::vector<unsigned> edge((size_t)nplanes * seg_start.size());
  for (int q = 0; q < nplanes; q++)
    for (size_t k = 0; k < seg_start.size(); k++)
      CU(cudaMemcpyAsync(&edge[q * seg_start.size() + k], h->deg.rank + (size_t)q * (stride + 1) + seg_start[k], sizeof(unsigned),
                         cudaMemcpyDeviceToHost, h->compute));
  CU(cudaStreamSynchronize(h->compute));
  for (int q = 0; q < nplanes; q++)
  {
    for (size_t k = 0; k + 1 < seg_start.size(); k++)
      counts[q * SLICER_NTYPES + h->segs[k].type] += (long long)(edge[q * seg_start.size() + k + 1] - edge[q * seg_start.size() + k]);
    h->deg.plane_total[q] = edge[q * seg_start.size() + seg_start.size() - 1];
  }
  h->deg.valid = true;
  return 0;
}

// Writes accumulator slots [0, nplanes) like a pass, but leaves their slot_pass_ev empty: a reduce of them waits for the whole
// compute stream.
extern "C" int slicer_deposit_degraded(slicer_handle *h, const slicer_plane_desc *planes, int nplanes, int snopt,
                                       const unsigned char *const *keep, int accumulate)
{
  PassParams P;
  size_t total = 0;
  if (degrade_prepare(h, planes, nplanes, &P, &total))
    return 1;
  if (snopt < 1 || snopt > 30)
    return fail("slicer_deposit_degraded: snopt %d outside 1..30", snopt);
  if (!h->deg.valid || h->deg.nplanes < nplanes)
    return fail("slicer_deposit_degraded: call slicer_count_accepted for this batch and these planes first");
  degrade::Dev G;
  memset(&G, 0, sizeof(G));
  size_t need = 0;
  for (int q = 0; q < nplanes; q++)
  {
    G.keep_off[q] = need;
    need += h->deg.plane_total[q];
    if (h->deg.plane_total[q] && (!keep || !keep[q]))
      return fail("slicer_deposit_degraded: keep table of plane %d is missing", q);
  }
  if (staging_fence(h) || claim_slots(h, 0, nplanes, accumulate != 0))
    return 1;
  if (total == 0)
    return maps_ready(h) || slots_written(h, 0, nplanes, nullptr);
  if (need > h->deg.keep_cap)
  {
    CU(cudaStreamSynchronize(h->compute));
    cudaFree(h->deg.keep);
    h->device_bytes -= h->deg.keep_cap;
    h->deg.keep = nullptr;
    h->deg.keep_cap = 0;
    if (dev_alloc(h, &h->deg.keep, need + need / 4 + 4096))
      return 1;
    h->deg.keep_cap = need + need / 4 + 4096;
  }
  for (int q = 0; q < nplanes; q++)
    if (h->deg.plane_total[q])
      CU(cudaMemcpyAsync(h->deg.keep + G.keep_off[q], keep[q], h->deg.plane_total[q], cudaMemcpyHostToDevice, h->compute));
  G.cnt = h->deg.cnt;
  G.rank = h->deg.rank;
  G.keep = h->deg.keep;
  G.stride = h->deg.stride;
  G.snopt = snopt;
  if (maps_ready(h) || degrade_launch<degrade::DEPOSIT>(h, P, G) || slots_written(h, 0, nplanes, nullptr))
    return 1;
  CU(cudaStreamSynchronize(h->compute)); // the caller's keep tables may be freed on return
  return 0;
}

extern "C" int slicer_synchronize(slicer_handle *h)
{
  if (!h)
    return fail("null handle");
  if (set_device(h))
    return 1;
  CU(cudaStreamSynchronize(h->copy));
  if (resolve_deferred(h))
    return 1;
  CU(cudaStreamSynchronize(h->compute));
  CU(cudaStreamSynchronize(h->settle));
  CU(cudaStreamSynchronize(h->comm_stream));
  return 0;
}

extern "C" int slicer_settle_slots(slicer_handle *h, int first_slot, int nplanes)
{
  if (!h)
    return fail("null handle");
  if (nplanes < 1 || first_slot < 0 || first_slot + nplanes > h->cfg.max_planes)
    return fail("slicer_settle_slots: slots %d..%d outside 0..%d", first_slot, first_slot + nplanes - 1, h->cfg.max_planes - 1);
  if (set_device(h))
    return 1;
  return resolve_deferred(h, first_slot, nplanes);
}

extern "C" int slicer_wait_staging(slicer_handle *h)
{
  if (!h)
    return fail("null handle");
  if (set_device(h))
    return 1;
  CU(cudaStreamSynchronize(h->copy));
  return 0;
}

// ------------------------------------------------------------------------------------------------------------
// read-out
// ------------------------------------------------------------------------------------------------------------
static int check_plane(slicer_handle *h, int plane, int type)
{
  if (!h)
    return fail("null handle");
  if (plane < 0 || plane >= h->cfg.max_planes)
    return fail("plane %d outside 0..%d", plane, h->cfg.max_planes - 1);
  if (h->plane_npix[plane] <= 0)
    return fail("plane %d has not been deposited", plane);
  if (type < -1 || type >= SLICER_NTYPES)
    return fail("type %d outside -1..5", type);
  if (type >= 0 && !h->cfg.per_type_maps)
    return fail("per-type maps were not requested (slicer_config.per_type_maps)");
  return set_device(h);
}

extern "C" int slicer_fetch(slicer_handle *h, int plane, int type, float *out_map, long long counts[SLICER_NTYPES],
                            long long ingrid[SLICER_NTYPES])
{
  if (check_plane(h, plane, type) || resolve_deferred(h, plane, 1) || wait_settled(h, false) || wait_slot_reduces(h, plane, 1))
    return 1;
  const size_t npix2 = (size_t)h->plane_npix[plane] * h->plane_npix[plane];
  const unsigned long long *base = h->d_acc + (size_t)plane * h->ntypes_alloc * h->npix2max;
  if (out_map)
  {
    const unsigned long long *src = type >= 0 ? base + (size_t)type * h->npix2max : base;
    const int nt = type >= 0 ? 1 : h->ntypes_alloc;
    const int blocks = (int)((npix2 + 255) / 256 < (size_t)h->sm_count * 8 ? (npix2 + 255) / 256 : (size_t)h->sm_count * 8);
    finalize_map_kernel<<<blocks, 256, 0, h->compute>>>(src, h->npix2max, nt, npix2, ldexp(1.0, -h->frac_bits), h->d_out, h->d_ovf);
    CU(cudaGetLastError());
    h->stats.launches++;
    CU(cudaMemcpyAsync(out_map, h->d_out, npix2 * sizeof(float), cudaMemcpyDeviceToHost, h->compute));
  }
  unsigned ovf = 0;
  CU(cudaMemcpyAsync(&ovf, h->d_ovf, sizeof(unsigned), cudaMemcpyDeviceToHost, h->compute));
  unsigned long long c[SLICER_NTYPES * 2];
  CU(cudaMemcpyAsync(c, h->d_counts + (size_t)plane * SLICER_NTYPES * 2, sizeof(c), cudaMemcpyDeviceToHost, h->compute));
  CU(cudaStreamSynchronize(h->compute));
  for (int t = 0; t < SLICER_NTYPES; t++)
  {
    if (counts)
      counts[t] = (long long)c[2 * t];
    if (ingrid)
      ingrid[t] = (long long)c[2 * t + 1];
  }
  if (ovf)
  {
    CU(cudaMemsetAsync(h->d_ovf, 0, sizeof(unsigned), h->compute));
    return fail("plane %d: a fixed-point accumulator exceeded 2^63 (more than %.3g mass units in one pixel at %d fraction bits); "
                "create the handle with a smaller slicer_config.frac_bits", plane, ldexp(1.0, 63 - h->frac_bits), h->frac_bits);
  }
  return 0;
}

extern "C" int slicer_fetch_fixed(slicer_handle *h, int plane, int type, long long *out)
{
  if (check_plane(h, plane, type) || resolve_deferred(h, plane, 1) || wait_settled(h, false) || wait_slot_reduces(h, plane, 1))
    return 1;
  if (!out)
    return fail("slicer_fetch_fixed: null output");
  const size_t npix2 = (size_t)h->plane_npix[plane] * h->plane_npix[plane];
  const unsigned long long *base = h->d_acc + (size_t)plane * h->ntypes_alloc * h->npix2max;
  const unsigned long long *src = type >= 0 ? base + (size_t)type * h->npix2max : base;
  const int nt = type >= 0 ? 1 : h->ntypes_alloc;
  const int blocks = (int)((npix2 + 255) / 256 < (size_t)h->sm_count * 8 ? (npix2 + 255) / 256 : (size_t)h->sm_count * 8);
  sum_types_kernel<<<blocks, 256, 0, h->compute>>>(src, h->npix2max, nt, npix2, h->d_sum, h->d_ovf);
  CU(cudaGetLastError());
  h->stats.launches++;
  CU(cudaMemcpyAsync(out, h->d_sum, npix2 * sizeof(long long), cudaMemcpyDeviceToHost, h->compute));
  unsigned ovf = 0;
  CU(cudaMemcpyAsync(&ovf, h->d_ovf, sizeof(unsigned), cudaMemcpyDeviceToHost, h->compute));
  CU(cudaStreamSynchronize(h->compute));
  if (ovf)
  {
    CU(cudaMemsetAsync(h->d_ovf, 0, sizeof(unsigned), h->compute));
    return fail("plane %d: a fixed-point accumulator exceeded 2^63 (more than %.3g mass units in one pixel at %d fraction bits); "
                "create the handle with a smaller slicer_config.frac_bits", plane, ldexp(1.0, 63 - h->frac_bits), h->frac_bits);
  }
  return 0;
}

extern "C" int slicer_get_stats(slicer_handle *h, slicer_stats *out)
{
  if (!h || !out)
    return fail("null argument");
  if (set_device(h))
    return 1;
  if (resolve_passes(h, 0))
    return 1;
  size_t res = 0;
  for (size_t i = 0; i < h->segs.size(); i++)
    res += h->segs[i].n;
  h->stats.resident_particles = res;
  h->stats.device_bytes = h->device_bytes;
  h->stats.sm_count = h->sm_count;
  *out = h->stats;
  return 0;
}

extern "C" int slicer_reset_stats(slicer_handle *h)
{
  if (!h)
    return fail("null handle");
  if (set_device(h) || resolve_passes(h, 0))
    return 1;
  h->stats.deposit_ms_sum = 0;
  h->stats.deposit_passes = 0;
  h->stats.deposit_launches = 0;
  h->stats.launches = 0;
  h->stats.particles_streamed = 0;
  return 0;
}

extern "C" int slicer_timer_begin(slicer_handle *h)
{
  if (!h)
    return fail("null handle");
  if (set_device(h))
    return 1;
  CU(cudaEventRecord(h->ev_t0, h->compute));
  return 0;
}

extern "C" int slicer_timer_end(slicer_handle *h, double *ms)
{
  if (!h || !ms)
    return fail("null argument");
  if (set_device(h))
    return 1;
  CU(cudaStreamSynchronize(h->copy));
  CU(cudaEventRecord(h->ev_t1, h->compute));
  CU(cudaEventSynchronize(h->ev_t1));
  float f = 0;
  CU(cudaEventElapsedTime(&f, h->ev_t0, h->ev_t1));
  *ms = f;
  return 0;
}

// ------------------------------------------------------------------------------------------------------------
// multi-GPU: ncclReduce(int64, sum) of the plane accumulators — replaces slicer-v2.cpp:214-217
// ------------------------------------------------------------------------------------------------------------
extern "C" int slicer_comm_unique_id(char id[128])
{
  if (load_nccl())
    return 1;
  ncclUniqueId u;
  NC(g_nccl.GetUniqueId(&u));
  static_assert(sizeof(ncclUniqueId) == 128, "ncclUniqueId is 128 bytes");
  memcpy(id, &u, 128);
  return 0;
}

extern "C" int slicer_comm_init_rank(slicer_handle *h, const char id[128], int nranks, int rank)
{
  if (!h)
    return fail("null handle");
  if (load_nccl() || set_device(h))
    return 1;
  if (h->comm)
    return fail("communicator already initialised");
  ncclUniqueId u;
  memcpy(&u, id, 128);
  NC(g_nccl.CommInitRank(&h->comm, nranks, u, rank));
  h->nranks = nranks;
  h->rank = rank;
  return 0;
}

extern "C" int slicer_comm_init_all(slicer_handle **handles, int n)
{
  if (!handles || n < 1)
    return fail("slicer_comm_init_all: bad arguments");
  if (load_nccl())
    return 1;
  std::vector<int> devs(n);
  std::vector<ncclComm_t> comms(n);
  for (int i = 0; i < n; i++)
  {
    if (!handles[i] || handles[i]->comm)
      return fail("slicer_comm_init_all: handle %d null or already in a communicator", i);
    devs[i] = handles[i]->cfg.device;
  }
  NC(g_nccl.CommInitAll(comms.data(), n, devs.data()));
  for (int i = 0; i < n; i++)
  {
    handles[i]->comm = comms[i];
    handles[i]->nranks = n;
    handles[i]->rank = i;
  }
  return 0;
}

// one ncclReduce per (plane, type) accumulator over the npix^2 cells that plane uses (not the npix_max^2 it is allocated with),
// on the handle's communication stream: passes into OTHER accumulator slots keep running on the compute stream meanwhile
static int enqueue_reduce(slicer_handle *h, int first_slot, int nplanes, int root)
{
  for (int q = first_slot; q < first_slot + nplanes; q++)
  {
    const size_t npix2 = h->plane_npix[q] > 0 ? (size_t)h->plane_npix[q] * h->plane_npix[q] : h->npix2max;
    for (int t = 0; t < h->ntypes_alloc; t++)
    {
      unsigned long long *a = h->d_acc + ((size_t)q * h->ntypes_alloc + t) * h->npix2max;
      NC(g_nccl.Reduce(a, a, npix2, ncclInt64, ncclSum, root, h->comm, h->comm_stream));
    }
  }
  unsigned long long *c = h->d_counts + (size_t)first_slot * SLICER_NTYPES * 2;
  NC(g_nccl.Reduce(c, c, (size_t)nplanes * SLICER_NTYPES * 2, ncclUint64, ncclSum, root, h->comm, h->comm_stream));
  return 0;
}

// order the reduce after the passes submitted so far, and everything that touches these slots later after the reduce
static int reduce_fence_before(slicer_handle *h, int first_slot, int nplanes)
{
  if (wait_slot_reduces(h, first_slot, nplanes)) // an earlier reduce of the same slots (same stream anyway)
    return 1;
  // after the last pass into each of these slots (not after passes into other slots submitted since) and after the deposits
  // of the pairs libm settled
  bool all = false;
  for (int q = first_slot; q < first_slot + nplanes; q++)
    all = all || !h->slot_pass_ev[q];
  if (all)
  {
    CU(cudaEventRecord(h->ev_pass_done, h->compute));
    CU(cudaStreamWaitEvent(h->comm_stream, h->ev_pass_done, 0));
  }
  else
  {
    cudaEvent_t seen = nullptr;
    for (int q = first_slot; q < first_slot + nplanes; q++)
      if (h->slot_pass_ev[q] != seen)
      {
        seen = h->slot_pass_ev[q];
        CU(cudaStreamWaitEvent(h->comm_stream, seen, 0));
      }
  }
  return wait_settled(h, true);
}
static int reduce_fence_after(slicer_handle *h, int first_slot, int nplanes)
{
  for (int q = first_slot; q < first_slot + nplanes; q++)
  {
    CU(cudaEventRecord(h->ev_slot[q], h->comm_stream));
    h->slot_reducing[q] = true;
  }
  return 0;
}

extern "C" int slicer_reduce_slots(slicer_handle *h, int first_slot, int nplanes, int root)
{
  if (!h)
    return fail("null handle");
  if (nplanes < 1 || first_slot < 0 || first_slot + nplanes > h->cfg.max_planes)
    return fail("slicer_reduce: slots %d..%d outside 0..%d", first_slot, first_slot + nplanes - 1, h->cfg.max_planes - 1);
  if (set_device(h) || resolve_deferred(h, first_slot, nplanes))
    return 1;
  if (!h->comm || h->nranks == 1)
    return 0;
  if (reduce_fence_before(h, first_slot, nplanes))
    return 1;
  NC(g_nccl.GroupStart());
  const int rc = enqueue_reduce(h, first_slot, nplanes, root);
  const ncclResult_t ge = g_nccl.GroupEnd(); // always closes the group, also when a reduce could not be enqueued
  if (rc)
    return rc;
  if (ge != ncclSuccess)
    return fail("ncclGroupEnd failed: %s", g_nccl.GetErrorString(ge));
  return reduce_fence_after(h, first_slot, nplanes);
}

extern "C" int slicer_reduce(slicer_handle *h, int nplanes, int root) { return slicer_reduce_slots(h, 0, nplanes, root); }

extern "C" int slicer_reduce_all_slots(slicer_handle **handles, int n, int first_slot, int nplanes, int root)
{
  if (!handles || n < 1)
    return fail("slicer_reduce_all: bad arguments");
  for (int i = 0; i < n; i++)
  {
    if (!handles[i])
      return fail("slicer_reduce_all: null handle");
    if (nplanes < 1 || first_slot < 0 || first_slot + nplanes > handles[i]->cfg.max_planes)
      return fail("slicer_reduce_all: slots %d..%d outside 0..%d", first_slot, first_slot + nplanes - 1, handles[i]->cfg.max_planes - 1);
    if (set_device(handles[i]) || resolve_deferred(handles[i], first_slot, nplanes))
      return 1;
  }
  if (n == 1)
    return 0;
  if (load_nccl())
    return 1;
  for (int i = 0; i < n; i++)
    if (set_device(handles[i]) || reduce_fence_before(handles[i], first_slot, nplanes))
      return 1;
  NC(g_nccl.GroupStart());
  int rc = 0;
  for (int i = 0; i < n && !rc; i++)
  {
    if (cudaSetDevice(handles[i]->cfg.device) != cudaSuccess)
      rc = fail("cudaSetDevice failed");
    else
      rc = enqueue_reduce(handles[i], first_slot, nplanes, root);
  }
  const ncclResult_t ge = g_nccl.GroupEnd();
  if (rc)
    return rc;
  if (ge != ncclSuccess)
    return fail("ncclGroupEnd failed: %s", g_nccl.GetErrorString(ge));
  for (int i = 0; i < n; i++)
    if (set_device(handles[i]) || reduce_fence_after(handles[i], first_slot, nplanes))
      return 1;
  return 0;
}

extern "C" int slicer_reduce_all(slicer_handle **handles, int n, int nplanes, int root)
{
  return slicer_reduce_all_slots(handles, n, 0, nplanes, root);
}
