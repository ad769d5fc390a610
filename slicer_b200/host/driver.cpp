// driver.cpp — createDensityMaps on the GPU and the plane driver of main() (slicer-v2.cpp:130-230), restructured:
// the reference walks the PLANES and re-reads + re-transforms a whole snapshot for each one (:138-207); here the
// loop is over SNAPSHOTS, every sub-file is read once into page-locked memory, copied once, and one CUDA pass
// deposits it into all the planes that use the snapshot.  Sub-files are dealt round-robin to the GPUs of the box
// (the reference deals them to MPI ranks, :162-175) and the planes are summed with ncclReduce instead of MPI_Reduce.
#include "slicer_host.h"

#include <atomic>
#include <chrono>
#include <cmath>
#include <cstring>
#include <filesystem>
#include <fstream>
#include <functional>
#include <iostream>
#include <map>
#include <memory>
#include <sstream>
#include <thread>

namespace slicer
{

// wall-clock phase totals of the last runLightCones (seconds): printed when SLICER_B200_TIMING is set
static double t_read = 0, t_submit = 0, t_fetch = 0, t_write = 0, t_engine = 0, t_gpu = 0; // t_gpu: device time of the passes
static double now_s() { return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count(); }

struct Engine
{
  std::vector<int> devices;
  std::vector<slicer_handle *> h;
  std::vector<SubFile> bufs; // two page-locked sub-file buffers per GPU
  std::vector<int> used;     // sub-files staged on each GPU since begin
  int npix_max = 0, mas = SLICER_MAS_TSC, deposit_mode = SLICER_DEPOSIT_AUTO;
  bool per_type = false;
  size_t capacity = 0;
  int max_planes = SLICER_MAX_PLANES; // accumulator slots per GPU
  // > 0: the slots are sized to free device memory each time the handles are made, want_slots at most, need_slots at least
  int want_slots = 0, need_slots = 0;
  bool comm = false;
};

// device time of the passes the handles ran (summed over the GPUs), before they are destroyed: SLICER_B200_TIMING only
static void add_gpu_time(Engine *e)
{
  if (!getenv("SLICER_B200_TIMING"))
    return;
  for (auto *hh : e->h)
  {
    slicer_stats st;
    if (hh && !slicer_get_stats(hh, &st))
      t_gpu += st.deposit_ms_sum / 1e3;
  }
}

// Accumulator slots per GPU for `want` planes per snapshot read: no more than the free device memory of the smallest GPU holds
// beside what else a handle allocates, and at least `need`.  Besides its accumulators (types x npix^2 x 8 B per slot) a handle
// owns two staging pools of 12 B positions + 4 B masses per particle, the binned deposit's records (26 B per particle of a slice,
// at most the particle capacity), two npix^2 read-out buffers (12 B per pixel) and the deferred-pair banks (2 x 24 B x 2^19 per
// 16 slots); 512 MiB cover the banks, the kernels' scratch and the context's own allocations.  Checked every time the handles
// are made, so a rebuild with a larger particle capacity (ensure_capacity) takes fewer slots rather than failing to allocate.
static int choose_slots(const std::vector<int> &devices, int want, int need, int npix_max, bool per_type, size_t capacity, int &slots)
{
  const size_t per_slot = (size_t)(per_type ? 6 : 1) * npix_max * npix_max * 8;
  const size_t reserve = capacity * (2 * 16 + 26) + (size_t)npix_max * npix_max * 12 + ((size_t)512 << 20);
  slots = want;
  for (int d : devices)
  {
    size_t free_b = 0, total_b = 0;
    if (slicer_device_memory(d, &free_b, &total_b))
    {
      std::cerr << "slicer_device_memory: " << slicer_last_error() << std::endl;
      return 1;
    }
    const size_t fit = free_b > reserve ? (free_b - reserve) / per_slot : 0;
    if ((int)std::min(fit, (size_t)want) < need)
    {
      std::cerr << "GPU " << d << ": " << free_b / double(1 << 30) << " GiB free hold " << fit << " plane accumulators of " << npix_max << "^2"
                << (per_type ? " x 6 particle types" : "") << " (" << per_slot / double(1 << 20) << " MiB each) beside the particle buffers of "
                << capacity << " particles; at least " << need << " are needed" << std::endl;
      return 1;
    }
    slots = (int)std::min((size_t)slots, fit);
  }
  return 0;
}

static int make_handles(Engine *e)
{
  add_gpu_time(e);
  for (auto *hh : e->h)
    slicer_destroy(hh);
  e->h.assign(e->devices.size(), nullptr);
  e->comm = false;
  if (e->want_slots > 0 && choose_slots(e->devices, e->want_slots, e->need_slots, e->npix_max, e->per_type, e->capacity, e->max_planes))
    return 1;
  // one thread per GPU: creating a CUDA context, loading the kernels and allocating the pools takes ~2 s per device, serially
  // that was most of an 8-GPU run's wall clock
  std::vector<std::string> errs(e->devices.size());
  auto make_one = [&](size_t g) {
    slicer_config cfg;
    memset(&cfg, 0, sizeof(cfg));
    cfg.device = e->devices[g];
    cfg.mas = e->mas;
    cfg.max_m = MAX_M;
    cfg.max_planes = e->max_planes;
    cfg.npix_max = e->npix_max;
    cfg.per_type_maps = e->per_type;
    cfg.particle_capacity = e->capacity;
    cfg.mass_capacity = e->capacity;
    cfg.kernel = SLICER_KERNEL_AUTO;
    cfg.staging_buffers = 2;
    cfg.deposit_mode = e->deposit_mode;
    if (slicer_create(&cfg, &e->h[g]))
      errs[g] = slicer_last_error(); // (thread-local: read it on the thread that made the call)
  };
  if (e->devices.size() == 1)
    make_one(0);
  else
  {
    std::vector<std::thread> th;
    for (size_t g = 0; g < e->devices.size(); g++)
      th.emplace_back(make_one, g);
    for (auto &t : th)
      t.join();
  }
  for (size_t g = 0; g < e->devices.size(); g++)
    if (!e->h[g])
    {
      std::cerr << "slicer_create failed on GPU " << e->devices[g] << ": " << errs[g] << std::endl;
      return 1;
    }
  if (e->h.size() > 1)
  {
    if (slicer_comm_init_all(e->h.data(), (int)e->h.size()))
    {
      std::cerr << "NCCL communicator: " << slicer_last_error() << std::endl;
      return 1;
    }
    e->comm = true;
  }
  return 0;
}

static Engine *engine_new(const std::vector<int> &devices, int npix_max, int mas, bool per_type_maps, size_t particle_capacity, int deposit_mode,
                          int max_planes, int want_slots, int need_slots)
{
  Engine *e = new Engine;
  e->devices = devices;
  e->max_planes = std::min(std::max(max_planes, 1), (int)SLICER_MAX_SLOTS);
  e->want_slots = want_slots;
  e->need_slots = need_slots;
  e->npix_max = npix_max;
  e->mas = mas;
  e->per_type = per_type_maps;
  e->capacity = particle_capacity;
  e->deposit_mode = deposit_mode;
  e->bufs = std::vector<SubFile>(2 * devices.size());
  e->used.assign(devices.size(), 0);
  if (make_handles(e))
  {
    engineDestroy(e);
    return nullptr;
  }
  return e;
}

Engine *engineCreate(const std::vector<int> &devices, int npix_max, int mas, bool per_type_maps, size_t particle_capacity, int deposit_mode,
                     int max_planes)
{
  return engine_new(devices, npix_max, mas, per_type_maps, particle_capacity, deposit_mode, max_planes, 0, 0);
}

void engineDestroy(Engine *e)
{
  if (!e)
    return;
  add_gpu_time(e);
  for (auto *hh : e->h)
    slicer_destroy(hh);
  delete e;
}

int engineGpuCount(const Engine *e) { return (int)e->h.size(); }

static slicer_plane_desc make_desc(const Lens &lens, const Random &random, int isnap, double rcase, double fovradiants, int npix)
{
  slicer_plane_desc d;
  memset(&d, 0, sizeof(d));
  d.sgn[0] = random.sgnX[isnap];
  d.sgn[1] = random.sgnY[isnap];
  d.sgn[2] = random.sgnZ[isnap];
  d.face = random.face[isnap];
  d.centre[0] = random.x0[isnap];
  d.centre[1] = random.y0[isnap];
  d.centre[2] = random.z0[isnap];
  d.rcase = (float)rcase; // createDensityMaps takes a double, readPos a float (densitymaps.h:162, gadget2io.h:123)
  d.ld = lens.ld[isnap];
  d.ld2 = lens.ld2[isnap];
  d.nrepperp = lens.nrepperp.empty() ? 0 : lens.nrepperp[isnap];
  d.fovradiants = fovradiants;
  d.npix = npix;
  return d;
}

static int fail_capi(const char *what)
{
  std::cerr << what << ": " << slicer_last_error() << std::endl;
  return 1;
}

// Stage every particle type of a sub-file that is already in `buf` (types in order: the order mapParticles walks them).
static int stage_subfile(slicer_handle *h, const SubFile &buf, bool hydro)
{
  size_t off = 0;
  for (int t = 0; t < 6; t++)
  {
    const size_t nt = (size_t)buf.header.npart[t];
    if (nt)
    {
      const bool pm = hydro && buf.header.massarr[t] == 0;
      if (slicer_stage_particles(h, t, buf.pos + 3 * off, SLICER_LAYOUT_AOS, pm ? buf.mass + off : nullptr, nt))
        return fail_capi("slicer_stage_particles");
    }
    off += nt;
  }
  return 0;
}

// The device staging pools must hold the largest sub-file of the snapshot (sub-files of one snapshot differ by tens of per cent
// with domain decomposition or gas).  The sub-file headers are scanned first (256 bytes each); if one needs more room than the
// handles have, the handles are rebuilt with that capacity before any work of this snapshot is queued.
static int ensure_capacity(Engine *e, const std::string &File, unsigned ffmin, unsigned ffmax)
{
  size_t largest = 0;
  for (unsigned ff = ffmin; ff < ffmax; ff++)
  {
    Header hd;
    if (readHeader(File + "." + std::to_string(ff), hd))
      return 1;
    size_t n = 0;
    for (int t = 0; t < 6; t++)
      n += (size_t)(hd.npart[t] > 0 ? hd.npart[t] : 0);
    largest = std::max(largest, n);
  }
  if (largest <= e->capacity)
    return 0;
  for (auto *hh : e->h)
    if (hh && slicer_synchronize(hh))
      return fail_capi("slicer_synchronize");
  e->capacity = largest + largest / 8 + 4096;
  return make_handles(e);
}

// Passes of one call: consecutive jobs [first, first + n), into accumulator slots first - (first job of the group) ...
struct PassSpan
{
  int first, n;
};

static bool same_xform(const slicer_plane_desc &a, const slicer_plane_desc &b)
{ // build_pass' test: planes with the same randomisation share one box transform in a pass
  return memcmp(a.sgn, b.sgn, sizeof(a.sgn)) == 0 && a.face == b.face && a.centre[0] == b.centre[0] && a.centre[1] == b.centre[1] &&
         a.centre[2] == b.centre[2] && a.rcase == b.rcase;
}

static int count_xforms(const slicer_plane_desc *d, int n)
{
  int nx = 0;
  for (int i = 0; i < n; i++)
  {
    bool seen = false;
    for (int j = 0; j < i && !seen; j++)
      seen = same_xform(d[j], d[i]);
    nx += !seen;
  }
  return nx;
}

// Jobs -> passes of at most `limit` planes (SLICER_MAX_PLANES, or the engine's slots if it has fewer): a realisation's
// consecutive jobs stay in one pass (split only beyond `limit` planes or SLICER_MAX_XFORMS randomisations); whole realisations
// are added to a pass while both limits hold.  One realisation with at most 16 planes per snapshot and an engine with slots for
// them gives one pass, exactly as before several realisations were possible.
static std::vector<PassSpan> plan_passes(const std::vector<PlaneJob> &jobs, const std::vector<slicer_plane_desc> &descs, int limit)
{
  std::vector<PassSpan> units;
  for (int j = 0; j < (int)jobs.size(); j++)
  {
    PassSpan *u = units.empty() ? nullptr : &units.back();
    if (u && jobs[u->first].random == jobs[j].random && u->n < limit &&
        count_xforms(&descs[u->first], u->n + 1) <= SLICER_MAX_XFORMS)
      u->n++;
    else
      units.push_back({j, 1});
  }
  std::vector<PassSpan> passes;
  for (const PassSpan &u : units)
  {
    PassSpan *q = passes.empty() ? nullptr : &passes.back();
    if (q && q->n + u.n <= limit && count_xforms(&descs[q->first], q->n + u.n) <= SLICER_MAX_XFORMS)
      q->n += u.n;
    else
      passes.push_back(u);
  }
  return passes;
}

// Passes [pass, end) of a group, each into its slots: the first sub-file of a GPU zeroes them, the others add to them.
static int deposit_passes(slicer_handle *h, const std::vector<slicer_plane_desc> &descs, const PassSpan *pass, const PassSpan *end, bool accumulate)
{
  const int j0 = pass->first;
  for (; pass != end; pass++)
    if (slicer_deposit_slots(h, &descs[pass->first], pass->n, pass->first - j0, accumulate))
      return 1;
  return 0;
}

// Stages sub-files [ffmin, ffmax) of File and calls action(g, ff) behind each, with one host thread per GPU (the reference: one
// MPI rank per group of sub-files, slicer-v2.cpp:162-175, densitymaps.cpp:432-484).  GPU g takes sub-files ffmin + g,
// ffmin + g + ngpu, ...; it reads sub-file k+1 into its second page-locked buffer while the copy and the work on sub-file k run.
// e->used[g] counts the sub-files GPU g has staged before the current one.  Log lines (with `log_tail`, when `log` is set) and
// errors are collected per thread and printed GPU by GPU afterwards.
static int walk_subfiles(Engine *e, const InputParams &p, const std::string &File, unsigned ffmin, unsigned ffmax, bool log,
                         const std::string &log_tail, const std::function<int(int, unsigned)> &action)
{
  const int ngpu = (int)e->h.size();
  std::fill(e->used.begin(), e->used.end(), 0);
  std::vector<int> rcs(ngpu, 0);
  std::vector<std::string> logs(ngpu), errs(ngpu);
  std::vector<double> read_s(ngpu, 0.0);
  auto work = [&](int g) {
    std::ostringstream out, err;
    for (unsigned ff = ffmin + (unsigned)g; ff < ffmax && !rcs[g]; ff += (unsigned)ngpu)
    {
      SubFile &buf = e->bufs[2 * g + (e->used[g] & 1)];
      if (e->used[g] >= 2 && slicer_wait_staging(e->h[g])) // the copy that last read this host buffer must be done
      {
        err << "slicer_wait_staging: " << slicer_last_error() << "\n";
        rcs[g] = 1;
        break;
      }
      const double tr0 = now_s();
      if (readSubFile(File + "." + std::to_string(ff), p.hydro, buf, true))
      {
        rcs[g] = 1;
        break;
      }
      read_s[g] += now_s() - tr0;
      const Header &data = buf.header;
      if (buf.ntotal > e->capacity)
      { // cannot happen after the header scan of ensure_capacity() unless the file changed in between
        err << "sub-file " << ff << " holds " << buf.ntotal << " particles, more than the engine's capacity " << e->capacity << "\n";
        rcs[g] = 1;
        break;
      }
      if (log)
        out << " sub-file " << ff << ": " << buf.ntotal << " particles -> GPU " << e->devices[g] << log_tail << "\n";
      int rc = e->used[g] == 0 ? slicer_begin_snapshot(e->h[g], data.boxsize, data.massarr, p.hydro) : slicer_next_batch(e->h[g]);
      if (!rc)
        rc = stage_subfile(e->h[g], buf, p.hydro);
      if (!rc)
        rc = action(g, ff);
      if (rc)
      {
        err << "GPU " << e->devices[g] << ", sub-file " << ff << ": " << slicer_last_error() << "\n";
        rcs[g] = 1;
        break;
      }
      e->used[g]++;
    }
    logs[g] = out.str();
    errs[g] = err.str();
  };
  if (ngpu == 1)
    work(0);
  else
  {
    std::vector<std::thread> th;
    for (int g = 0; g < ngpu; g++)
      th.emplace_back(work, g);
    for (auto &t : th)
      t.join();
  }
  for (int g = 0; g < ngpu; g++)
  {
    t_read += read_s[g] / ngpu;
    std::cout << logs[g];
    std::cerr << errs[g];
    if (rcs[g])
      return 1;
  }
  return 0;
}

// The end of a group of passes [pass, end) after walk_subfiles: a GPU without sub-files still contributes zero maps to the sum
// (slicer-v2.cpp:162-175: ranks with no files), the group's slots are summed on GPU 0 and its jobs' maps and counts read out.
static int finish_group(Engine *e, const InputParams &p, const std::string &File, unsigned ffmin, unsigned ffmax, const std::vector<PlaneJob> &jobs,
                        const std::vector<slicer_plane_desc> &descs, const PassSpan *pass, const PassSpan *end,
                        std::vector<std::valarray<float>> &mapxytot, std::vector<std::valarray<float>> &mapxytoti, std::vector<long long> &ntotxyi)
{
  const int ngpu = (int)e->h.size();
  const int j0 = pass->first, j1 = (end - 1)->first + (end - 1)->n;
  for (int g = 0; g < ngpu; g++)
    if (e->used[g] == 0)
    {
      Header hd;
      const bool have_header = ffmax > ffmin && readHeader(File + "." + std::to_string(ffmin), hd) == 0;
      const double zero[6] = {0, 0, 0, 0, 0, 0};
      if (slicer_begin_snapshot(e->h[g], have_header ? hd.boxsize : 1.0, have_header ? hd.massarr : zero, p.hydro) ||
          deposit_passes(e->h[g], descs, pass, end, false))
        return fail_capi("slicer_deposit");
    }
  if (ngpu > 1 && slicer_reduce_all_slots(e->h.data(), ngpu, 0, j1 - j0, 0)) // replaces the 7 MPI_Reduce of slicer-v2.cpp:214-217
    return fail_capi("slicer_reduce_all");
  const double tf0 = now_s();
  for (int j = j0; j < j1; j++)
  {
    const int npix = jobs[j].npix;
    long long counts[6];
    mapxytot[j].resize((size_t)npix * npix);
    if (slicer_fetch(e->h[0], j - j0, -1, &mapxytot[j][0], counts, nullptr))
      return fail_capi("slicer_fetch");
    for (int t = 0; t < 6; t++)
    {
      ntotxyi[(size_t)j * 6 + t] = counts[t];
      if (e->per_type)
      {
        mapxytoti[(size_t)j * 6 + t].resize((size_t)npix * npix);
        if (slicer_fetch(e->h[0], j - j0, t, &mapxytoti[(size_t)j * 6 + t][0], nullptr, nullptr))
          return fail_capi("slicer_fetch");
      }
    }
  }
  t_fetch += now_s() - tf0;
  return 0;
}

// `Part. Degradation` (snopt > 0, densitymaps.cpp:387-397).  The reference consumes one libc rand() per accepted
// (particle, replica) pair, plane after plane, sub-file after sub-file, type after type, particle after particle —
// one serial stream that continues from randomizeBox's last srand().  Sweep 1 counts the accepted pairs of every
// (plane, sub-file, type); the draws are then made here, in that order, with the same libc generator; sweep 2 applies
// them on the device by rank (slicer_count_accepted / slicer_deposit_degraded).
static int createDensityMapsDegraded(Engine *e, const InputParams &p, const std::vector<PlaneJob> &jobs, const std::vector<slicer_plane_desc> &descs,
                                     unsigned ffmin, unsigned ffmax, const std::string &File, std::vector<std::valarray<float>> &mapxytot,
                                     std::vector<std::valarray<float>> &mapxytoti, std::vector<long long> &ntotxyi, int myid)
{
  const int nj = (int)jobs.size();
  if (nj > std::min(e->max_planes, (int)SLICER_MAX_PLANES))
  {
    std::cerr << "Part. Degradation: more than " << std::min(e->max_planes, (int)SLICER_MAX_PLANES) << " planes share one snapshot; not supported"
              << std::endl;
    return 1;
  }
  const unsigned nff = ffmax - ffmin;
  // ---- sweep 1: accepted pairs per (plane, sub-file, type)
  std::vector<long long> cnt((size_t)nff * nj * 6, 0);
  if (walk_subfiles(e, p, File, ffmin, ffmax, false, "", [&](int g, unsigned ff) {
        return slicer_count_accepted(e->h[g], descs.data(), nj, &cnt[(size_t)(ff - ffmin) * nj * 6]);
      }))
    return 1;
  // ---- the draws, in the reference's order: plane-major, then sub-file, then type/particle/replica
  const double thr = 1. / pow(2, p.snopt);
  std::vector<std::vector<unsigned char>> keep((size_t)nj * nff);
  for (int j = 0; j < nj; j++)
    for (unsigned f = 0; f < nff; f++)
    {
      long long n = 0;
      for (int t = 0; t < 6; t++)
        n += cnt[((size_t)f * nj + j) * 6 + t];
      std::vector<unsigned char> &k = keep[(size_t)j * nff + f];
      k.resize((size_t)n);
      for (long long i = 0; i < n; i++)
        k[i] = (sharedRand().next() / float(RAND_MAX) < thr) ? 1 : 0; // densitymaps.cpp:393
    }
  // ---- sweep 2: deposit with the draws applied by rank
  if (walk_subfiles(e, p, File, ffmin, ffmax, myid == 0, " (degradation 2^-" + std::to_string(p.snopt) + ")", [&](int g, unsigned ff) {
        std::vector<long long> again((size_t)nj * 6);
        std::vector<const unsigned char *> kp(nj);
        for (int j = 0; j < nj; j++)
          kp[j] = keep[(size_t)j * nff + (ff - ffmin)].data();
        return slicer_count_accepted(e->h[g], descs.data(), nj, again.data()) ||
               slicer_deposit_degraded(e->h[g], descs.data(), nj, p.snopt, kp.data(), e->used[g] > 0);
      }))
    return 1;
  const PassSpan all = {0, nj};
  return finish_group(e, p, File, ffmin, ffmax, jobs, descs, &all, &all + 1, mapxytot, mapxytoti, ntotxyi);
}

int createDensityMapsMulti(Engine *e, InputParams &p, Lens &lens, Random &random, const std::vector<PlaneJob> &jobs, unsigned ffmin,
                           unsigned ffmax, const std::string &File, double fovradiants, std::vector<std::valarray<float>> &mapxytot,
                           std::vector<std::valarray<float>> &mapxytoti, std::vector<long long> &ntotxyi, int myid)
{
  const int njobs = (int)jobs.size();
  mapxytot.assign(njobs, std::valarray<float>());
  mapxytoti.assign((size_t)njobs * 6, std::valarray<float>());
  ntotxyi.assign((size_t)njobs * 6, 0);
  std::vector<slicer_plane_desc> descs;
  for (const PlaneJob &job : jobs)
    descs.push_back(make_desc(lens, job.random ? *job.random : random, job.isnap, job.rcase, fovradiants, job.npix));
  // (before the passes are planned: rebuilt handles may have fewer slots)
  if (ensure_capacity(e, File, ffmin, ffmax))
    return 1;
  if (p.snopt > 0)
    return createDensityMapsDegraded(e, p, jobs, descs, ffmin, ffmax, File, mapxytot, mapxytoti, ntotxyi, myid);
  const std::vector<PassSpan> passes = plan_passes(jobs, descs, std::min(e->max_planes, (int)SLICER_MAX_PLANES));
  // groups of consecutive passes that fit the engine's slots: each group reads the sub-files once
  for (size_t p0 = 0; p0 < passes.size();)
  {
    size_t p1 = p0;
    int nslots = 0;
    while (p1 < passes.size() && nslots + passes[p1].n <= e->max_planes)
      nslots += passes[p1++].n;
    const PassSpan *first = &passes[p0], *end = first + (p1 - p0);
    if (walk_subfiles(e, p, File, ffmin, ffmax, myid == 0, "",
                      [&](int g, unsigned) { return deposit_passes(e->h[g], descs, first, end, e->used[g] > 0); }) ||
        finish_group(e, p, File, ffmin, ffmax, jobs, descs, first, end, mapxytot, mapxytoti, ntotxyi))
      return 1;
    p0 = p1;
  }
  return 0;
}

int createDensityMaps(Engine *e, InputParams &p, Lens &lens, Random &random, int isnap, unsigned ffmin, unsigned ffmax,
                      const std::string &File, double fovradiants, double rcase, std::valarray<float> &mapxytot,
                      std::valarray<float> (&mapxytoti)[6], int (&ntotxyi)[6], int myid)
{
  std::vector<PlaneJob> jobs = {{isnap, rcase, p.npix}};
  std::vector<std::valarray<float>> tot, per;
  std::vector<long long> cnt;
  if (createDensityMapsMulti(e, p, lens, random, jobs, ffmin, ffmax, File, fovradiants, tot, per, cnt, myid))
    return 1;
  mapxytot = tot[0];
  for (int i = 0; i < 6; i++)
  {
    if (e->per_type)
      mapxytoti[i] = per[i];
    else
      mapxytoti[i].resize((size_t)p.npix * p.npix); // zero-filled, as the reference's resize() leaves them
    ntotxyi[i] = (int)cnt[i];
  }
  return 0;
}

static std::string plane_label(int pll)
{ // slicer-v2.cpp:154-159
  char b[32];
  snprintf(b, sizeof(b), "%03d", pll);
  return b;
}

// ---- several realisations in one run ---------------------------------------------------------------------------------
// Realisations of one run share the plan, the engine and every read of a snapshot: their inis must agree on every entry that
// shapes them.  Checked before anything is read, allocated or written.
static int check_realisations(const std::vector<std::string> &inis, const std::vector<InputParams> &ps)
{
  auto num = [](double v) {
    std::ostringstream o;
    o.precision(17);
    o << v;
    return o.str();
  };
  struct Shared
  {
    const char *entry;
    std::function<std::string(const InputParams &)> value;
  };
  const Shared shared[] = {
      {"entry 1 (map pixels)", [](const InputParams &q) { return std::to_string(q.npix); }},
      {"entry 2 (source redshift)", [&](const InputParams &q) { return num(q.zs); }},
      {"entry 3 (field of view)", [&](const InputParams &q) { return num(q.fov); }},
      {"entry 4 (snapshot list)", [](const InputParams &q) { return q.filredshiftlist; }},
      {"entry 5 (snapshot path)", [](const InputParams &q) { return q.pathsnap; }},
      {"entry 10 (one map per particle type)", [](const InputParams &q) { return std::to_string((int)q.partinplanes); }},
      {"entry 14 (dark-energy w)", [&](const InputParams &q) { return num(q.w); }},
  };
  for (size_t k = 1; k < ps.size(); k++)
    for (const Shared &sh : shared)
      if (sh.value(ps[k]) != sh.value(ps[0]))
      {
        std::cerr << inis[k] << ": " << sh.entry << " is '" << sh.value(ps[k]) << "', " << inis[0] << " has '" << sh.value(ps[0])
                  << "': the light cones of one run share the plan and every snapshot read, so they must agree on it" << std::endl;
        return 1;
      }
  int degraded = -1;
  for (size_t k = 0; k < ps.size(); k++)
    if (ps[k].snopt > 0)
    {
      if (degraded >= 0)
      {
        std::cerr << inis[k] << ": entry 13 (particle degradation) is " << ps[k].snopt << ", and " << inis[degraded] << " sets it too: at most one "
                  << "light cone of a run may degrade particles (the degradation draws one serial random stream per run)" << std::endl;
        return 1;
      }
      degraded = (int)k;
    }
  // no two realisations may write the same file: the planes list (output directory + suffix) or a plane (+ simulation name)
  std::map<std::string, size_t> owner;
  for (size_t k = 0; k < ps.size(); k++)
    for (const std::string &f : {ps[k].directory + "planes_list_" + ps[k].suffix + ".txt", fileOutput(ps[k], plane_label(0))})
    {
      std::error_code ec;
      std::string key = std::filesystem::weakly_canonical(std::filesystem::absolute(f, ec), ec).string();
      if (ec)
        key = f;
      auto ins = owner.insert({key, k});
      if (!ins.second && ins.first->second != k)
      {
        std::cerr << inis[k] << ": writes " << f << " as " << inis[ins.first->second] << " does: entries 6, 11 and 12 (simulation name, "
                  << "output directory, output suffix) must give every light cone of a run its own files" << std::endl;
        return 1;
      }
    }
  return 0;
}

int runLightCones(const std::vector<std::string> &inifiles, const RunOptions &opt)
{
  const int myid = opt.quiet ? 1 : 0;
  const double t_begin = now_s();
  t_read = t_submit = t_fetch = t_write = t_engine = t_gpu = 0;
  const int K = (int)inifiles.size();
  if (K == 0)
  {
    std::cerr << "no InputParams.ini given" << std::endl;
    return 1;
  }
  std::vector<InputParams> ps(K);
  for (int k = 0; k < K; k++)
  {
    if (readInput(ps[k], inifiles[k]))
      return 1;
    if (ps[k].simType == "SubFind")
    {
      std::cerr << "npix == 0 selects the SubFind halo catalogue branch, which this build does not provide" << std::endl;
      return 1;
    }
  }
  if (check_realisations(inifiles, ps))
    return 1;
  // the plan is the same for every realisation: it is made from the first ini
  InputParams &p = ps[0];
  std::vector<std::string> snappath;
  std::vector<double> snapred, snapbox;
  if (readRedList(p.filredshiftlist, snapred, snappath, snapbox, p))
    return 1;
  Header simdata;
  if (readHeader(p.pathsnap + snappath[0] + ".0", simdata))
    return 1;
  CosmoTable cosmo;
  cosmo.build(simdata.om0, simdata.oml, p.w, p.zs);
  for (InputParams &q : ps)
  {
    testHydro(q, simdata); // decided once from the first listed snapshot (slicer-v2.cpp:74-76)
    q.Ds = cosmo.getDl.eval(q.zs);
  }
  Lens lens;
  if (buildPlanes(p, lens, snapred, snappath, snapbox, cosmo.getDl, cosmo.getZl, numberOfLensPerSnap, 0)) // rank 0 writes planes_list
    return 1;
  for (int k = 1; k < K; k++)
    writePlanesList(ps[k], lens);
  double fovradiants = 0;
  for (size_t i = 0; i < lens.ld.size(); i++)
  {
    if (i == 0)
      lens.nrepperp.assign(lens.ld.size(), 0);
    const double boxl = snapbox[lens.fromsnapi[i]] / 1e3 * POS_U;
    if (!opt.replication)
    {
      if (testFov(p.fov, boxl, lens.ld2[i], 0, fovradiants))
        return 1;
    }
    else
      computeReplications(p.fov, boxl, lens.ld2[i], myid, fovradiants, lens.nrepperp[i]);
  }
  // one randomisation per realisation; a degrading one last: its draws continue the shared stream its randomizeBox left
  std::vector<Random> randoms(K);
  int degraded = -1;
  for (int k = 0; k < K; k++)
    if (ps[k].snopt > 0)
      degraded = k;
    else
      randomizeBox(randoms[k], lens, ps[k], numberOfLensPerSnap, 1, opt.fixed_vertex);
  if (degraded >= 0)
    randomizeBox(randoms[degraded], lens, ps[degraded], numberOfLensPerSnap, 1, opt.fixed_vertex);

  // per-plane rcase and npix, exactly as the sequential loop of slicer-v2.cpp:137-185 would see them
  std::vector<double> rcase(lens.nplanes, 0.0);
  std::vector<int> npix(lens.nplanes, p.npix);
  float rc = 0.0f;
  int npix_max = 1;
  for (int isnap = 0; isnap < lens.nplanes; isnap++)
  {
    if (p.physical)
      npix[isnap] = int((lens.ld2[isnap] + lens.ld[isnap]) / 2 * fovradiants / p.rgrid * 1e3 / POS_U) + 1;
    if (lens.randomize[isnap])
      rc = lens.ld[isnap] / snapbox[lens.fromsnapi[isnap]] * 1e3 / POS_U;
    rcase[isnap] = rc;
    npix_max = std::max(npix_max, npix[isnap]);
  }
  if (p.partinplanes && myid == 0)
    std::cout << "!It is not possible to resume a Gadget run with partinplanes == true!" << std::endl
              << "!!               Files on Output folder will be overwritten        !!" << std::endl;

  Engine *e = nullptr;
  int status = 0;
  // The planes of a snapshot are written by background threads while the next snapshot is read and deposited (an 8192^2
  // plane is 256 MiB of byte-swapped FITS).  At most one snapshot's planes are in flight.
  std::thread writer;
  int writer_status = 0;
  double writer_seconds = 0;
  auto join_writer = [&]() {
    if (writer.joinable())
    {
      writer.join();
      t_write += writer_seconds;
      if (writer_status)
        status = 1;
    }
  };
  for (int s0 = 0; s0 < lens.nplanes && !status;)
  {
    // planes [s0, s1) use the same snapshot
    int s1 = s0 + 1;
    while (s1 < lens.nplanes && lens.fromsnapi[s1] == lens.fromsnapi[s0])
      s1++;
    // the planes of every realisation still to be made, realisation after realisation; a degrading one's apart
    std::vector<PlaneJob> jobs, djobs;
    std::vector<int> owner;
    for (int k = 0; k < K; k++)
      for (int isnap = s0; isnap < s1; isnap++)
      {
        const std::string out = fileOutput(ps[k], plane_label(lens.pll[isnap]));
        if (!p.partinplanes && std::ifstream(out))
        { // resume: this plane was already written (slicer-v2.cpp:188-196)
          if (myid == 0)
            std::cout << out << " Already exists" << std::endl;
          continue;
        }
        (k == degraded ? djobs : jobs).push_back({isnap, rcase[isnap], npix[isnap], &randoms[k]});
        if (k != degraded)
          owner.push_back(k);
      }
    const std::string File = p.pathsnap + lens.fromsnap[s0];
    Header snapdata;
    if (readHeader(File + ".0", snapdata))
    {
      status = 1;
      break;
    }
    if (!jobs.empty() || !djobs.empty())
    {
      if (!e)
      {
        size_t tot = 0;
        for (int i = 0; i < 6; i++)
          tot += (size_t)snapdata.npartTotal[i] + ((size_t)(uint32_t)snapdata.nTotalHW[i] << 32);
        const size_t cap = tot / std::max(1, snapdata.numfiles) * 5 / 4 + 65536;
        const double te0 = now_s();
        int most = 1; // the most planes one snapshot feeds
        for (int a = 0; a < lens.nplanes;)
        {
          int b = a + 1;
          while (b < lens.nplanes && lens.fromsnapi[b] == lens.fromsnapi[a])
            b++;
          most = std::max(most, b - a);
          a = b;
        }
        // slots for every realisation's planes of a snapshot, so that it is read once; fewer if the GPUs hold fewer or the caller
        // asks for fewer (opt.max_slots), but at least one realisation's planes of a snapshot (up to a pass: 16): the degrading
        // light cone needs them in one pass, and fewer would read a snapshot once per part of a light cone
        const int batched = std::max(1, K - (degraded >= 0 ? 1 : 0));
        int want = std::min((int)SLICER_MAX_SLOTS, most * batched), need = std::min(most, (int)SLICER_MAX_PLANES);
        if (opt.max_slots > 0)
        {
          want = std::min(want, opt.max_slots);
          if (degraded < 0)
            need = std::min(need, want);
          want = std::max(want, need);
        }
        e = engine_new(opt.devices, npix_max, opt.mas, p.partinplanes, cap, opt.deposit_mode, want, want, need);
        t_engine += now_s() - te0;
        if (!e)
        {
          status = 1;
          break;
        }
      }
      std::vector<std::valarray<float>> tot, per;
      std::vector<long long> cnt;
      if (!jobs.empty() &&
          createDensityMapsMulti(e, ps[owner[0]], lens, randoms[owner[0]], jobs, 0, snapdata.numfiles, File, fovradiants, tot, per, cnt, myid))
      {
        status = 1;
        break;
      }
      if (!djobs.empty())
      {
        std::vector<std::valarray<float>> dtot, dper;
        std::vector<long long> dcnt;
        if (createDensityMapsMulti(e, ps[degraded], lens, randoms[degraded], djobs, 0, snapdata.numfiles, File, fovradiants, dtot, dper, dcnt,
                                   myid))
        {
          status = 1;
          break;
        }
        for (auto &m : dtot)
          tot.push_back(std::move(m));
        for (auto &m : dper)
          per.push_back(std::move(m));
        cnt.insert(cnt.end(), dcnt.begin(), dcnt.end());
        jobs.insert(jobs.end(), djobs.begin(), djobs.end());
        owner.insert(owner.end(), djobs.size(), degraded);
      }
      join_writer(); // the previous snapshot's planes
      if (status)
        break;
      struct Batch
      {
        std::vector<PlaneJob> jobs;
        std::vector<int> owner;
        std::vector<double> zsim;
        std::vector<std::valarray<float>> tot, per;
        std::vector<long long> cnt;
        Header snapdata;
      };
      auto batch = std::make_shared<Batch>();
      batch->jobs = jobs;
      batch->owner = owner;
      for (size_t j = 0; j < jobs.size(); j++)
        batch->zsim.push_back(cosmo.getZl.eval((lens.ld2[jobs[j].isnap] + lens.ld[jobs[j].isnap]) / 2.0));
      batch->tot = std::move(tot);
      batch->per = std::move(per);
      batch->cnt = std::move(cnt);
      batch->snapdata = snapdata;
      writer_status = 0;
      writer_seconds = 0;
      // the files are independent: several realisations' planes (hundreds of MB per snapshot at 2048^2) go out on several threads
      writer = std::thread([batch, K, &ps, &lens, &writer_status, &writer_seconds]() {
        const double tw0 = now_s();
        std::atomic<size_t> next{0};
        std::atomic<int> failed{0};
        auto write_some = [&]() {
          for (size_t j; !failed && (j = next++) < batch->jobs.size();)
          {
            const int isnap = batch->jobs[j].isnap;
            InputParams pj = ps[batch->owner[j]];
            pj.npix = batch->jobs[j].npix;
            try
            {
              writeMaps(pj, batch->snapdata, lens, isnap, batch->zsim[j], plane_label(lens.pll[isnap]), batch->tot[j],
                        pj.partinplanes ? &batch->per[j * 6] : nullptr, &batch->cnt[j * 6], 0);
            }
            catch (const SliceError &err)
            {
              std::cerr << "It was not possible to create the map: " + err.what + "\n" << std::flush;
              failed = 1;
            }
          }
        };
        // (one light cone: one thread, so that its messages come out in plane order as they always did)
        const size_t nthreads =
            K == 1 ? 1 : std::min({batch->jobs.size(), (size_t)8, (size_t)std::max(1u, std::thread::hardware_concurrency() / 2)});
        std::vector<std::thread> more;
        for (size_t t = 1; t < nthreads; t++)
          more.emplace_back(write_some);
        write_some();
        for (auto &t : more)
          t.join();
        writer_status = failed;
        writer_seconds = now_s() - tw0;
      });
    }
    s0 = s1;
  }
  join_writer();
  engineDestroy(e);
  if (getenv("SLICER_B200_TIMING"))
    std::cerr << "[timing] total " << now_s() - t_begin << " s: engine/CUDA set-up " << t_engine << ", sub-file reads " << t_read << ", fetch (waits for the GPU) " << t_fetch
              << ", FITS writes (background thread) " << t_write << ", device passes " << t_gpu << " (" << K << " light cone" << (K > 1 ? "s" : "") << ")"
              << std::endl;
  return status;
}

int runLightCone(const std::string &inifile, const RunOptions &opt) { return runLightCones({inifile}, opt); }

} // namespace slicer
