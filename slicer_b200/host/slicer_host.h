// slicer_host.h — the C++ host side of the B200 light-cone mass-map path.
//
// Everything a user of SLICER's Gadget branch touches on this path, with the reference's names, argument meaning
// and error behaviour, but driving the CUDA library through the C ABI of include/slicer_b200.h:
//   InputParams / readInput        SLICER/data.h:29-49, data.cpp:8-87      (positional InputParams.ini)
//   Header / readHeader / POS, MASS, BHMA blocks   data.h:59-95, gadget2io.cpp:8-31,125-165,189-202
//   readRedList                    gadget2io.cpp:613-661
//   CosmoTable (w0waCDM recurrence) + CubicSpline   w0waCDM.cpp:18-84, slicer-v2.cpp:79-96 (GSL natural cspline)
//   Lens / buildPlanes / getSnap   data.h:104-117, densitymaps.cpp:9-156
//   Random / randomizeBox          data.h:126-131, densitymaps.cpp:166-248
//   testFov / computeReplications  densitymaps.cpp:255-283
//   createDensityMaps              densitymaps.cpp:419-524 (densitymaps.h:161-165)  -> CUDA pass(es)
//   writeMaps / fileOutput         densitymaps.cpp:530-649                          -> FITS primary image
//   runLightCone(s)                slicer-v2.cpp:23-230 (the plane driver), restructured per SNAPSHOT, for one or several
//                                  realisations of the light cone (InputParams.ini files that differ in seeds and output)
#pragma once
#include <cstdint>
#include <cstdio>
#include <functional>
#include <string>
#include <valarray>
#include <vector>

#include "../../include/slicer_b200.h"

namespace slicer
{

constexpr double POS_U = 1.0;           // gadget2io.h:14
constexpr double MAX_M = 1e3;           // densitymaps.h:21
constexpr int numberOfLensPerSnap = 4;  // densitymaps.h:23
constexpr int neval = 1000;             // slicer-v2.cpp:5
constexpr double speedcunit = 2.99792458e+3; // utilities.h:19

struct InputParams // data.h:29-49
{
  int npix = 0;
  double zs = 0, Ds = 0, fov = 0;
  bool hydro = false;
  std::string simType, filredshiftlist, pathsnap, simulation, directory, suffix, snpix;
  int rgrid = 0;
  int seedcenter = 0, seedface = 0, seedsign = 0;
  bool partinplanes = false;
  int snopt = 0;
  bool physical = false;
  double w = -1;
};

#pragma pack(push, 1)
struct Header // data.h:59-79 — the 256-byte GADGET header as the reference reads it
{
  int32_t npart[6];
  double massarr[6];
  double time;
  double redshift;
  int32_t flag_sfr;
  int32_t flag_feedback;
  uint32_t npartTotal[6];
  int32_t flag_cooling;
  int32_t numfiles;
  double boxsize;
  double om0;
  double oml;
  double h;
  int32_t flag_sage;
  int32_t flag_metals;
  int32_t nTotalHW[6];
  int32_t flag_entropy;
  int32_t la[15];
};
#pragma pack(pop)
static_assert(sizeof(Header) == 256, "GADGET header is 256 bytes");

struct Lens // data.h:104-117
{
  int nplanes = 0;
  std::vector<int> replication, pll, fromsnapi, nrepperp;
  std::vector<std::string> fromsnap;
  std::vector<double> zsimlens, ld, ld2, zfromsnap;
  std::vector<bool> randomize;
};

struct Random // data.h:126-131
{
  std::vector<double> x0, y0, z0;
  std::vector<int> sgnX, sgnY, sgnZ, face;
};

// GSL's gsl_interp_cspline (natural cubic spline), restated: see plan.cpp
class CubicSpline
{
public:
  void init(const std::vector<double> &x, const std::vector<double> &y);
  double eval(double x) const; // NaN outside [x0, xn] (GSL raises GSL_EDOM)
private:
  std::vector<double> x_, y_, c_;
};

struct CosmoTable // slicer-v2.cpp:79-96
{
  std::vector<double> zl, dl;
  CubicSpline getDl, getZl;
  void build(double om0, double oml, double w, double zs);
};

// glibc's rand()/srand() (random_r.c, TYPE_3: additive feedback x^31 + x^3 + 1, seeded by the 16807 Lehmer LCG, 310
// outputs discarded), restated so that the draws of randomizeBox and of `Part. Degradation` do not depend on — and are
// not disturbed by — the process-wide libc state (CUDA, NCCL or user code may call rand()).  Checked against libc in
// tests/test_host_layer.py.
class GlibcRand
{
public:
  void seed(unsigned int s);
  int next(); // 0 .. RAND_MAX (2147483647)
private:
  int32_t r_[34];
  int f_ = 3, b_ = 0;
};
GlibcRand &sharedRand(); // the stream the reference's global rand() state corresponds to

struct SliceError
{
  std::string what;
};

// ---- configuration and plan ------------------------------------------------------------------------------
int readInput(InputParams &p, const std::string &name); // exits(1) if the file is missing, like data.cpp:13-19
int readHeader(const std::string &file_in, Header &header);
void testHydro(InputParams &p, const Header &data);
int readRedList(const std::string &filredshiftlist, std::vector<double> &snapred, std::vector<std::string> &snappath,
                std::vector<double> &snapbox, InputParams &p);
int getSnap(const std::vector<double> &zsnap, const CubicSpline &getDl, double dlens);
int buildPlanes(InputParams &p, Lens &lens, std::vector<double> &snapred, std::vector<std::string> &snappath,
                std::vector<double> &snapbox, const CubicSpline &getDl, const CubicSpline &getZl, int numOfLensPerSnap, int myid);
void writePlanesList(const InputParams &p, const Lens &lens); // planes_list_<suffix>.txt of a plan (buildPlanes writes it on rank 0)
void randomizeBox(Random &random, const Lens &lens, const InputParams &p, int numOfLensPerSnap, int myid, bool fixedVertex = false);
int testFov(double fov, double boxl, double Ds, int myid, double &fovradiants);
void computeReplications(double fov, double boxl, double Ds, int myid, double &fovradiants, int &nrepperp);

// ---- convergence maps ----------------------------------------------------------------------------------------
// Flat-sky, thin-plane Born weights of every plane of `lens` for each source redshift zs[k] (comoving Mpc/h, masses in the planes'
// unit of 1e10 Msun/h).  For plane i: chi = (ld + ld2) / 2, z = getZl(chi), V = (ld2^3 - ld^3) / (3 chi^2),
// g = (1 + z) chi (chi_s - chi) / chi_s with chi_s = getDl(zs[k]); for chi < chi_s
//   scale[i*S + k] = A g / (rho_c Omega_pix chi^2),   offset[i*S + k] = -A om0 g V,   A = 1.5 / speedcunit^2, Omega_pix = (fov / npix)^2,
// and 0, 0 (the plane does not contribute) otherwise.  slicer_kappa_add applies them to the int64 planes.
constexpr double rho_crit = 27.753662724817193; // 3 (100 km/s/Mpc)^2 / (8 pi G), G = 4.30091727e-9 Mpc (km/s)^2 / Msun: 1e10 Msun/h per (Mpc/h)^3
void kappaWeights(const Lens &lens, const CosmoTable &cosmo, double om0, double oml, double fovradiants, int npix, const std::vector<double> &zs,
                  std::vector<double> &scale, std::vector<double> &offset);

// ---- shear maps -----------------------------------------------------------------------------------------------
// Kaiser–Squires γ1, γ2 of each convergence map (slicer_shear, csrc/shear.cuh) on a zero-padded grid of P^2: the smallest power of
// two >= 2 npix, so that mass near one edge does not wrap onto the other.  The device workspace that takes: two P^2 grids of
// complex doubles, the P-entry twiddle table and the two npix^2 double maps.
inline int shearFftSize(int npix)
{
  int P = 1;
  while (P < 2 * npix)
    P *= 2;
  return P;
}
inline size_t shearWorkspaceBytes(int P, int npix) { return 2 * 16 * (size_t)P * P + 16 * (size_t)P + 16 * (size_t)npix * npix; }

// ---- snapshot sub-files ------------------------------------------------------------------------------------
struct SubFile
{
  Header header;
  // pinned (slicer_alloc_pinned) when `pinned` is set, so that slicer_stage_particles copies asynchronously
  float *pos = nullptr;   // POS payload: npart_total x 3 floats, the six types concatenated in type order
  float *mass = nullptr;  // per-particle masses in the same particle order (0 where the type has massarr != 0)
  size_t capacity = 0;    // particles the buffers can hold
  size_t ntotal = 0;
  bool pinned = false;
  ~SubFile();
  SubFile() = default;
  SubFile(const SubFile &) = delete;
  SubFile &operator=(const SubFile &) = delete;
};
// Reads header + POS (+ MASS / BHMA when `hydro`) of one sub-file with bulk reads.  Returns 0 / 1 like readHeader.
int readSubFile(const std::string &file, bool hydro, SubFile &out, bool pinned);

// ---- the map makers ----------------------------------------------------------------------------------------
struct Engine; // one handle per GPU + staging buffers
Engine *engineCreate(const std::vector<int> &devices, int npix_max, int mas, bool per_type_maps, size_t particle_capacity,
                     int deposit_mode = SLICER_DEPOSIT_AUTO, int max_planes = SLICER_MAX_PLANES);
void engineDestroy(Engine *e);
int engineGpuCount(const Engine *e);

// Drop-in for the reference's createDensityMaps (densitymaps.h:161-165): ONE plane, sub-files [ffmin, ffmax) of File,
// same outputs (resized and zero-filled float maps; ntotxyi are filled — the reference leaves them untouched because
// of the shadowed local at densitymaps.cpp:497).  Returns 0 ok / 1 error like the reference.
int createDensityMaps(Engine *e, InputParams &p, Lens &lens, Random &random, int isnap, unsigned ffmin, unsigned ffmax,
                      const std::string &File, double fovradiants, double rcase, std::valarray<float> &mapxytot,
                      std::valarray<float> (&mapxytoti)[6], int (&ntotxyi)[6], int myid);

// The same for ALL planes that use snapshot File in one sweep over its sub-files (each particle is read once per group of
// jobs that fits the engine's accumulator slots).  Jobs may come from several realisations of the light cone (same plan,
// other seeds): `random` is the realisation's randomisation, nullptr for the call's.  A realisation's consecutive jobs share
// one pass (up to SLICER_MAX_PLANES planes and SLICER_MAX_XFORMS randomisations); passes fill the engine's slots in job order.
struct PlaneJob
{
  int isnap;
  double rcase;
  int npix;
  const Random *random = nullptr;
  bool fetch = true;  // read the maps and counts back (mapxytot / mapxytoti / ntotxyi); false: neither (the plane is not written)
  int kappa_map = -1; // first of the convergence maps this plane adds to (slicer_kappa_add; -1: none)
};
int createDensityMapsMulti(Engine *e, InputParams &p, Lens &lens, Random &random, const std::vector<PlaneJob> &jobs, unsigned ffmin,
                           unsigned ffmax, const std::string &File, double fovradiants, std::vector<std::valarray<float>> &mapxytot,
                           std::vector<std::valarray<float>> &mapxytoti /* [job*6+type] */, std::vector<long long> &ntotxyi /* [job*6+type] */,
                           int myid);

// ---- output --------------------------------------------------------------------------------------------------
std::string fileOutput(const InputParams &p, const std::string &snappl, int label = 0);
// <dir><sim>.<map>_<snpix>_zs<%.4f>_<suffix>.fits, map = kappa, gamma1 or gamma2
std::string kappaFileOutput(const InputParams &p, double zs, const char *map = "kappa");
// FITS primary image (BITPIX -32, NAXIS1 = NAXIS2 = npix, pixel [gx + npix*gy], big-endian) + the reference's keys.
// Throws SliceError if the file exists or cannot be created (CCfits FITS::CantCreate).
void writeFitsImage(const std::string &file, const float *map, int npix, const std::vector<std::pair<std::string, double>> &dkeys,
                    const std::vector<std::pair<std::string, long long>> &ikeys, const std::vector<std::string> &order);
void writeMaps(const InputParams &p, const Header &data, const Lens &lens, int isnap, double zsim, const std::string &snappl,
               const std::valarray<float> &mapxytotrecv, const std::valarray<float> *mapxytotirecv /* [6] */, const long long *ntotxyi,
               int myid);

// ---- the processes of one job (group.cpp) -----------------------------------------------------------------------
// Rank and world size as a launcher hands them to each process: OMPI_COMM_WORLD_RANK/SIZE (Open MPI), PMI_RANK/PMI_SIZE
// (MPICH, Intel MPI), SLURM_PROCID/SLURM_STEP_NUM_TASKS (srun; an sbatch script's batch step is one process), RANK/WORLD_SIZE
// (torchrun), the first family that is set.  The local rank comes from OMPI_COMM_WORLD_LOCAL_RANK, MPI_LOCALRANKID, SLURM_LOCALID
// or LOCAL_RANK (the global rank without one).  With more than one rank, MASTER_ADDR / MASTER_PORT name where rank 0 listens for
// the others; under torchrun (TORCHELASTIC_RUN_ID set), whose agent keeps its own store on MASTER_PORT, rank 0 listens on
// MASTER_PORT + 1.
struct Launch
{
  int rank = 0, nranks = 1, local_rank = 0;
  std::string master_addr;
  int master_port = 0;
};
// `env` looks a variable up (getenv in main).  Returns 1 with a message in `err` for malformed values, or more than one rank without
// MASTER_ADDR / MASTER_PORT.
int launchFromEnv(const std::function<const char *(const char *)> &env, Launch &out, std::string &err);
int defaultDevice(const Launch &l, int ndevices); // a rank's GPU when --gpus is not given: local rank modulo the visible devices

// The host control channel between the ranks of a job: plain TCP, every other rank connected to rank 0.  Every call is collective
// (all ranks make it, in the same order) and returns 0, or 1 once the group is broken: a connection failed or closed (a rank left
// the job).  A broken group fails every later call, and rank 0 then closes every connection, so each rank stops at its next call.
class Group
{
public:
  enum class Op
  {
    Min,
    Max,
    Sum
  };
  ~Group();
  // rank 0 listens on `addr`:`port`, the others connect (retrying until `timeout_s`).  One rank: no sockets, every call a no-op.
  int open(int rank, int nranks, const std::string &addr, int port, double timeout_s);
  int bcast(std::string &blob);                                       // rank 0's blob to every rank
  int allgather(const std::string &mine, std::vector<std::string> &all); // every rank's blob to every rank
  int allreduce(std::vector<long long> &v, Op op);                    // elementwise, same length on every rank
  int agree(int status);       // 1 on every rank if any rank's status is non-zero (or the group is broken)
  void close();                // leave the job: the others fail at their next call
  int rank() const { return rank_; }
  int size() const { return size_; }

private:
  int broken(const std::string &what);
  int rank_ = 0, size_ = 1, listen_fd_ = -1;
  bool broken_ = false;
  std::vector<int> fds_; // rank 0: one per rank; others: [0] to rank 0
};

// Global GPU (0 .. G-1 over the GPUs of every rank, rank after rank) that takes sub-file ff of a snapshot: the round-robin of
// slicer-v2.cpp:162-175 over all GPUs of the job.
int subfileGpu(unsigned ff, unsigned ffmin, int G);
std::vector<unsigned> gpuSubfiles(unsigned ffmin, unsigned ffmax, int gpu, int G); // the sub-files of the job's GPU `gpu`
// per_rank[r]: GPUs of rank r.  Returns G, the job's GPUs; gpu0 = the job's index of rank `rank`'s first GPU
int jobGpus(const std::vector<int> &per_rank, int rank, int &gpu0);

// ---- the whole Gadget branch of main() (slicer-v2.cpp:23-230) -------------------------------------------------
struct RunOptions
{
  std::vector<int> devices = {0}; // this rank's GPUs
  bool replication = false;   // CMake USE_REPLICATION (-DReplicationOnPerpendicularPlane)
  bool fixed_vertex = false;  // CMake USE_FIXED_PLC_VERTEX (-DFixedPLCVertex)
  int mas = SLICER_MAS_TSC;   // densitymaps.h:22 DO_NGP
  int deposit_mode = SLICER_DEPOSIT_AUTO;
  bool quiet = false;
  int max_slots = 0;          // accumulator slots per GPU at most (0: as many as the realisations' planes of a snapshot need, up
                              // to SLICER_MAX_SLOTS, as far as device memory allows); fewer slots mean more reads of a snapshot
  // One job of several processes (nranks > 1): every rank runs runLightCones with the same inis and switches; the sub-files are
  // dealt over the GPUs of all ranks, the planes summed with NCCL, and rank 0 alone writes.  Rank 0 listens on
  // master_addr:master_port for the others, which wait up to connect_timeout_s for it.
  int rank = 0, nranks = 1;
  std::string master_addr;
  int master_port = 0;
  double connect_timeout_s = 300;
  // Convergence maps: one per realisation and source redshift (at most SLICER_KAPPA_MAX_SOURCES), formed on the GPU from the
  // planes; empty = none.  An entry that is NaN stands for the ini's source redshift (entry 2).
  std::vector<double> kappa_zs;
  bool write_planes = true; // false: convergence maps only (planes_list is still written)
  // Shear maps γ1, γ2 of every convergence map (a run with none makes the one of the ini's source redshift), formed on the GPU
  bool shear = false;
};
// One light cone per ini.  The inis must agree on what shapes the plan and the engine (map pixels, source redshift, field of
// view, w, snapshot list and directory, one map per particle type); seeds, simulation name, output directory and suffix may
// differ, no two may write the same file, and at most one may set a particle degradation.  Every snapshot sub-file is read
// once for all of them (once per group of realisations when their planes exceed the accumulators the GPUs hold).  Each
// realisation's files are the bytes runLightCone(its ini) writes.  Nothing is written when the inis are refused.
int runLightCones(const std::vector<std::string> &inifiles, const RunOptions &opt);
int runLightCone(const std::string &inifile, const RunOptions &opt); // runLightCones({inifile}, opt)

} // namespace slicer
