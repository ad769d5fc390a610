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
};
int createDensityMapsMulti(Engine *e, InputParams &p, Lens &lens, Random &random, const std::vector<PlaneJob> &jobs, unsigned ffmin,
                           unsigned ffmax, const std::string &File, double fovradiants, std::vector<std::valarray<float>> &mapxytot,
                           std::vector<std::valarray<float>> &mapxytoti /* [job*6+type] */, std::vector<long long> &ntotxyi /* [job*6+type] */,
                           int myid);

// ---- output --------------------------------------------------------------------------------------------------
std::string fileOutput(const InputParams &p, const std::string &snappl, int label = 0);
// FITS primary image (BITPIX -32, NAXIS1 = NAXIS2 = npix, pixel [gx + npix*gy], big-endian) + the reference's keys.
// Throws SliceError if the file exists or cannot be created (CCfits FITS::CantCreate).
void writeFitsImage(const std::string &file, const float *map, int npix, const std::vector<std::pair<std::string, double>> &dkeys,
                    const std::vector<std::pair<std::string, long long>> &ikeys, const std::vector<std::string> &order);
void writeMaps(const InputParams &p, const Header &data, const Lens &lens, int isnap, double zsim, const std::string &snappl,
               const std::valarray<float> &mapxytotrecv, const std::valarray<float> *mapxytotirecv /* [6] */, const long long *ntotxyi,
               int myid);

// ---- the whole Gadget branch of main() (slicer-v2.cpp:23-230) -------------------------------------------------
struct RunOptions
{
  std::vector<int> devices = {0};
  bool replication = false;   // CMake USE_REPLICATION (-DReplicationOnPerpendicularPlane)
  bool fixed_vertex = false;  // CMake USE_FIXED_PLC_VERTEX (-DFixedPLCVertex)
  int mas = SLICER_MAS_TSC;   // densitymaps.h:22 DO_NGP
  int deposit_mode = SLICER_DEPOSIT_AUTO;
  bool quiet = false;
  int max_slots = 0;          // accumulator slots per GPU at most (0: as many as the realisations' planes of a snapshot need, up
                              // to SLICER_MAX_SLOTS, as far as device memory allows); fewer slots mean more reads of a snapshot
};
// One light cone per ini.  The inis must agree on what shapes the plan and the engine (map pixels, source redshift, field of
// view, w, snapshot list and directory, one map per particle type); seeds, simulation name, output directory and suffix may
// differ, no two may write the same file, and at most one may set a particle degradation.  Every snapshot sub-file is read
// once for all of them (once per group of realisations when their planes exceed the accumulators the GPUs hold).  Each
// realisation's files are the bytes runLightCone(its ini) writes.  Nothing is written when the inis are refused.
int runLightCones(const std::vector<std::string> &inifiles, const RunOptions &opt);
int runLightCone(const std::string &inifile, const RunOptions &opt); // runLightCones({inifile}, opt)

} // namespace slicer
