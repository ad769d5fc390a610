// plan.cpp — configuration and the light-cone plan (host, O(#planes)): readInput, readRedList, cosmology table,
// natural cubic spline, buildPlanes, randomizeBox, testFov, computeReplications.  The outputs are the parameters of
// the CUDA pass; they are reproduced with the reference's own expressions (including its numerical quirks, SURVEY.md
// App. D.7) so that a real InputParams.ini + snapshot list gives the reference's planes.
#include "slicer_host.h"

#include <cmath>
#include <cstdlib>
#include <cstring>
#include <fstream>
#include <iterator>
#include <functional>
#include <iostream>
#include <limits>

namespace slicer
{

static std::string sconv_int(int v)
{
  char b[64];
  snprintf(b, sizeof(b), "%i", v); // utilities.h:22 fINT
  return b;
}

// ---------------------------------------------------------------------------------------------------------------
// InputParams.ini (format of data.cpp:8-87): a positional file of 14 entries, each a label line followed by a value line.
// The parse is table driven: entry k of the table says where value k goes and how it is converted; zs, fov and w go
// through float precision because the reference parses them with stof (data.cpp:26,29,83).
// ---------------------------------------------------------------------------------------------------------------
namespace
{
enum class Conv { Int, Float, Flag, Text };
struct IniEntry
{
  const char *what;
  Conv conv;
  void (*store)(InputParams &, const std::string &, long, float);
};
const IniEntry kIniLayout[14] = {
    {"map pixels", Conv::Int, [](InputParams &q, const std::string &, long i, float) { q.npix = (int)i; }},
    {"source redshift", Conv::Float, [](InputParams &q, const std::string &, long, float f) { q.zs = f; }},
    {"field of view", Conv::Float, [](InputParams &q, const std::string &, long, float f) { q.fov = f; }},
    {"snapshot list", Conv::Text, [](InputParams &q, const std::string &t, long, float) { q.filredshiftlist = t; }},
    {"snapshot path", Conv::Text, [](InputParams &q, const std::string &t, long, float) { q.pathsnap = t; }},
    {"simulation name", Conv::Text, [](InputParams &q, const std::string &t, long, float) { q.simulation = t; }},
    {"seed of the box centres", Conv::Int, [](InputParams &q, const std::string &, long i, float) { q.seedcenter = (int)i; }},
    // the next two labels are crossed in the reference's example file: entry 8 drives the axis permutation, entry 9 the mirrors
    {"seed of the axis permutation", Conv::Int, [](InputParams &q, const std::string &, long i, float) { q.seedface = (int)i; }},
    {"seed of the reflections", Conv::Int, [](InputParams &q, const std::string &, long i, float) { q.seedsign = (int)i; }},
    {"one map per particle type", Conv::Flag, [](InputParams &q, const std::string &, long i, float) { q.partinplanes = i != 0; }},
    {"output directory", Conv::Text, [](InputParams &q, const std::string &t, long, float) { q.directory = t; }},
    {"output suffix", Conv::Text, [](InputParams &q, const std::string &t, long, float) { q.suffix = t; }},
    {"particle degradation", Conv::Int, [](InputParams &q, const std::string &, long i, float) { q.snopt = (int)i; }},
    {"dark-energy w", Conv::Float, [](InputParams &q, const std::string &, long, float f) { q.w = f; }},
};
} // namespace

int readInput(InputParams &p, const std::string &name)
{
  std::ifstream ini(name.c_str());
  if (!ini)
  { // the reference leaves the process here as well (data.cpp:13-19)
    std::cerr << "slicer-b200: cannot open the parameter file '" << name << "'" << std::endl;
    exit(1);
  }
  std::vector<std::string> lines;
  for (std::string l; std::getline(ini, l);)
    lines.push_back(l);
  for (int k = 0; k < 14; k++)
  {
    // value k sits on line 2k+1 (0-based); a file that ends early yields empty values, which the numeric conversions reject
    const std::string text = (size_t)(2 * k + 1) < lines.size() ? lines[2 * k + 1] : std::string();
    const IniEntry &e = kIniLayout[k];
    long iv = 0;
    float fv = 0.f;
    try
    {
      if (e.conv == Conv::Int || e.conv == Conv::Flag)
        iv = std::stoi(text);
      else if (e.conv == Conv::Float)
        fv = std::stof(text);
    }
    catch (const std::exception &)
    {
      std::cerr << "slicer-b200: '" << name << "': entry " << k + 1 << " (" << e.what << ") is not a number: '" << text << "'" << std::endl;
      throw; // std::stoi / std::stof throw out of the reference's readInput too
    }
    e.store(p, text, iv, fv);
  }
  // derived fields (data.cpp:60-81): npix == 0 selects the halo branch, npix < 0 asks for a physical pixel size in kpc/h
  p.simType = p.npix == 0 ? "SubFind" : "Gadget";
  p.physical = p.npix < 0;
  p.snpix = sconv_int(p.physical ? -p.npix : p.npix);
  if (p.physical)
  {
    p.snpix += "_kpc";
    p.rgrid = -p.npix;
  }
  if (p.snopt < 0)
  {
    std::cerr << "slicer-b200: the particle degradation exponent must not be negative (got " << p.snopt << ")" << std::endl;
    return 1;
  }
  return 0;
}

// ---------------------------------------------------------------------------------------------------------------
// The snapshot list (gadget2io.cpp:613-661): whitespace-separated snapshot names in order of increasing redshift; snapshots are
// taken up to and including the first one at or beyond the source.  One behaviour of the reference's extraction loop is part
// of the contract (SURVEY.md App. C): when the list is exhausted before such a snapshot and the file does not end right
// after the last name, the last snapshot is entered a second time.
// ---------------------------------------------------------------------------------------------------------------
int readRedList(const std::string &filredshiftlist, std::vector<double> &snapred, std::vector<std::string> &snappath,
                std::vector<double> &snapbox, InputParams &p)
{
  std::ifstream in(filredshiftlist.c_str(), std::ios::binary);
  if (!in)
  {
    std::cerr << "slicer-b200: cannot open the snapshot list '" << filredshiftlist << "'" << std::endl;
    return 1;
  }
  const std::string text((std::istreambuf_iterator<char>(in)), std::istreambuf_iterator<char>());
  std::vector<std::string> names;
  size_t at = 0, last_end = 0;
  while (true)
  {
    while (at < text.size() && isspace((unsigned char)text[at]))
      at++;
    if (at >= text.size())
      break;
    size_t e = at;
    while (e < text.size() && !isspace((unsigned char)text[e]))
      e++;
    names.push_back(text.substr(at, e - at));
    at = last_end = e;
  }
  const bool ends_after_last_name = last_end == text.size();
  if (names.empty())
    names.push_back(std::string()); // the reference then looks for "<path>.0" and reports it missing
  // the sequence of names the reference's loop visits
  std::vector<std::string> visit = names;
  if (!ends_after_last_name)
    visit.push_back(names.back());
  double z_prev = -999.9;
  for (const std::string &name : visit)
  {
    Header hd;
    snappath.push_back(name);
    if (readHeader(p.pathsnap + name + ".0", hd))
    {
      std::cerr << "slicer-b200: snapshot '" << name << "' of the list has no readable sub-file 0 under '" << p.pathsnap << "'" << std::endl;
      return 1;
    }
    if (hd.redshift < z_prev)
    {
      std::cerr << "slicer-b200: the snapshots in '" << filredshiftlist << "' must be in order of increasing redshift" << std::endl;
      return 1;
    }
    z_prev = std::abs(hd.redshift) < 1e-5 ? 0.0 : hd.redshift;
    snapred.push_back(z_prev);
    snapbox.push_back(hd.boxsize);
    if (!(hd.redshift < p.zs))
      break; // the first snapshot at or beyond the source closes the list
  }
  return 0;
}

// A Gadget snapshot is "hydro" when some particle type present in sub-file 0 has no entry in the mass table, i.e. carries
// per-particle masses in a MASS block (gadget2io.cpp:34-48)
void testHydro(InputParams &p, const Header &data)
{
  if (p.simType != "Gadget")
    return;
  long with_own_mass = 0;
  for (int t = 0; t < 6; t++)
    with_own_mass += data.massarr[t] == 0 ? data.npart[t] : 0;
  p.hydro = with_own_mass != 0;
}

// ---------------------------------------------------------------------------------------------------------------
// GSL gsl_interp_cspline: natural boundary (c_0 = c_n = 0), interior second-derivative coefficients from the
// symmetric tridiagonal system diag_i = 2(h_i + h_{i+1}), offdiag_i = h_{i+1}, rhs_i = 3(dy_{i+1}/h_{i+1} - dy_i/h_i)
// solved by the L D L^T recurrence of GSL's solve_tridiag, evaluated as y_i + t(b + t(c_i + t d)).
// ---------------------------------------------------------------------------------------------------------------
void CubicSpline::init(const std::vector<double> &x, const std::vector<double> &y)
{
  x_ = x;
  y_ = y;
  const size_t n = x.size();
  c_.assign(n, 0.0);
  if (n < 3)
    return;
  const size_t N = n - 2;
  std::vector<double> g(N), diag(N), off(N);
  for (size_t i = 0; i < N; i++)
  {
    const double h_i = x[i + 1] - x[i], h_ip1 = x[i + 2] - x[i + 1];
    const double dy_i = y[i + 1] - y[i], dy_ip1 = y[i + 2] - y[i + 1];
    const double g_i = (h_i != 0.0) ? 1.0 / h_i : 0.0, g_ip1 = (h_ip1 != 0.0) ? 1.0 / h_ip1 : 0.0;
    off[i] = h_ip1;
    diag[i] = 2.0 * (h_ip1 + h_i);
    g[i] = 3.0 * (dy_ip1 * g_ip1 - dy_i * g_i);
  }
  if (N == 1)
  {
    c_[1] = g[0] / diag[0];
    return;
  }
  std::vector<double> alpha(N), gamma(N), cc(N), z(N);
  alpha[0] = diag[0];
  gamma[0] = off[0] / alpha[0];
  for (size_t i = 1; i + 1 < N; i++)
  {
    alpha[i] = diag[i] - off[i - 1] * gamma[i - 1];
    gamma[i] = off[i] / alpha[i];
  }
  alpha[N - 1] = diag[N - 1] - off[N - 2] * gamma[N - 2];
  z[0] = g[0];
  for (size_t i = 1; i < N; i++)
    z[i] = g[i] - gamma[i - 1] * z[i - 1];
  for (size_t i = 0; i < N; i++)
    cc[i] = z[i] / alpha[i];
  c_[N] = cc[N - 1];
  for (size_t i = N - 1; i-- > 0;)
    c_[i + 1] = cc[i] - gamma[i] * c_[i + 2];
}

double CubicSpline::eval(double x) const
{
  const size_t n = x_.size();
  if (n < 2 || x < x_[0] || x > x_[n - 1])
    return std::numeric_limits<double>::quiet_NaN();
  size_t lo = 0, hi = n - 1;
  while (hi > lo + 1)
  {
    const size_t mid = (hi + lo) / 2;
    if (x_[mid] > x)
      hi = mid;
    else
      lo = mid;
  }
  const double dx = x_[lo + 1] - x_[lo], dy = y_[lo + 1] - y_[lo];
  const double b = (dy / dx) - dx * (c_[lo + 1] + 2.0 * c_[lo]) / 3.0;
  const double d = (c_[lo + 1] - c_[lo]) / (3.0 * dx);
  const double t = x - x_[lo];
  return y_[lo] + t * (b + t * (c_[lo] + t * d));
}

// w0waCDM.cpp:18-84 as main drives it (slicer-v2.cpp:79-86): H0 = 100, wa = 0, z_i = i (zs+1)/(neval-1) ascending.
// comovingDistance integrates each table point from the previous cached one with dz = (z - lastZ)/100 and a
// `zi < z` loop that often takes a 101st step; the cached (unscaled) value accumulates.  Reproduced as is.
static double Hz(double z, double H0, double om, double ol, double w0, double wa)
{
  const double rhoLambda = ol * pow(1 + z, 3 * (1 + w0 + wa)) * exp(-3 * wa * z / (1 + z));
  const double rhoM = om * pow(1 + z, 3);
  const double rhoTot = rhoLambda + rhoM + (1 - om - ol) * pow(1 + z, 2);
  return H0 * sqrt(rhoTot);
}

void CosmoTable::build(double om0, double oml, double w, double zs)
{
  const double CSPEEDOFLIGHT = speedcunit * 100, H0 = 100.0, wa = 0.0;
  zl.assign(neval, 0.0);
  dl.assign(neval, 0.0);
  bool have_prev = false;
  double prev_z = 0, prev_d = 0;
  for (int i = 0; i < neval; i++)
  {
    const double z = i * (zs + 1.0) / (neval - 1);
    zl[i] = z;
    double distance = 0, lastZ = 0, dz = 1e-4;
    if (have_prev && prev_z == z)
    { // cache hit returns the UNSCALED value (w0waCDM.cpp:30-33); unreachable for strictly increasing z
      dl[i] = prev_d;
      continue;
    }
    if (have_prev)
    {
      distance = prev_d;
      lastZ = prev_z;
      dz = (z - lastZ) / 100;
    }
    for (double zi = lastZ; zi < z; zi += dz)
      distance += 0.5 * dz * (1.0 / Hz(zi, H0, om0, oml, w, wa) + 1.0 / Hz(zi + dz, H0, om0, oml, w, wa));
    prev_z = z;
    prev_d = distance;
    have_prev = true;
    const double D_C = distance * CSPEEDOFLIGHT;
    if (fabs(1 - om0 - oml) < 1e-5)
      dl[i] = D_C;
    else
    {
      const double OmegaK = 1.0 - om0 - oml, s = sqrt(fabs(OmegaK));
      dl[i] = OmegaK < 0 ? CSPEEDOFLIGHT / H0 / s * sinh(s * H0 / CSPEEDOFLIGHT * D_C) : CSPEEDOFLIGHT / H0 / s * sin(s * H0 / CSPEEDOFLIGHT * D_C);
    }
  }
  getDl.init(zl, dl);
  getZl.init(dl, zl);
}

void kappaWeights(const Lens &lens, const CosmoTable &cosmo, double om0, double, double fovradiants, int npix, const std::vector<double> &zs,
                  std::vector<double> &scale, std::vector<double> &offset)
{
  const size_t S = zs.size();
  scale.assign((size_t)lens.nplanes * S, 0.0);
  offset.assign((size_t)lens.nplanes * S, 0.0);
  const double A = 1.5 / (speedcunit * speedcunit);
  const double pix = fovradiants / npix, omega_pix = pix * pix; // flat sky: the cos(dec) of the (dec, ra) pixels is left out
  for (int i = 0; i < lens.nplanes; i++)
  {
    const double ld = lens.ld[i], ld2 = lens.ld2[i];
    const double chi = (ld + ld2) / 2.0;
    const double z = cosmo.getZl.eval(chi);
    // comoving depth of the cone segment per unit solid angle over chi^2: makes the mean term exact (ld2 - ld is 33 % off on the
    // first plane)
    const double V = (ld2 * ld2 * ld2 - ld * ld * ld) / (3.0 * chi * chi);
    for (size_t k = 0; k < S; k++)
    {
      const double chis = cosmo.getDl.eval(zs[k]);
      if (!(chi < chis))
        continue;
      const double g = (1.0 + z) * chi * (chis - chi) / chis;
      scale[i * S + k] = A * g / (rho_crit * omega_pix * chi * chi);
      offset[i * S + k] = -(A * om0 * g * V);
    }
  }
}

// The snapshot whose comoving distance is nearest to dlens (densitymaps.cpp:9-32); the first one wins ties.  The reference
// narrows the separation to FLOAT before comparing, which decides near-ties: kept.
int getSnap(const std::vector<double> &zsnap, const CubicSpline &getDl, double dlens)
{
  int nearest = -1;
  double smallest = 99999;
  for (int i = 0; i < (int)zsnap.size(); i++)
  {
    const float separation = (float)std::abs(getDl.eval(zsnap[i]) - dlens);
    if (separation < smallest)
    {
      smallest = separation;
      nearest = i;
    }
  }
  return zsnap.empty() ? -1 : (nearest < 0 ? 0 : nearest);
}

// ---------------------------------------------------------------------------------------------------------------
// The light-cone plan (what densitymaps.cpp:46-156 computes).  Planes are stacked outwards from the observer; a plane is
// 1/numOfLensPerSnap of the box of the snapshot it is cut from.  For every new plane:
//   1. each snapshot from the current one on is tried as the source of the NEXT plane: the plane would end at
//      far_i = edge + box_i / L; the snapshot nearest to far_i in comoving distance is a candidate, scored by how far its
//      redshift is from z(far_i); inside a group of L planes only candidates with the current box size are allowed;
//   2. the winner fixes the plane's thickness; the plane is finally assigned to the snapshot nearest to its MIDDLE.
// `edge` is a running sum and every quotient is formed as box / (1e3 / POS_U) / L, as in the reference: the plane edges are
// part of the output contract (FITS keys DlLOW / DlUP, planes_list) and have to agree to the last bit.
// ---------------------------------------------------------------------------------------------------------------
namespace
{
struct PlanePlan
{
  double near_edge, far_edge; // comoving Mpc/h
  double z_mid;               // redshift of the plane's middle
  int snap;                   // index in the snapshot list
  bool new_group;             // first plane of a randomisation group
  int run_end;                // 1-based index of the last plane of this plane's run of equal snapshots
};

inline double slabThickness(double box, int lensPerSnap) { return box / (1e3 / POS_U) / lensPerSnap; }

std::vector<PlanePlan> planLightCone(const std::vector<double> &zsnap, const std::vector<double> &box, const CubicSpline &distOfZ,
                                     const CubicSpline &zOfDist, int lensPerSnap, double sourceDistance)
{
  std::vector<PlanePlan> plan;
  int current = 0; // snapshot of the previous plane
  double edge = 0.0;
  do
  {
    const int k = (int)plan.size(); // 0-based index of the plane being planned
    const bool opens_group = k % lensPerSnap == 0;
    int winner = current;
    double best = 9999;
    for (size_t i = (size_t)current; i < zsnap.size(); i++)
    {
      const double far_i = edge + slabThickness(box[i], lensPerSnap);
      const int cand = getSnap(zsnap, distOfZ, far_i);
      const double score = fabs(zsnap[cand] - zOfDist.eval(far_i));
      if (score < best && (opens_group || box[cand] == box[current]))
      {
        winner = cand;
        best = score;
      }
    }
    const double thick = slabThickness(box[winner], lensPerSnap);
    edge += thick;
    const double middle = edge - 0.5 * thick;
    PlanePlan pl;
    pl.snap = getSnap(zsnap, distOfZ, middle);
    pl.far_edge = edge;
    pl.near_edge = edge - slabThickness(box[pl.snap], lensPerSnap);
    pl.z_mid = zOfDist.eval(middle);
    pl.new_group = opens_group;
    pl.run_end = 0;
    plan.push_back(pl);
    current = pl.snap;
  } while (edge < sourceDistance);
  // runs of consecutive planes cut from the same snapshot: every plane remembers where its run ends
  for (size_t i = plan.size(); i-- > 0;)
    plan[i].run_end = (i + 1 < plan.size() && plan[i + 1].snap == plan[i].snap) ? plan[i + 1].run_end : (int)i + 1;
  return plan;
}
} // namespace

int buildPlanes(InputParams &p, Lens &lens, std::vector<double> &snapred, std::vector<std::string> &snappath,
                std::vector<double> &snapbox, const CubicSpline &getDl, const CubicSpline &getZl, int numOfLensPerSnap, int myid)
{
  if (snapred.empty())
  {
    std::cerr << "slicer-b200: the snapshot list is empty, there is nothing to plan" << std::endl;
    return 1;
  }
  const std::vector<PlanePlan> plan = planLightCone(snapred, snapbox, getDl, getZl, numOfLensPerSnap, p.Ds);
  const int total = (int)plan.size();
  for (const PlanePlan &pl : plan)
  {
    lens.ld.push_back(pl.near_edge);
    lens.ld2.push_back(pl.far_edge);
    lens.zsimlens.push_back(pl.z_mid);
    lens.zfromsnap.push_back(snapred[pl.snap]);
    lens.fromsnap.push_back(snappath[pl.snap]);
    lens.fromsnapi.push_back(pl.snap);
    lens.randomize.push_back(pl.new_group);
    lens.replication.push_back(pl.run_end);
    lens.pll.push_back((int)lens.pll.size());
  }
  lens.replication.push_back(total); // Lens.replication carries one entry more than there are planes (data.h:108); its last is nplanes
  lens.nplanes = total;
  if (myid != 0)
    return 0;
  std::cout << " light cone to " << p.Ds << " Mpc/h comoving: " << total << " planes from " << snapred.size() << " snapshots" << std::endl;
  for (int i = 0; i < total; i++)
  {
    const PlanePlan &pl = plan[i];
    std::cout << "   plane " << i << ": " << pl.near_edge << " - " << pl.far_edge << " Mpc/h, z = " << pl.z_mid << ", cut from " << snappath[pl.snap]
              << (pl.new_group ? "  [new randomisation]" : "") << std::endl;
  }
  writePlanesList(p, lens);
  return 0;
}

// planes_list_<suffix>.txt: one row per plane, columns as Lens/kslicer.py:29 reads them
//   index   z(middle)   near edge   far edge   last plane of the snapshot run   snapshot   z(snapshot)  first of a group
void writePlanesList(const InputParams &p, const Lens &lens)
{
  std::ofstream list((p.directory + "planes_list_" + p.suffix + ".txt").c_str());
  for (int i = 0; i < lens.nplanes; i++)
    list << i << "   " << lens.zsimlens[i] << "   " << lens.ld[i] << "   " << lens.ld2[i] << "   " << lens.replication[i] << "   " << lens.fromsnap[i]
         << "   " << lens.zfromsnap[i] << "  " << (bool)lens.randomize[i] << std::endl;
}

void GlibcRand::seed(unsigned int s)
{
  if (s == 0)
    s = 1;
  r_[0] = (int32_t)s;
  for (int i = 1; i < 31; i++)
  {
    const long hi = r_[i - 1] / 127773, lo = r_[i - 1] % 127773;
    long word = 16807 * lo - 2836 * hi;
    if (word < 0)
      word += 2147483647;
    r_[i] = (int32_t)word;
  }
  f_ = 3;
  b_ = 0;
  for (int i = 0; i < 310; i++)
    next();
}

int GlibcRand::next()
{
  const uint32_t v = (uint32_t)r_[f_] + (uint32_t)r_[b_];
  r_[f_] = (int32_t)v;
  f_ = f_ + 1 == 31 ? 0 : f_ + 1;
  b_ = b_ + 1 == 31 ? 0 : b_ + 1;
  return (int)(v >> 1);
}

GlibcRand &sharedRand()
{
  static GlibcRand g;
  return g;
}

// The randomisation of every group of planes (what densitymaps.cpp:166-248 draws with libc srand/rand; GlibcRand is the same
// generator with private state): three streams, re-seeded per group with seed + group * {13, 5, 8}: the box centre (three
// uniform draws), the axis permutation `face` in 1..6 (redrawn until in range) and the three mirror signs.  A uniform draw is
// rand() / float(RAND_MAX), a FLOAT division by 2147483648.f.  Planes inside a group inherit the group's values.
void randomizeBox(Random &random, const Lens &lens, const InputParams &p, int numOfLensPerSnap, int myid, bool fixedVertex)
{
  struct Draw
  {
    double centre[3];
    int face;
    int sign[3];
  };
  auto uniform = [](GlibcRand &g) { return g.next() / float(RAND_MAX); };
  const size_t count = lens.replication.back();
  std::vector<int> *const signs[3] = {&random.sgnX, &random.sgnY, &random.sgnZ};
  std::vector<double> *const centres[3] = {&random.x0, &random.y0, &random.z0};
  for (int k = 0; k < 3; k++)
  {
    signs[k]->assign(count, 0);
    centres[k]->assign(count, 0.0);
  }
  random.face.assign(count, 0);
  Draw d = {};
  for (size_t i = 0; i < count; i++)
  {
    if (lens.randomize[i])
    {
      GlibcRand &g = sharedRand();
      const unsigned group = (unsigned)(i / numOfLensPerSnap);
      g.seed(p.seedcenter + group * 13);
      for (int k = 0; k < 3; k++)
        d.centre[k] = fixedVertex ? (k == 2 ? 0.5 : 0.0) : (double)uniform(g); // -DFixedPLCVertex: the vertex sits on a box face
      g.seed(p.seedface + group * 5);
      do
        d.face = int(1 + uniform(g) * 5. + 0.5);
      while (d.face < 1 || d.face > 6);
      g.seed(p.seedsign + group * 8);
      for (int k = 0; k < 3; k++)
      {
        int bit;
        do
          bit = int(uniform(g) + 0.5);
        while (bit < 0 || bit > 1);
        d.sign[k] = bit ? 1 : -1;
      }
    }
    for (int k = 0; k < 3; k++)
    {
      (*centres[k])[i] = d.centre[k];
      (*signs[k])[i] = d.sign[k];
    }
    random.face[i] = d.face;
    if (myid == 0)
      std::cout << "   plane " << i << ": centre (" << d.centre[0] << ", " << d.centre[1] << ", " << d.centre[2] << "), axis permutation " << d.face
                << ", mirrors (" << d.sign[0] << ", " << d.sign[1] << ", " << d.sign[2] << ")" << std::endl;
  }
}

// The field must fit into one box at the far edge of the plane (densitymaps.cpp:255-269): fov [rad] * distance <= box.  As in the
// reference only rank 0 reports (and returns) the failure.
int testFov(double fov, double boxl, double Ds, int myid, double &fovradiants)
{
  fovradiants = fov / 180. * M_PI;
  const bool too_wide = fovradiants * Ds > boxl;
  if (too_wide && myid == 0)
  {
    std::cerr << "slicer-b200: a field of " << fov << " deg does not fit into the " << boxl << " Mpc/h box at " << Ds
              << " Mpc/h (at most " << boxl / Ds * 180. / M_PI << " deg); build with replication on the perpendicular plane for wider fields"
              << std::endl;
    return 1;
  }
  return 0;
}

// Box copies needed on either side, perpendicular to the line of sight, for the field at distance Ds (densitymaps.cpp:275-283)
void computeReplications(double fov, double boxl, double Ds, int, double &fovradiants, int &nrepperp)
{
  fovradiants = fov / 180. * M_PI;
  const double half_width = Ds * tan(fovradiants / 2.0);
  nrepperp = half_width <= boxl / 2.0 ? 0 : (int)ceil((Ds * tan(fovradiants / 2) - boxl / 2.0) / boxl);
}

} // namespace slicer
