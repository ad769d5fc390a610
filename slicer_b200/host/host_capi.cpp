// host_capi.cpp — C entry points over the C++ host layer, for the Python tests (ctypes).  Thin marshalling only.
#include "slicer_host.h"

#include <chrono>
#include <cstring>

using namespace slicer;

extern "C"
{

  int shost_cosmo_table(double om0, double oml, double w, double zs, double *zl, double *dl)
  {
    CosmoTable c;
    c.build(om0, oml, w, zs);
    for (int i = 0; i < neval; i++)
    {
      zl[i] = c.zl[i];
      dl[i] = c.dl[i];
    }
    return 0;
  }

  // slicer-v2.cpp:79-100 on caller-supplied snapshot redshifts / box sizes: mirrors oracle/ref_harness.cpp:ref_plan
  int shost_plan(double om0, double oml, double w, double zs, int nsnaps, const double *snapred_in, const double *snapbox_in,
                 const char *directory, const char *suffix, int cap, int *nplanes, double *Ds, double *ld, double *ld2, double *zsimlens,
                 double *zfromsnap, int *fromsnapi, int *randomize, int *replication, int *nreplication)
  {
    CosmoTable c;
    c.build(om0, oml, w, zs);
    InputParams p;
    p.zs = zs;
    p.directory = directory;
    p.suffix = suffix;
    p.Ds = c.getDl.eval(p.zs);
    *Ds = p.Ds;
    std::vector<double> snapred(snapred_in, snapred_in + nsnaps), snapbox(snapbox_in, snapbox_in + nsnaps);
    std::vector<std::string> snappath;
    for (int i = 0; i < nsnaps; i++)
      snappath.push_back("snap_" + std::to_string(i));
    Lens lens;
    if (buildPlanes(p, lens, snapred, snappath, snapbox, c.getDl, c.getZl, numberOfLensPerSnap, 0))
      return 1;
    *nplanes = lens.nplanes;
    *nreplication = (int)lens.replication.size();
    if ((int)lens.ld.size() > cap || (int)lens.replication.size() > cap)
      return 2;
    for (size_t i = 0; i < lens.ld.size(); i++)
    {
      ld[i] = lens.ld[i];
      ld2[i] = lens.ld2[i];
      zsimlens[i] = lens.zsimlens[i];
      zfromsnap[i] = lens.zfromsnap[i];
      fromsnapi[i] = lens.fromsnapi[i];
      randomize[i] = lens.randomize[i] ? 1 : 0;
    }
    for (size_t i = 0; i < lens.replication.size(); i++)
      replication[i] = lens.replication[i];
    return 0;
  }

  int shost_randomize_box(int seedcenter, int seedface, int seedsign, int nplanes, const int *randomize, int fixed_vertex, double *x0,
                          double *y0, double *z0, int *face, int *sx, int *sy, int *sz)
  {
    InputParams p;
    p.seedcenter = seedcenter;
    p.seedface = seedface;
    p.seedsign = seedsign;
    Lens lens;
    lens.replication.assign(1, nplanes);
    for (int i = 0; i < nplanes; i++)
      lens.randomize.push_back(randomize[i] != 0);
    Random r;
    randomizeBox(r, lens, p, numberOfLensPerSnap, 1, fixed_vertex != 0);
    for (int i = 0; i < nplanes; i++)
    {
      x0[i] = r.x0[i];
      y0[i] = r.y0[i];
      z0[i] = r.z0[i];
      face[i] = r.face[i];
      sx[i] = r.sgnX[i];
      sy[i] = r.sgnY[i];
      sz[i] = r.sgnZ[i];
    }
    return 0;
  }

  // n outputs of GlibcRand after seed(s) (tests compare with libc srand/rand)
  int shost_glibc_rand(unsigned int s, int n, int *out)
  {
    GlibcRand g;
    g.seed(s);
    for (int i = 0; i < n; i++)
      out[i] = g.next();
    return 0;
  }

  int shost_read_input(const char *file, int *ints /* npix, seedcenter, seedface, seedsign, partinplanes, snopt, physical, rgrid */,
                       double *dbl /* zs, fov, w */, char *strings /* 6 x 512: list, pathsnap, simulation, directory, suffix, snpix */)
  {
    InputParams p;
    if (readInput(p, file))
      return 1;
    ints[0] = p.npix;
    ints[1] = p.seedcenter;
    ints[2] = p.seedface;
    ints[3] = p.seedsign;
    ints[4] = p.partinplanes;
    ints[5] = p.snopt;
    ints[6] = p.physical;
    ints[7] = p.rgrid;
    dbl[0] = p.zs;
    dbl[1] = p.fov;
    dbl[2] = p.w;
    const std::string *s[6] = {&p.filredshiftlist, &p.pathsnap, &p.simulation, &p.directory, &p.suffix, &p.snpix};
    for (int i = 0; i < 6; i++)
      snprintf(strings + 512 * i, 512, "%s", s[i]->c_str());
    return 0;
  }

  // header + POS (+ masses) of one sub-file through the product's reader (pageable memory: no GPU needed)
  int shost_read_subfile(const char *file, int hydro, int *npart, double *massarr, double *scalars /* time,z,box,om0,oml,h */, int *numfiles,
                         float *pos, float *mass, long long cap)
  {
    SubFile s;
    if (readSubFile(file, hydro != 0, s, false))
      return 1;
    for (int i = 0; i < 6; i++)
    {
      npart[i] = s.header.npart[i];
      massarr[i] = s.header.massarr[i];
    }
    scalars[0] = s.header.time;
    scalars[1] = s.header.redshift;
    scalars[2] = s.header.boxsize;
    scalars[3] = s.header.om0;
    scalars[4] = s.header.oml;
    scalars[5] = s.header.h;
    *numfiles = s.header.numfiles;
    if ((long long)s.ntotal > cap)
      return 2;
    if (pos)
      memcpy(pos, s.pos, s.ntotal * 12);
    if (mass && s.mass)
      memcpy(mass, s.mass, s.ntotal * 4);
    return 0;
  }

  // measurement aid (tools/probe_reader.py): best wall time of `repeats` readSubFile calls into one (pinned) buffer
  int shost_time_read_subfile(const char *file, int hydro, int pinned, int repeats, double *best_seconds, long long *bytes)
  {
    SubFile s;
    *best_seconds = 1e30;
    for (int r = 0; r < repeats; r++)
    {
      const auto t0 = std::chrono::steady_clock::now();
      if (readSubFile(file, hydro != 0, s, pinned != 0))
        return 1;
      const double dt = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
      if (dt < *best_seconds)
        *best_seconds = dt;
    }
    *bytes = (long long)s.ntotal * 12;
    return 0;
  }

  int shost_write_fits(const char *file, const float *map, int npix, int nd, const char **dnames, const double *dvals, int ni, const char **inames,
                       const long long *ivals)
  {
    std::vector<std::pair<std::string, double>> d;
    std::vector<std::pair<std::string, long long>> k;
    std::vector<std::string> order;
    for (int i = 0; i < nd; i++)
    {
      d.push_back({dnames[i], dvals[i]});
      order.push_back(dnames[i]);
    }
    for (int i = 0; i < ni; i++)
    {
      k.push_back({inames[i], ivals[i]});
      order.push_back(inames[i]);
    }
    try
    {
      writeFitsImage(file, map, npix, d, k, order);
    }
    catch (const SliceError &)
    {
      return 1;
    }
    return 0;
  }

  int shost_run_light_cone(const char *ini, const int *devices, int ndev, int replication, int fixed_vertex, int ngp, int deposit_mode)
  {
    RunOptions o;
    o.devices.assign(devices, devices + ndev);
    o.replication = replication != 0;
    o.fixed_vertex = fixed_vertex != 0;
    o.mas = ngp ? SLICER_MAS_NGP : SLICER_MAS_TSC;
    o.deposit_mode = deposit_mode;
    o.quiet = true;
    return runLightCone(ini, o);
  }

  // one light cone per ini, every snapshot read once for all (runLightCones)
  int shost_run_light_cones(const char **inis, int nini, const int *devices, int ndev, int replication, int fixed_vertex, int ngp,
                            int deposit_mode, int max_slots)
  {
    RunOptions o;
    o.devices.assign(devices, devices + ndev);
    o.replication = replication != 0;
    o.fixed_vertex = fixed_vertex != 0;
    o.mas = ngp ? SLICER_MAS_NGP : SLICER_MAS_TSC;
    o.deposit_mode = deposit_mode;
    o.quiet = true;
    o.max_slots = max_slots;
    return runLightCones(std::vector<std::string>(inis, inis + nini), o);
  }
}
