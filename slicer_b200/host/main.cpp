// SLICER_b200 — same command line as the reference (README.md:80-84):   SLICER_b200 InputParams.ini
// Several ini files make one light cone each (realisations that differ in seeds and output), with one read of every snapshot:
//   SLICER_b200 [switches] A.ini B.ini C.ini ...
// Optional switches stand in for the reference's compile-time options:
//   --gpus 0,1,..      GPUs of this process that share the sub-files (default 0; in a job of several processes the local
//                      rank modulo the visible GPUs)                                   [MPI ranks, slicer-v2.cpp:28-30]
//   --replication      CMake USE_REPLICATION   (-DReplicationOnPerpendicularPlane, CMakeLists.txt:20-22)
//   --fixed-vertex     CMake USE_FIXED_PLC_VERTEX (-DFixedPLCVertex, CMakeLists.txt:23-26)
//   --ngp              `#define DO_NGP true`   (densitymaps.h:22)
//   --max-slots N      at most N plane accumulators per GPU (device memory; default: what the inis' planes of a snapshot need)
//   --kappa            also write a convergence map per light cone for the ini's source redshift (entry 2), formed on the GPU
//   --kappa-zs z1,z2,..  the same for up to 8 source redshifts in (0, entry 2] (implies --kappa)
//   --no-planes        write the convergence maps only (and planes_list), no plane FITS files
//   --shear            also write the shear maps γ1, γ2 of every convergence map (Kaiser–Squires on the GPU; alone: implies --kappa)
// Started by a launcher (mpirun -np N, srun, torchrun), the processes form one job: rank and world size come from the launcher's
// environment (slicer::launchFromEnv), MASTER_ADDR / MASTER_PORT name where rank 0 listens for the others, the sub-files of every
// snapshot are dealt over the GPUs of all ranks and rank 0 writes the planes.
#include "slicer_host.h"

#include <cmath>
#include <cstdlib>
#include <cstring>
#include <iostream>

int main(int argc, char **argv)
{
  slicer::RunOptions opt;
  slicer::Launch launch;
  std::string err;
  if (slicer::launchFromEnv([](const char *name) -> const char * { return getenv(name); }, launch, err))
  {
    std::cerr << err << std::endl;
    return 255;
  }
  opt.rank = launch.rank;
  opt.nranks = launch.nranks;
  opt.master_addr = launch.master_addr;
  opt.master_port = launch.master_port;
  bool gpus_given = false, kappa_ini = false;
  std::vector<std::string> inis;
  for (int i = 1; i < argc; i++)
  {
    if (!strcmp(argv[i], "--gpus") && i + 1 < argc)
    {
      gpus_given = true;
      opt.devices.clear();
      for (char *t = strtok(argv[++i], ","); t; t = strtok(nullptr, ","))
        opt.devices.push_back(atoi(t));
    }
    else if (!strcmp(argv[i], "--replication"))
      opt.replication = true;
    else if (!strcmp(argv[i], "--fixed-vertex"))
      opt.fixed_vertex = true;
    else if (!strcmp(argv[i], "--ngp"))
      opt.mas = SLICER_MAS_NGP;
    else if (!strcmp(argv[i], "--quiet"))
      opt.quiet = true;
    else if (!strcmp(argv[i], "--max-slots") && i + 1 < argc)
      opt.max_slots = atoi(argv[++i]);
    else if (!strcmp(argv[i], "--kappa"))
      kappa_ini = true;
    else if (!strcmp(argv[i], "--kappa-zs") && i + 1 < argc)
    {
      for (char *t = strtok(argv[++i], ","); t; t = strtok(nullptr, ","))
      {
        char *end = nullptr;
        const double z = strtod(t, &end);
        if (end == t || *end)
        {
          std::cerr << "--kappa-zs: '" << t << "' is not a number" << std::endl;
          return 1;
        }
        opt.kappa_zs.push_back(z);
      }
    }
    else if (!strcmp(argv[i], "--no-planes"))
      opt.write_planes = false;
    else if (!strcmp(argv[i], "--shear"))
      opt.shear = true;
    else
      inis.push_back(argv[i]);
  }
  if (kappa_ini && opt.kappa_zs.empty())
    opt.kappa_zs.push_back(std::nan("")); // the ini's source redshift
  if (inis.empty())
  {
    std::cerr << "usage: SLICER_b200 [--gpus 0,1,..] [--replication] [--fixed-vertex] [--ngp] [--quiet] [--max-slots N] [--kappa | --kappa-zs z1,z2,..]\n"
                 "                   [--shear] [--no-planes] InputParams.ini [more.ini ...]\n"
                 "  one light cone per ini; the inis must agree on everything but the seeds (entries 7-9), the simulation name and\n"
                 "  the output directory and suffix (entries 6, 11, 12), and at most one may set a particle degradation.\n"
                 "  --kappa writes a convergence map per light cone for the source redshift of entry 2 (--kappa-zs: for up to 8 others),\n"
                 "  --shear also the shear maps gamma1, gamma2 of each (alone: of the source redshift of entry 2), --no-planes only\n"
                 "  those maps"
              << std::endl;
    return 1;
  }
  if (opt.nranks > 1 && !gpus_given)
  {
    int ndev = 0;
    if (slicer_device_count(&ndev) || ndev < 1)
    {
      std::cerr << "rank " << opt.rank << ": no CUDA device: " << slicer_last_error() << std::endl;
      return 255;
    }
    opt.devices = {slicer::defaultDevice(launch, ndev)};
  }
  return slicer::runLightCones(inis, opt) ? 255 : 0; // the reference ends in MPI_Abort(-1) on every error
}
