// SLICER_b200 — same command line as the reference (README.md:80-84):   SLICER_b200 InputParams.ini
// Several ini files make one light cone each (realisations that differ in seeds and output), with one read of every snapshot:
//   SLICER_b200 [switches] A.ini B.ini C.ini ...
// Optional switches stand in for the reference's compile-time options:
//   --gpus 0,1,..      GPUs of this box that share the sub-files (default 0)        [MPI ranks, slicer-v2.cpp:28-30]
//   --replication      CMake USE_REPLICATION   (-DReplicationOnPerpendicularPlane, CMakeLists.txt:20-22)
//   --fixed-vertex     CMake USE_FIXED_PLC_VERTEX (-DFixedPLCVertex, CMakeLists.txt:23-26)
//   --ngp              `#define DO_NGP true`   (densitymaps.h:22)
//   --max-slots N      at most N plane accumulators per GPU (device memory; default: what the inis' planes of a snapshot need)
#include "slicer_host.h"

#include <cstring>
#include <iostream>

int main(int argc, char **argv)
{
  slicer::RunOptions opt;
  std::vector<std::string> inis;
  for (int i = 1; i < argc; i++)
  {
    if (!strcmp(argv[i], "--gpus") && i + 1 < argc)
    {
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
    else
      inis.push_back(argv[i]);
  }
  if (inis.empty())
  {
    std::cerr << "usage: SLICER_b200 [--gpus 0,1,..] [--replication] [--fixed-vertex] [--ngp] [--quiet] [--max-slots N] InputParams.ini [more.ini ...]\n"
                 "  one light cone per ini; the inis must agree on everything but the seeds (entries 7-9), the simulation name and\n"
                 "  the output directory and suffix (entries 6, 11, 12), and at most one may set a particle degradation"
              << std::endl;
    return 1;
  }
  return slicer::runLightCones(inis, opt) ? 255 : 0; // the reference ends in MPI_Abort(-1) on every error
}
