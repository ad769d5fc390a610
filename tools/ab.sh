#!/bin/bash
# measurement aid: A/B two builds of the CUDA library in ONE gpurun call (same box, same clocks).
#   tools/ab.sh "<nvcc flags of A>" "<nvcc flags of B>" [PGROUPS, default 0,2,4,8]
# e.g. tools/ab.sh "" "-DSLICER_CHECKS"      (A = the default build, B = the build with device-side bounds checks)
# Builds slicer_b200/_build/libslicer_b200_{a,b}.so here, then runs tools/probe_groups.py twice per variant on the GPU box.
set -e
HERE="$(cd "$(dirname "$0")/.." && pwd)"
make -s -C "$HERE/slicer_b200/csrc" variant NAME=a EXTRA="$1"
make -s -C "$HERE/slicer_b200/csrc" variant NAME=b EXTRA="$2"
G="${3:-0,2,4,8}"
/usr/local/graft/bin/gpurun --timeout 900 -- "for r in 1 2; do for v in a b; do echo variant \$v; SLICER_B200_LIB=\$PWD/slicer_b200/_build/libslicer_b200_\$v.so PGROUPS=$G python tools/probe_groups.py; done; done" 2>&1 | grep -v '^\[gpurun\] sending'
rm -f "$HERE/slicer_b200/_build/libslicer_b200_a.so" "$HERE/slicer_b200/_build/libslicer_b200_b.so"
