#!/bin/bash
# Build a variant of the library into scratch/variants/lib_<name>.so with extra nvcc flags: scratch/build_variant.sh <name> [-DFLAG ...]
set -e
cd "$(dirname "$0")/.."
name=$1; shift
nvcc -O3 -std=c++17 --threads 4 -gencode arch=compute_100a,code=sm_100a -lineinfo -Xcompiler -fPIC -shared -Xlinker -soname=libgolemflavor_b200.so "$@" \
  -o scratch/variants/lib_$name.so golemflavor_b200/csrc/gf_api.cu golemflavor_b200/csrc/gf_lnprob.cu golemflavor_b200/csrc/gf_scan.cu golemflavor_b200/csrc/gf_ensemble.cu golemflavor_b200/csrc/gf_profile.cu golemflavor_b200/csrc/gf_sources.cu
echo built scratch/variants/lib_$name.so
