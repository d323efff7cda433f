#!/bin/bash
# Before / after of the fast-path cut in one call: the former cut (sin^2(phi/3) >= 1.4e-6) and the current one, same
# code otherwise, alternated three times.  Builds the two variants if they are missing (scratch/build_variant.sh).
# scratch/cut_cost.sh [output directory, default scratch/variants]: the log is <dir>/cut_cost.log.
set -e
cd "$(dirname "$0")/.."
out=${1:-scratch/variants}
mkdir -p scratch/variants "$out"
[ -f scratch/variants/lib_cut_old.so ] || scratch/build_variant.sh cut_old -DGFP_FAST_MIN_SIN2=1.4e-6
[ -f scratch/variants/lib_cut_new.so ] || scratch/build_variant.sh cut_new
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv,noheader | tee "$out/cut_cost.log"
for rep in 1 2 3; do
  for v in cut_old cut_new; do
    GOLEMFLAVOR_B200_LIB=scratch/variants/lib_$v.so python scratch/cut_cost.py | tee -a "$out/cut_cost.log"
  done
done
