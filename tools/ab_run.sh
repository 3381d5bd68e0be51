#!/bin/bash
# Developer tool (GPU box): timing of the k_viterbi2 variants built by tools/build_variants.sh (one process each).
#   tools/ab_run.sh "variant[:layout]" ...     -> gpurun_out/ab.txt
cd "$(dirname "$0")/.."
R=$PWD/vibrato_b200
out=gpurun_out/ab.txt; : > $out
for cfg in "$@"; do
  v="${cfg%%:*}"; l=1; [[ "$cfg" == *:* ]] && l="${cfg#*:}"
  VBT_SWEEP_TAG="$v/L$l" VBT_MATRIX_LAYOUT=$l VBT_SO=$R/libvibrato_b200_$v.so python tools/sweep.py synth-unidic 1000000 2>&1 | grep lanes >> $out
done
cat $out
