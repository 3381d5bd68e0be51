#!/bin/bash
# Developer tool: builds kernel variants as extra shared objects (vibrato_b200/libvibrato_b200_<name>.so) for A/B runs
# with tools/ab_multi.py.      tools/build_variants.sh "name:-DFLAG=..,-DFLAG2=.." ...
set -e
cd "$(dirname "$0")/../vibrato_b200/csrc"
make -s all
for spec in "$@"; do
  name="${spec%%:*}"; flags="${spec#*:}"; flags="${flags//,/ }"
  /usr/local/cuda/bin/nvcc -gencode arch=compute_100a,code=sm_100a -lineinfo -O3 -std=c++17 -Xcompiler -fPIC \
      -Xptxas -v --expt-relaxed-constexpr $flags -c kernels.cu -o /tmp/kernels_$name.o 2> /tmp/kernels_$name.log
  /usr/local/cuda/bin/nvcc -gencode arch=compute_100a,code=sm_100a -shared -o ../libvibrato_b200_$name.so \
      host_dict.o device_blob.o capi.o engine.o multi_engine.o evaluate.o /tmp/kernels_$name.o -cudart static -ldl
  echo "$name: $(grep -A2 'k_viterbi2ILi0ELb1ELb0E' /tmp/kernels_$name.log | grep -E 'spill|Used' | tr -s ' ' | tr '\n' ' ')"
done
