#!/bin/bash
# Builds tuning variants of libbp5b200.so (cells per tile, row chunking, ...) into build/tune/<name>/
# usage: scripts/tune_cpt.sh   (then run scripts/gpu_perf_probe.py with BP5_LIB=build/tune/<name>/libbp5b200.so)
set -e
ROOT=$(cd "$(dirname "$0")/.." && pwd)
CS=$ROOT/deal-and-ceed-on-gpu_b200/csrc
# the library's other objects as the Makefile lists them (build them first: make -C $CS)
OBJS=$(make -s -C $CS -pn | sed -n 's/^OBJS := //p' | sed 's/\bapply\.o\b//')
declare -A SETS
SETS[S3]="-DBP5_CPT_P7=3"
SETS[S2]="-DBP5_CPT_P7=2"
for name in "${!SETS[@]}"; do
  out=$ROOT/build/tune/$name; mkdir -p $out
  ( cd $CS && /usr/local/cuda/bin/nvcc -gencode arch=compute_100a,code=sm_100a -O3 -std=c++17 -lineinfo -Xcompiler -fPIC -ccbin /usr/bin/g++ ${SETS[$name]} -c apply.cu -o $out/apply.o \
    && /usr/local/cuda/bin/nvcc -gencode arch=compute_100a,code=sm_100a -shared -o $out/libbp5b200.so $out/apply.o $OBJS -ccbin /usr/bin/g++ ) &
done
wait
ls -la $ROOT/build/tune/*/libbp5b200.so
