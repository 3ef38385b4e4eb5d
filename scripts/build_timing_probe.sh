#!/bin/bash
# Builds deepflows_b200/lib/tc_timing_probe.bin: the library sources compiled with -DDFB_TC_TIMING plus
# scripts/tc_timing_probe.cu, statically in one executable (the shipped libdfb200.so is untouched).
set -e
cd "$(dirname "$0")/.."
out=deepflows_b200/lib/obj_timing
mkdir -p $out
flags="-gencode arch=compute_100a,code=sm_100a -lineinfo -O3 -std=c++17 --expt-relaxed-constexpr -DDFB_TC_TIMING"
pids=()
for f in runtime ewise gemm_simt gemm_tc conv_direct gemm nn_ops data_ops optim comm peer; do
  if [ ! -f $out/$f.o ] || [ deepflows_b200/csrc/$f.cu -nt $out/$f.o ] || [ "$f" = gemm_tc ]; then
    nvcc $flags -c deepflows_b200/csrc/$f.cu -o $out/$f.o &
    pids+=($!)
  fi
done
for p in "${pids[@]}"; do wait $p; done
nvcc $flags scripts/tc_timing_probe.cu $out/*.o -o deepflows_b200/lib/tc_timing_probe.bin -cudart static -ldl
echo built deepflows_b200/lib/tc_timing_probe.bin
