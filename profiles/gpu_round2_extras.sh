#!/bin/bash
# Round-2 side measurements: N = 64 comb throughput vs batch size,
# clock64() phase timing of the new kernel, DFMA issue rate of a lone warp.
set -u
OUT=gpurun_out
mkdir -p $OUT
python tools/comb_bench.py 592 1024 2368 4736 9472 18944 2>&1 | tail -7 > $OUT/r2_comb_bench.txt
python tools/comb_phase_timing.py 2>&1 | grep -v "^$" | tail -12 > $OUT/r2_comb8_phase_cycles.txt
nvcc -gencode arch=compute_100a,code=sm_100a -O3 -o /tmp/dfma_warp_probe.bin tools/dfma_warp_probe.cu && /tmp/dfma_warp_probe.bin > $OUT/r2_dfma_warp_probe.txt
cat $OUT/r2_comb_bench.txt $OUT/r2_comb8_phase_cycles.txt
