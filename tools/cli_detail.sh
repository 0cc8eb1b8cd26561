#!/bin/bash
# Phase detail of the command line on the benchmark's FASTQ files (bench.py writes them to /dev/shm/kb_bench_cache):
# KB_CLI_TIMING=2 prints every phase and round; `strace -c`-free, just wall clocks.  Usage: tools/cli_detail.sh [devices]
D=$(ls -d /dev/shm/kb_bench_cache/g62000_p2000000_k*_L100 | head -1)
IDX=$(python -c 'import bench; print(bench.DATA)')/g62000.kidx
DEV=${1:-0}
for i in 1 2 ${KB_DETAIL_REPS:-3}; do
  S=$(date +%s%N)
  if [[ "$DEV" == *,* ]]; then A="--devices $DEV"; else A="--device $DEV"; fi
  KB_CLI_TIMING=1 kallisto_b200/kallisto_b200 quant -i $IDX -o $D/cli_detail_out --plaintext -t 64 $A $D/r_1.fq $D/r_2.fq 2>&1 | grep -a "timing\|processed"
  E=$(date +%s%N)
  echo "process wall: $(python3 -c "print(($E-$S)/1e9)") s"
done
