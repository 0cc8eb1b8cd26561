#!/bin/bash
# Parser-side accounting of the CLI's read loop (KB_FASTX_DEBUG=1: per input file, time spent parsing windows and time the
# reader waited for a parsed window).  Needs the benchmark's FASTQ files.
D=$(ls -d /dev/shm/kb_bench_cache/g62000_p2000000_k20_w5_L100 | head -1)
for cfg in "16 4" "32 8"; do set -- $cfg
  echo "== KB_FASTX_CAP=$1 KB_FASTX_COPY=$2"
  KB_FASTX_CAP=$1 KB_FASTX_COPY=$2 KB_FASTX_DEBUG=1 KB_CLI_TIMING=1 KB_CLI_CLEANUP=1 kallisto_b200/kallisto_b200 quant -i $(python -c 'import bench; print(bench.DATA)')/g62000.kidx -o $D/dbg_out --plaintext -t 64 --device 0 $D/r_1.fq $D/r_2.fq 2>&1 | grep -a "fastx\]\|read + pseudoalign loop"
done
