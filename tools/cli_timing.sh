#!/bin/bash
# Phase timing of the CLI on the bench workload (needs the benchmark's index, built by a bench.py run on the same machine)
python - <<'PY'
import sys, os, numpy as np
sys.path.insert(0, '.')
import bench, benchdata, torch
idx, concat, lens = bench.workload(62000)
sim = benchdata.TorchSimulator(concat, lens, "cuda:0", read_len=100)
for c0 in range(0, 8000000, 1000000):
    r = sim.pairs(1000000, seed=5000 + c0).cpu().numpy()
    benchdata.write_fastq_fast('/dev/shm/c_1.fq', r[:, 0], 1, append=c0 > 0)
    benchdata.write_fastq_fast('/dev/shm/c_2.fq', r[:, 1], 2, append=c0 > 0)
benchdata.write_fastq_fast('/dev/shm/t_1.fq', r[:1, 0], 1)
benchdata.write_fastq_fast('/dev/shm/t_2.fq', r[:1, 1], 2)
PY
for t in 64 8 2; do
  echo "== -t $t"
  KB_CLI_TIMING=2 KB_FASTX_DEBUG=1 kallisto_b200/kallisto_b200 quant -i $(python -c 'import bench; print(bench.DATA)')/g62000.kidx -o /dev/shm/o1 --plaintext -t $t /dev/shm/c_1.fq /dev/shm/c_2.fq 2>&1 | grep -E "timing|fastx|processed"
done
echo "== one pair"
KB_CLI_TIMING=1 kallisto_b200/kallisto_b200 quant -i $(python -c 'import bench; print(bench.DATA)')/g62000.kidx -o /dev/shm/o2 --plaintext -t 64 /dev/shm/t_1.fq /dev/shm/t_2.fq 2>&1 | grep -E "timing"
