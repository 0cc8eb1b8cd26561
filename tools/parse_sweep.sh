#!/bin/bash
# Ingest A/B of the command line on the benchmark's 40 M-pair FASTQ files: parser threads per file (KB_FASTX_CAP) x copy
# threads (KB_FASTX_COPY).  Prints the read + pseudoalign loop phase and the process wall clock per configuration.
python - <<'PY'
import sys, os
sys.path.insert(0, os.getcwd())
import torch, bench, benchdata
idx, concat, lens = bench.workload(62000)
bench.fastq_job_files(62000, 2000000, 20, 5, lambda: benchdata.TorchSimulator(concat, lens, "cuda:0", read_len=100))
PY
D=$(ls -d /dev/shm/kb_bench_cache/g62000_p2000000_k20_w5_L100 | head -1)
IDX=$(python -c 'import bench; print(bench.DATA)')/g62000.kidx
python - <<'PY' &
import torch, time
torch.zeros(1, device="cuda")      # keeps the GPU initialised, as the benchmark's parent process does
time.sleep(600)
PY
HOLD=$!
sleep 8
for cfg in "16 4" "16 8" "24 8" "32 8" "32 16" "48 16"; do
  set -- $cfg
  for rep in 1 2; do
    S=$(date +%s%N)
    L=$(KB_FASTX_CAP=$1 KB_FASTX_COPY=$2 KB_CLI_TIMING=1 kallisto_b200/kallisto_b200 quant -i $IDX -o $D/sweep_out --plaintext -t 128 --device 0 $D/r_1.fq $D/r_2.fq 2>&1 | grep -a "read + pseudoalign loop\|index load:" | tr '\n' ' ')
    E=$(date +%s%N)
    echo "cap=$1 copy=$2 wall=$(python3 -c "print(($E-$S)/1e9)") $L"
  done
done
kill $HOLD
