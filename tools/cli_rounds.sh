#!/bin/bash
# Where does the read + pseudoalign loop of the CLI spend its time?  KB_CLI_TIMING=2 prints, per round, the time inside
# kb_pseudoalign_batch_pe (offset scan + H2D copies, waits for the copy) and the wall clock; the rest of a round is
# waiting for the parser.  Needs the benchmark's FASTQ files (bench.py / tools/parse_sweep.sh write them).
D=$(ls -d /dev/shm/kb_bench_cache/g62000_p2000000_k20_w5_L100 | head -1)
KB_CLI_TIMING=2 kallisto_b200/kallisto_b200 quant -i $(python -c 'import bench; print(bench.DATA)')/g62000.kidx -o $D/rounds_out --plaintext -t 64 --device 0 $D/r_1.fq $D/r_2.fq 2>&1 | grep -a "timing" > /tmp/rounds.log
python3 - <<'PY'
import re
calls=[]; ats=[]
for l in open('/tmp/rounds.log', errors='replace'):
    m=re.search(r"round of (\d+) reads: call ([0-9.e+-]+) s, at ([0-9.e+-]+) s", l)
    if m: calls.append(float(m.group(2))); ats.append(float(m.group(3)))
    elif 'index load:' in l or 'read + pseudoalign loop' in l: print(l.strip())
if calls:
    span=ats[-1]-ats[0]+calls[0]
    print("rounds %d, sum of call times %.3f s, span of the loop %.3f s -> %.0f %% of the loop inside the batch call (copy), the rest waiting for the parser" % (len(calls), sum(calls), span, 100*sum(calls)/span))
    print("call time per round: min %.4f median %.4f max %.4f s" % (min(calls), sorted(calls)[len(calls)//2], max(calls)))
PY
