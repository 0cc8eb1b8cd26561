#!/usr/bin/env python
"""bench.py -- paired reads/s of the `kallisto quant` hot path on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--dump-outputs DIR]

Workload (config.workload): BASELINE config 2 -- a human-GENCODE-v44-like transcriptome index
(built by the unmodified reference `kallisto index`, k=31; synthetic stand-in, see benchdata.py)
and synthetic 2x100 bp paired reads.  One step = one batch of `pairs_per_step` read pairs through
pseudoalignment (k-mer probes + EC intersection + EC counting); after the K timed steps the EC
table is finalised and the EM is run ONCE, inside the timed region (it is part of the job).
  value  = K * pairs_per_step * N / time, reads resident in HBM before the timed region starts (the job
           is run once untimed, then timed twice: the second timed run is reported, both are listed);
  e2e    = the same reads as FASTQ files through the drop-in command line `kallisto_b200 quant` ->
           abundance.tsv: pairs / process wall clock (median of three runs), index load included (SURVEY.md 8d); the pinned-
           host-buffer figure of the C ABI is listed under config.pinned_host_buffers;
  roofline  = match_kernel: algorithmic bytes (SURVEY.md 8d / DESIGN.md) / CUDA-event time, vs
           MEASURED_PEAKS.json hbm_gbs;
  --impl reference = oracle/_ref/kallisto (the unmodified reference, built from its sources by
           oracle/Makefile) `quant -t <best>` on the SAME FASTQ files (all K x P pairs of rank 0's job, one
           run, process wall clock); cpu_baseline = that run when it happened on this box, else a 2 M-pair sample.
  --dump-outputs DIR = what the reported timed job returned to its caller, as DIR/<name>.npy (float64): est_counts,
           eff_lens, em_rounds, the fragment-length histogram and the EC table (counts, set sizes, transcript ids;
           arrays longer than 2^20 are replaced by a fixed seeded sample of 2^20 entries, < 64 MB in all).  The inputs
           are pure functions of the arguments, so two builds can be compared output for output.
Every step uses different reads and each batch (pairs_per_step x 200 B) is larger than L2.
The index, the transcriptome and the FASTQ files are cached in temporary directories, never in the source tree.
"""
import argparse
import json
import os
import re
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
import benchdata  # noqa: E402

DATA = os.path.join(tempfile.gettempdir(), "kallisto_b200_bench_data_%d" % os.getuid())
READ_LEN = 100


def log(*a):
    print("[bench]", *a, file=sys.stderr, flush=True)


# ---------------------------------------------------------------------------------------------
# workload: index + transcriptome (cached under DATA, rebuilt with the reference if absent)
# ---------------------------------------------------------------------------------------------
def workload(genes):
    import fcntl
    os.makedirs(DATA, exist_ok=True)
    idx = os.path.join(DATA, "g%d.kidx" % genes)
    txf = os.path.join(DATA, "g%d.tx.npz" % genes)
    with open(os.path.join(DATA, ".lock"), "w") as lockf:   # ranks of one node: one builds, the others wait
        fcntl.flock(lockf, fcntl.LOCK_EX)
        try:
            _build_workload(genes, idx, txf)
        finally:
            fcntl.flock(lockf, fcntl.LOCK_UN)
    z = np.load(txf)
    packed, lens = z["packed"], z["lens"]
    concat = np.empty(len(packed) * 4, np.uint8)
    lut = np.frombuffer(b"ACGT", np.uint8)
    for j in range(4):
        concat[j::4] = lut[(packed >> (2 * j)) & 3]
    concat = concat[: int(lens.sum())]
    return idx, concat, lens


def _build_workload(genes, idx, txf):
    if not (os.path.exists(idx) and os.path.exists(txf)):
        from oracle import oracle as O
        log("building workload for %d genes (one-off, cached in %s)" % (genes, DATA))
        t0 = time.time()
        tx = benchdata.make_transcriptome(genes, seed=44)
        codes = np.zeros(256, np.uint8)
        for i, c in enumerate(b"ACGT"):
            codes[c] = i
        c = codes[tx.concat]
        pad = (-len(c)) % 4
        c = np.concatenate([c, np.zeros(pad, np.uint8)]).reshape(-1, 4)
        packed = (c[:, 0] | (c[:, 1] << 2) | (c[:, 2] << 4) | (c[:, 3] << 6)).astype(np.uint8)
        np.savez(txf + ".tmp.npz", packed=packed, lens=tx.lens)
        os.replace(txf + ".tmp.npz", txf)
        if not os.path.exists(idx):     # oracle/_ref/kallisto is built by __graft_entry__.build(), not here: the tree may be read-only
            with tempfile.TemporaryDirectory(dir=DATA) as td:
                fa = os.path.join(td, "tx.fa")
                tx.write_fasta(fa)
                # -T: the reference's scratch directory defaults to ./tmp, and the working directory may be read-only
                O.ref_run(["index", "-t", str(min(32, os.cpu_count() or 8)), "-T", os.path.join(td, "tmp"), "-i", idx + ".tmp", fa])
            os.replace(idx + ".tmp", idx)
        log("workload built in %.0f s" % (time.time() - t0))


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.rows = []
        self.p = None

    def start(self):
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q,
                                       "--format=csv,noheader,nounits", "-lms", "20"], stdout=subprocess.PIPE,
                                      stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.p = None

    def _read(self):
        for line in self.p.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if not self.p:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.p.terminate()
        try:
            self.p.wait(timeout=2)
        except Exception:
            self.p.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            a = [x.strip() for x in r.split(",")]
            if len(a) < 9:
                continue
            try:
                sm.append(float(a[1]))
                mx.append(float(a[2]))
            except ValueError:
                continue
            for nm, v in zip(names, a[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


CACHE_ROOT = os.path.join("/dev/shm" if os.path.isdir("/dev/shm") else DATA, "kb_bench_cache")


def job_seeds(rank, W, K):
    """Seeds of the K timed batches of `rank` (the W warm-up batches use the seeds before them)."""
    return [1000 + rank * 100003 + s for s in range(W, W + K)]


def fastq_job_files(genes, P, K, W, sim_factory):
    """FASTQ files of rank 0's timed job (K batches of P pairs, plain text, in shared memory), shared by the
    reference arm and our arm through a cache directory: both arms run back to back on the same box, and both
    derive the reads from the same seeds anyway.  -> (dir, r1, r2, sample1, sample2, tiny1, tiny2)"""
    import fcntl
    import torch
    key = "g%d_p%d_k%d_w%d_L%d" % (genes, P, K, W, READ_LEN)
    d = os.path.join(CACHE_ROOT, key)
    os.makedirs(d, exist_ok=True)
    f1, f2 = os.path.join(d, "r_1.fq"), os.path.join(d, "r_2.fq")
    s1, s2 = os.path.join(d, "sample_1.fq"), os.path.join(d, "sample_2.fq")
    t1, t2 = os.path.join(d, "tiny_1.fq"), os.path.join(d, "tiny_2.fq")
    done = os.path.join(d, "complete")
    with open(os.path.join(d, ".lock"), "w") as lockf:
        fcntl.flock(lockf, fcntl.LOCK_EX)
        try:
            if not os.path.exists(done):
                t0 = time.time()
                sim = sim_factory()
                for f in (f1, f2):
                    open(f, "wb").close()
                for j, seed in enumerate(job_seeds(0, W, K)):
                    reads = sim.pairs(P, seed=seed)
                    for f, m in ((f1, 0), (f2, 1)):
                        img = benchdata.fastq_image(reads[:, m], m + 1, j * P)
                        with open(f, "ab") as fh:
                            img.cpu().numpy().tofile(fh)
                    if j == 0:
                        n_s = min(P, 2000000)
                        for f, m in ((s1, 0), (s2, 1)):
                            benchdata.fastq_image(reads[:n_s, m], m + 1, 0).cpu().numpy().tofile(f)
                        for f, m in ((t1, 0), (t2, 1)):
                            benchdata.fastq_image(reads[:1, m], m + 1, 0).cpu().numpy().tofile(f)
                    del reads
                if torch.cuda.is_available():
                    torch.cuda.empty_cache()
                open(done, "w").write("%d pairs\n" % (K * P))
                log("FASTQ of the timed job (%d pairs, %.1f GB) written to %s in %.0f s" % (
                    K * P, (os.path.getsize(f1) + os.path.getsize(f2)) / 1e9, d, time.time() - t0))
        finally:
            fcntl.flock(lockf, fcntl.LOCK_UN)
    return d, f1, f2, s1, s2, t1, t2


def cli_run(idx, files, n_pairs, devices, outdir, repeats=3):
    """File to file through the drop-in command line: `kallisto_b200 quant` (csrc/cli_main.cpp) on plain FASTQ in
    shared memory -> abundance.tsv + run_info.json.  The measurement SURVEY.md 8(d) defines: wall clock of the
    process from start to outputs written, index load included (and listed)."""
    exe = os.path.join(ROOT, "kallisto_b200", "kallisto_b200")
    if not os.path.exists(exe):
        return None
    cores = os.cpu_count() or 1
    threads = min(cores, 64)
    runs = []
    for _ in range(repeats):
        env = dict(os.environ, KB_CLI_TIMING="1")
        cmd = [exe, "quant", "-i", idx, "-o", outdir, "--plaintext", "-t", str(threads)]
        if len(devices) > 1:
            cmd += ["--devices", ",".join(str(x) for x in devices)]
        else:
            cmd += ["--device", str(devices[0])]
        t0 = time.perf_counter()
        r = subprocess.run(cmd + files, stdout=subprocess.DEVNULL, stderr=subprocess.PIPE, text=True, env=env)
        dt = time.perf_counter() - t0
        if r.returncode != 0:
            raise RuntimeError("kallisto_b200 quant failed: " + r.stderr[-400:])
        ph = {}
        for m in re.finditer(r"\[timing\] ([^:\n]+): ([0-9.eE+-]+) s \(at", r.stderr):
            ph[m.group(1)] = float(m.group(2))
        runs.append((dt, ph))
    # a fresh process pays the CUDA context (0.5-1.1 s on the same box, run to run): the MEDIAN of the runs is reported, all are listed
    dt, ph = sorted(runs, key=lambda x: x[0])[len(runs) // 2]
    work = sum(v for k2, v in ph.items() if k2 not in ("index load", "run set-up"))
    return {"seconds_process_wall": round(dt, 3), "seconds_process_wall_runs": [round(x[0], 3) for x in runs],
            "seconds_reads_to_outputs": round(work, 4), "phases_s": {k2: round(v, 4) for k2, v in ph.items()},
            "pairs": n_pairs, "threads": threads, "devices": list(devices),
            "pairs_per_s_reads_to_outputs": n_pairs / max(1e-9, work)}


def random_sector_peak(table_bytes):
    """Hardware ceiling for the probe pattern of match_kernel: independent random 32-byte sector reads over a
    table of this size (tools/randbench.cu, run live, a few seconds)."""
    exe = os.path.join(ROOT, "tools", "randbench")
    if not os.path.exists(exe):
        return None
    gib = max(1, int(round(table_bytes / 2.0 ** 30)))
    gib = 1 << (gib.bit_length() - 1)          # the benchmark rounds down to a power of two anyway
    try:
        out = subprocess.run([exe, str(gib)], capture_output=True, text=True, timeout=120).stdout
        rows = [json.loads(l) for l in out.splitlines() if l.startswith("{")]
        best = max(rows, key=lambda r: r["gsectors_per_s"])
        return {"gsectors_per_s": best["gsectors_per_s"], "gb_per_s": best["gb_per_s_32B"], "table_gib": best["table_gib"],
                "source": "tools/randbench (live): independent random 32-byte sector reads, 1536 threads/SM x 4 in flight"}
    except Exception as e:
        log("randbench failed: %r" % e)
        return None


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


# ---------------------------------------------------------------------------------------------
# reference arm: the unmodified reference's CPU path on the host cores, on the SAME reads as our timed job
# ---------------------------------------------------------------------------------------------
def _ref_time(args):
    from oracle import oracle as O
    t0 = time.perf_counter()
    r = O.ref_run(args, check=False)
    return time.perf_counter() - t0, r


def reference_full(idx, files, n_pairs):
    """`kallisto quant --plaintext -t T` on the FASTQ of the whole timed job (file to file, one run).  T is chosen
    first on a 2 M-pair sample (the reference's reader lock makes very high thread counts slower).
    -> dict(value = pairs / process wall clock, index load included and listed)."""
    d, f1, f2, s1, s2, t1, t2 = files
    cores = os.cpu_count() or 1
    with open(idx, "rb") as f:            # page cache
        while f.read(1 << 26):
            pass
    out = os.path.join(d, "ref_out")
    t_load, _ = _ref_time(["quant", "-i", idx, "-o", out, "--plaintext", "-t", "4", t1, t2])   # one pair: start-up + index load
    tried = {}
    n_s = sum(1 for _ in open(s1, "rb")) // 4
    for threads in sorted({min(cores, 16), min(cores, 32), min(cores, 64), cores}):
        dt, _ = _ref_time(["bus", "-x", "bulk", "--paired", "-i", idx, "-o", out + "_cal", "-t", str(threads), s1, s2])
        tried[threads] = round(n_s / max(1e-9, dt - t_load))
    best_t = max(tried, key=tried.get)
    dt, r = _ref_time(["quant", "-i", idx, "-o", out, "--plaintext", "-t", str(best_t), f1, f2])
    if r.returncode != 0:
        raise RuntimeError("reference quant failed: " + r.stderr.decode(errors="replace")[-300:])
    m = re.search(r"ran for ([0-9,]+) rounds", r.stderr.decode(errors="replace"))
    return dict(value=n_pairs / dt, seconds_process_wall=round(dt, 2), seconds_index_load=round(t_load, 2), threads=best_t,
                host_cores=cores, pairs=n_pairs, em_rounds=int(m.group(1).replace(",", "")) if m else None,
                alignment_pairs_per_s_by_threads_on_sample=tried, when=time.time())


def reference_sample(idx, files, repeats=1):
    """Bounded CPU baseline (our arm's cpu_baseline when no full reference run from this box is at hand): the 2 M-pair
    sample at -t min(cores, 32), start-up + index load subtracted.  The reference's single-threaded EM (~14 s on this
    workload whatever the read count) weighs much more on a sample than on the full job: said so in `sample`."""
    d, f1, f2, s1, s2, t1, t2 = files
    cores = os.cpu_count() or 1
    threads = min(cores, 32)
    out = os.path.join(d, "ref_out_sample")
    t_load, _ = _ref_time(["quant", "-i", idx, "-o", out, "--plaintext", "-t", str(threads), t1, t2])
    n_s = sum(1 for _ in open(s1, "rb")) // 4
    dt, _ = _ref_time(["quant", "-i", idx, "-o", out, "--plaintext", "-t", str(threads), s1, s2])
    return dict(value=n_s / max(1e-9, dt - t_load), threads=threads, host_cores=cores, pairs=n_s, t_load=round(t_load, 2),
                t_total=round(dt, 2))


DUMP_MAX_ELEMS = 1 << 20


def dump_outputs(d, em, ec_table, flens):
    """The arrays the timed job handed to its caller, as float64 .npy files (7 arrays of at most 2^20 entries)."""
    eo, et, ec, _ = ec_table
    out = {"est_counts": em["est_counts"], "eff_lens": em["eff_lens"], "em_rounds": np.array([em["rounds"]]),
           "fragment_lengths": flens, "ec_counts": ec, "ec_sizes": np.diff(eo.astype(np.int64)), "ec_tids": et}
    os.makedirs(d, exist_ok=True)
    for name, a in out.items():
        a = np.asarray(a, np.float64)
        if len(a) > DUMP_MAX_ELEMS:     # fixed seed: the same positions for arrays of the same length
            a = a[np.sort(np.random.default_rng(0).choice(len(a), DUMP_MAX_ELEMS, replace=False))]
        np.save(os.path.join(d, name + ".npy"), a)
    log("outputs of the timed job written to %s" % d)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=15)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="quant", choices=["quant", "bus10xv3", "bootstrap"])
    ap.add_argument("--genes", type=int, default=int(os.environ.get("KB_BENCH_GENES", "62000")))
    ap.add_argument("--pairs-per-step", type=int, default=int(os.environ.get("KB_BENCH_PAIRS", "2000000")))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the reported timed job to DIR/<name>.npy")
    args = ap.parse_args()

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    N = args.gpus
    K, W, P = args.steps, max(args.warmup, 0), args.pairs_per_step
    workload_name = ("human-GENCODE-v44-like synthetic transcriptome (%d genes, seed 44; reference-built k=31 index), "
                     "synthetic 2x100bp pairs" % args.genes)
    if args.workload != "quant":
        import bench_extra
        return bench_extra.main(args, rank, world, local_rank, workload_name)

    import torch

    def sim_factory(dev=None):
        d = dev if dev is not None else ("cuda:%d" % local_rank if torch.cuda.is_available() else "cpu")
        return benchdata.TorchSimulator(concat, lens, d, read_len=READ_LEN)

    if args.impl == "reference":
        if rank != 0:
            return 0
        idx, concat, lens = workload(args.genes)
        files = fastq_job_files(args.genes, P, K, W, sim_factory)
        info = reference_full(idx, files, K * P)
        v = info["value"]
        line = {
            "metric": "paired reads/sec quant", "value": v, "unit": "pairs/s", "n_gpus": N, "steps": K, "warmup": W,
            "ms_per_step": info["seconds_process_wall"] * 1e3 / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "u64/f64", "data": "synthetic", "impl": "reference",
            "config": {"workload": workload_name, "pairs_per_step": P, "read_len": READ_LEN,
                       "reference": "oracle/_ref/kallisto quant --plaintext -t %d on the %d pairs of the timed job (rank 0's), plain "
                                    "FASTQ in /dev/shm -> abundance.tsv; value = pairs / process wall clock, index load (%.1f s) "
                                    "included" % (info["threads"], K * P, info["seconds_index_load"]), **info},
            "cpu_baseline": {"value": v, "unit": "pairs/s", "cores": info["threads"], "kind": "reference",
                             "sample": "all %d pairs of the job, one run" % (K * P)},
            "e2e": {"value": v, "unit": "pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        }
        with open(os.path.join(files[0], "reference_line.json"), "w") as f:
            json.dump(line, f)
        print(json.dumps(line), flush=True)
        return 0

    # ---------------------------------- our arm ----------------------------------
    import torch.distributed as dist
    import kallisto_b200 as K200
    gloo = None
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
        gloo = dist.new_group(backend="gloo")       # host-side waits that must not occupy the GPUs
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    idx, concat, lens = workload(args.genes)
    files = None
    need_files = (not os.environ.get("KB_BENCH_NO_CLI")) or (not args.no_cpu_baseline and world == 1)
    if rank == 0 and need_files:
        files = fastq_job_files(args.genes, P, K, W, sim_factory)     # before the big allocations: uses the GPU for simulation
    t0 = time.time()
    index = K200.KmerIndex(idx, device=local_rank, threads=min(16, os.cpu_count() or 4))
    log("rank %d: index loaded in %.1f s (parse %.1f s, device build %.1f s): %s" % (
        rank, time.time() - t0, index.info["load_seconds"], index.info["build_seconds"], index.info))
    sim = sim_factory(dev)
    t0 = time.time()
    seeds = [1000 + rank * 100003 + s for s in range(W)] + job_seeds(rank, W, K)
    d_batches = [sim.pairs(P, seed=sd) for sd in seeds]
    torch.cuda.synchronize()
    log("rank %d: %d x %d pairs simulated on the device in %.1f s" % (rank, W + K, P, time.time() - t0))
    h_batches = [torch.empty((P, 2, READ_LEN), dtype=torch.uint8, pin_memory=True) for _ in range(K)]
    for h, d in zip(h_batches, d_batches[W:]):
        h.copy_(d)
    torch.cuda.synchronize()
    stream = torch.cuda.current_stream()
    n_reads = 2 * P

    comm = None
    if world > 1:
        # the NCCL communicator of the library's own merge (csrc/comm.cu): id from rank 0, spread with torch.distributed
        uid = [K200.Comm.unique_id() if rank == 0 else None]
        dist.broadcast_object_list(uid, src=0)
        comm = K200.Comm(world, rank, uid[0], local_rank)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def new_run():
        mc = K200.MinCollector(index, paired=True, collect_fld=True, max_batch_reads=P, max_batch_bases=P * 2 * READ_LEN + 64)
        mc.set_stream(stream.cuda_stream)
        return mc

    def job(batches, device_input, timed):
        """One whole job: K batches through pseudoalignment, the EC merge across ranks, EC numbering + EM on rank 0.
        -> (total ms, align ms, run, em result) -- CUDA events on the launching stream, max over ranks."""
        mc = new_run()
        if timed:
            mc.enable_timing(True)
        barrier()
        ev0, ev1, ev2 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
        t_host = time.perf_counter()
        ev0.record(stream)
        for b in batches:
            if device_input:
                mc.process_buffer_device(b.data_ptr(), None, n_reads, READ_LEN)
            else:
                mc.process_buffer_ptr(b.data_ptr(), None, n_reads, READ_LEN, None)
        ev1.record(stream)
        if world > 1:
            mc.merge_nccl(comm)               # the one exchange step (collective)
        em = mc.run_em() if rank == 0 else None   # EC ids, CSR/CSC and the EM kernel on the device; est_counts back on the host
        ev2.record(stream)
        torch.cuda.synchronize()
        t_host = time.perf_counter() - t_host
        barrier()
        tt = torch.tensor([ev0.elapsed_time(ev2), ev0.elapsed_time(ev1), t_host * 1e3], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        return float(tt[0]), float(tt[1]), float(tt[2]), mc, em

    # ---- warm-up: W steps, then one complete untimed job (work buffers, memo tables, NCCL, clocks) ----
    mcw = new_run()
    for s in range(W):
        mcw.process_buffer_device(d_batches[s].data_ptr(), None, n_reads, READ_LEN)
    if world > 1:
        mcw.merge_nccl(comm)
    if rank == 0:
        mcw.run_em()
    mcw.close()
    w_total, _, _, mcx, _ = job(d_batches[W:], True, False)
    mcx.close()

    # ---- value: inputs resident in HBM; the job is timed twice, the SECOND run is reported, both are listed ----
    sampler = ClockSampler(local_rank)
    runs = []
    first = job(d_batches[W:], True, True)
    first[3].close()
    runs.append(first[0])
    sampler.start()
    t_total_ms, t_align_ms, _, mc, em = job(d_batches[W:], True, True)
    clocks = sampler.stop()
    runs.append(t_total_ms)
    st = mc.finalize()
    tm = mc.timings()       # after run_em: includes the EC numbering / CSR / CSC / EM launches
    em_shape = None
    if rank == 0:
        eo, et, ec, _ = mc.ec_table()
        ln = np.diff(eo.astype(np.int64))
        em_shape = {"n_ecs": int(len(ln)), "n_multi_ecs": int((ln > 1).sum()), "nnz_multi": int(ln[ln > 1].sum())}
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, em, (eo, et, ec, None), mc.flens)
    mc.close()

    # ---- pinned host buffers through the C ABI, H2D inside (host wall clock) ----
    p_total_ms, _, p_host_ms, mc2, _ = job(h_batches, False, False)
    mc2.close()

    total_pairs = K * P * world
    value = total_pairs / (t_total_ms * 1e-3)
    pinned_value = total_pairs / (p_host_ms * 1e-3)

    # ---- roofline of the dominant kernel (match_kernel) ----
    probes_per_pair = st["n_probes"] / max(1, K * P)          # this rank's own fragments
    visits_per_pair = st["n_slot_visits"] / max(1, K * P)
    # algorithmic bytes per pair (SURVEY.md 8d): read bases + one 32-byte sector per executed probe +
    # the per-pair result; EC-list bytes are only touched by the (rare) resolve kernel
    bytes_per_pair = 2 * READ_LEN + probes_per_pair * 32 + 16
    peak, peak_src = measured_peak()
    match_ms_per_launch = tm["match_ms"] / max(1, tm["match_launches"])
    achieved = bytes_per_pair * P / (match_ms_per_launch * 1e-3) / 1e9
    roofline = {"bound": "hbm", "kernel": "match_kernel", "achieved": achieved, "peak": peak, "unit": "GB/s",
                "frac": achieved / peak, "peak_source": peak_src, "traffic": None,
                "bytes_per_pair": bytes_per_pair, "probes_per_pair": probes_per_pair,
                "slot_visits_per_pair": visits_per_pair, "ms_per_launch": match_ms_per_launch,
                "resolve_ms_per_launch": tm["resolve_ms"] / max(1, tm["resolve_launches"]),
                "pack_ms_per_launch": tm["pack_ms"] / max(1, tm["match_launches"]), "em_ms": tm["em_ms"],
                "em_prep_ms": tm["em_prep_ms"], "em_rounds": em["rounds"] if em else None}
    if world == 1 and not os.environ.get("KB_BENCH_NO_RANDBENCH"):
        rs = random_sector_peak(index.info["table_slots"] * 32)
        if rs:
            sectors_per_s = visits_per_pair * P / (match_ms_per_launch * 1e-3) / 1e9
            roofline["random_sector_peak"] = rs
            roofline["sectors_per_s_achieved"] = sectors_per_s
            roofline["frac_random"] = sectors_per_s / rs["gsectors_per_s"]
    roofline_em = None
    if em and em_shape and tm["em_ms"] > 0:
        # SURVEY.md 8(d): B_K4 per round = nnz (tid 4 + w 8 + alpha gather 8 + next accumulate 8) + multi-ECs (count 4 + denom 8)
        # + T (alpha read, next write, compare: 24)
        b_round = em_shape["nnz_multi"] * 28 + em_shape["n_multi_ecs"] * 12 + index.num_trans * 24
        ach = b_round * em["rounds"] / (tm["em_ms"] * 1e-3) / 1e9
        roofline_em = {"bound": "hbm", "kernel": "em_kernel", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                       "bytes_per_round": b_round, "rounds": em["rounds"], "us_per_round": tm["em_ms"] * 1e3 / max(1, em["rounds"]),
                       "note": "the problem lives in L2: bound by the L2 gather rate and the grid barriers of a round, not by HBM",
                       **em_shape}
    prof = os.path.join(ROOT, "profiles", "match_kernel_traffic.json")
    if os.path.exists(prof):
        try:
            roofline["traffic"] = json.load(open(prof))["dram_bytes_per_launch"]
        except Exception:
            pass

    # ---- e2e: the drop-in command line, FASTQ files -> abundance.tsv, process wall clock (rank 0 drives all N GPUs
    #      through --devices; the other ranks wait on the host) ----
    del d_batches, h_batches, sim
    index.close()
    torch.cuda.empty_cache()
    cli = None
    if world > 1:
        dist.barrier(group=gloo)
    if rank == 0 and not os.environ.get("KB_BENCH_NO_CLI"):
        try:
            fl = [files[1], files[2]] * world           # weak scaling: the job's file pair once per GPU (config 5 does the same)
            cli = cli_run(idx, fl, K * P * world, list(range(world)), os.path.join(files[0], "cli_out"))
        except Exception as e:
            cli = {"error": repr(e)[:300]}
    if world > 1:
        dist.barrier(group=gloo)
        dist.barrier()
        dist.destroy_process_group()
    if rank != 0:
        return 0
    if cli and "seconds_process_wall" in cli:
        e2e = {"value": K * P * world / cli["seconds_process_wall"], "unit": "pairs/s", "h2d_bytes_per_step": P * 2 * READ_LEN * world,
               "d2h_bytes_per_step": int(index.num_trans * 8 / K),
               "api": "kallisto_b200 quant --plaintext -t %d %s(plain FASTQ in /dev/shm -> abundance.tsv + run_info.json): pairs / "
                      "process wall clock, index load included" % (cli["threads"], "--devices 0..%d " % (world - 1) if world > 1 else ""),
               **cli}
    else:
        e2e = {"value": pinned_value, "unit": "pairs/s", "h2d_bytes_per_step": P * 2 * READ_LEN, "d2h_bytes_per_step": int(index.num_trans * 8 / K),
               "api": "kb_pseudoalign_batch (pinned host bases) x K, kb_quant_merge_nccl, kb_em_run", "cli": cli}
    cpu = None
    if not args.no_cpu_baseline and world == 1:
        try:
            ref_line = os.path.join(files[0], "reference_line.json")
            if os.path.exists(ref_line) and time.time() - os.path.getmtime(ref_line) < 7200:
                rl = json.load(open(ref_line))
                cpu = dict(rl["cpu_baseline"])
                cpu["sample"] += " (the --impl reference run on this box %.0f s earlier: -t %d, process wall %.1f s incl. %.1f s index load)" % (
                    time.time() - os.path.getmtime(ref_line), rl["config"]["threads"], rl["config"]["seconds_process_wall"],
                    rl["config"]["seconds_index_load"])
            else:
                info = reference_sample(idx, files)
                cpu = {"value": info["value"], "unit": "pairs/s", "cores": info["threads"], "kind": "reference",
                       "sample": "%d pairs of the job, oracle/_ref/kallisto quant -t %d on %d cores, one-pair run (%.1f s: start-up + index "
                                 "load) subtracted; the reference's single-threaded EM weighs far more on this sample than on the whole "
                                 "job (see --impl reference)" % (info["pairs"], info["threads"], info["host_cores"], info["t_load"])}
        except Exception as e:   # the baseline must never take the measurement down
            cpu = {"value": None, "unit": "pairs/s", "cores": os.cpu_count(), "kind": "reference", "sample": "failed: %r" % e}
    line = {
        "metric": "paired reads/sec quant", "value": value, "unit": "pairs/s", "n_gpus": world, "steps": K, "warmup": W,
        "ms_per_step": t_total_ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "u64/f64", "data": "synthetic",
        "config": {"workload": workload_name, "pairs_per_step": P, "read_len": READ_LEN, "parallelism": "dp%d" % world,
                   "l2": "every step reads a different %d MB batch (> 126 MB L2)" % (P * 2 * READ_LEN // 1000000),
                   "em_in_timed_region": True, "align_ms": t_align_ms, "total_ms": t_total_ms,
                   "total_ms_runs": [round(x, 3) for x in runs], "reported_run": "second of two timed runs of the whole job "
                   "(after W warm-up steps and one untimed job)", "untimed_job_ms": round(w_total, 3),
                   "pinned_host_buffers": {"value": pinned_value, "unit": "pairs/s", "seconds": p_host_ms * 1e-3,
                                           "api": "kb_pseudoalign_batch (pinned host bases, H2D inside) x K, merge, kb_em_run; host wall clock"},
                   "n_ecs": st["n_ecs"], "n_ec_entries": st["n_ec_entries"], "n_resolved": st["n_resolved"],
                   "n_memo_hits": st["n_memo_hits"],
                   "p_pseudoaligned": st["n_pseudoaligned"] / max(1, st["n_processed"]),
                   "index": {k: index.info[k] for k in ("n_targets", "n_kmers", "n_unitigs", "n_ec_sets", "table_slots")}},
        "clocks": clocks,
        "e2e": e2e,
        "gpu_launches": int(tm["kernel_launches"]),   # counted by the engine (pack, match, resolve, fld, import, EC numbering, EM)
        "roofline": roofline,
    }
    if roofline_em:
        line["roofline_em"] = roofline_em
    if cpu:
        line["cpu_baseline"] = cpu
    print(json.dumps(line), flush=True)
    return 0


if __name__ == "__main__":
    sys.exit(main())
