"""CPU: the oracle (oracle/kb_oracle.cpp) against the UNMODIFIED reference binary (oracle/_ref/kallisto) on small
random transcriptomes that are generated on the fly -- other k, shared exons, short transcripts, Ns, read lengths
around k.  Strengthens the pin of the oracle beyond the committed fixtures.  The reference's indices of these
transcriptomes and its results on them are stored under tests/golden/fuzz (`python -m tests.test_oracle_fuzz`
rewrites them with oracle/_ref/kallisto)."""
import os
import sys

import numpy as np
import pytest

from oracle import oracle as O
from tests import util

COMP = bytes.maketrans(b"ACGT", b"TGCA")
FUZZ = os.path.join(util.GOLDEN, "fuzz")
INDICES = os.path.join(FUZZ, "indices.npz")          # `kallisto index -t 1` of every make_case transcriptome
REF_RESULTS = os.path.join(FUZZ, "ref_ec_dump.npz")   # `kallisto bus -x bulk --num -t 1` of every test case
CASES = [(1, 31, 75), (2, 21, 50), (3, 15, 36), (4, 31, 33), (5, 27, 150)]
MODES = ["paired", "single", "paired_fr", "single_rf"]


def make_case(tmp, seed, k, read_len, n_reads, build_index=False):
    rng = np.random.default_rng(seed)
    lut = np.frombuffer(b"ACGT", np.uint8)
    exons = [bytes(lut[rng.integers(0, 4, int(rng.integers(k + 3, 220)))]) for _ in range(24)]
    txs = []
    for g in range(8):
        pool = list(rng.choice(len(exons), size=int(rng.integers(2, 6)), replace=False))
        for _ in range(int(rng.integers(1, 5))):
            sub = sorted(rng.choice(pool, size=int(rng.integers(1, len(pool) + 1)), replace=False))
            t = b"".join(exons[i] for i in sub)
            if len(t) >= k + 5:
                txs.append(t)
    txs = list(dict.fromkeys(txs))            # the reference refuses duplicate sequences only by name, keep it simple
    fa = os.path.join(tmp, "t.fa")
    with open(fa, "wb") as f:
        for i, t in enumerate(txs):
            f.write(b">tx%d\n%s\n" % (i, t))
    idx = os.path.join(tmp, "t.kidx")
    if build_index:
        O.ref_index(fa, idx, k=k)
    else:
        with np.load(INDICES) as z:
            z["seed%d_k%d" % (seed, k)].tofile(idx)
    r1, r2 = [], []
    for _ in range(n_reads):
        t = txs[int(rng.integers(0, len(txs)))]
        fl = int(min(len(t), rng.integers(read_len, read_len + 120)))
        s = int(rng.integers(0, len(t) - fl + 1))
        frag = t[s:s + fl]
        a = bytearray(frag[:read_len])
        b = bytearray(frag[-read_len:].translate(COMP)[::-1])
        for r in (a, b):
            for p in range(len(r)):
                x = rng.random()
                if x < 0.01:
                    r[p] = b"ACGT"[int(rng.integers(0, 4))]
                elif x < 0.013:
                    r[p] = ord("N")
        if rng.random() < 0.5:
            a, b = b, a
        if rng.random() < 0.03:               # unrelated sequence
            a = bytearray(bytes(lut[rng.integers(0, 4, read_len)]))
        r1.append(bytes(a))
        r2.append(bytes(b))
    paths = []
    for m, rs in ((1, r1), (2, r2)):
        p = os.path.join(tmp, "r_%d.fq" % m)
        with open(p, "wb") as f:
            for i, r in enumerate(rs):
                f.write(b"@r%d/%d\n%s\n+\n%s\n" % (i, m, r, b"I" * len(r)))
        paths.append(p)
    return idx, r1, r2, paths


def mode_opts(mode):
    paired = mode.startswith("paired")
    strand = {"fr": 1, "rf": 2}.get(mode.split("_")[-1], 0)
    return paired, strand


def reference_ec_dump(idx, r1, paths, mode, out):
    """-> {name: array}: per-fragment EC ids, EC sets (offsets, ids) and the fragment-length histogram of the reference."""
    paired, strand = mode_opts(mode)
    extra = {0: [], 1: ["--fr-stranded"], 2: ["--rf-stranded"]}[strand]
    rec, ecs, flens = O.ref_ec_dump(idx, out, paths if paired else paths[:1], paired=paired, extra=extra)
    want = np.full(len(r1), -1, np.int64)
    want[rec["flags"]] = rec["ec"]
    off = np.cumsum([0] + [len(e) for e in ecs])
    res = {"fragments": want, "ec_offsets": off, "ec_tids": np.array([t for e in ecs for t in e], np.int64)}
    if paired and flens is not None:
        res["flens"] = flens
    return res


@pytest.mark.parametrize("seed,k,read_len", CASES)
@pytest.mark.parametrize("mode", MODES)
def test_random_transcriptome(seed, k, read_len, mode, tmp_path):
    paired, strand = mode_opts(mode)
    idx, r1, r2, paths = make_case(str(tmp_path), seed, k, read_len, 1500)
    key = "seed%d_%s_" % (seed, mode)
    with np.load(REF_RESULTS) as z:
        want = z[key + "fragments"]
        eo_ref, et_ref = z[key + "ec_offsets"], z[key + "ec_tids"]
        flens = z[key + "flens"] if key + "flens" in z.files else None
    ecs = util.ec_sets(eo_ref, et_ref)

    ix = O.OracleIndex(idx)
    run = O.OracleRun(ix, paired, strand, True)
    bases, off = O.to_batch(r1, r2 if paired else None)
    got = run.pseudoalign(bases, off)
    eo, et, ec = run.ec_table()
    np.testing.assert_array_equal(got, want)
    assert util.ec_sets(eo, et) == [tuple(e) for e in ecs]
    if paired and flens is not None:
        np.testing.assert_array_equal(run.flens(), flens)


if __name__ == "__main__":
    # rewrite the fixtures from the unmodified reference binary: the indices of this test's and of
    # tests/test_oracle_bus_fuzz.py's transcriptomes, and this test's reference results
    import tempfile
    from tests.test_oracle_bus_fuzz import INDEX_CASES
    os.makedirs(FUZZ, exist_ok=True)
    indices, results = {}, {}
    for seed, k, read_len in CASES + INDEX_CASES:
        with tempfile.TemporaryDirectory() as td:
            idx, r1, r2, paths = make_case(td, seed, k, read_len, 1500, build_index=True)
            indices["seed%d_k%d" % (seed, k)] = np.fromfile(idx, np.uint8)
            if (seed, k, read_len) in CASES:
                for mode in MODES:
                    for name, a in reference_ec_dump(idx, r1, paths, mode, os.path.join(td, mode)).items():
                        results["seed%d_%s_%s" % (seed, mode, name)] = a
    np.savez_compressed(INDICES, **indices)
    np.savez_compressed(REF_RESULTS, **results)
    sys.exit(0)
