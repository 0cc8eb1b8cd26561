"""CPU: the BUS record model (oracle/oracle.py:bus_model -- the rules the CUDA path is held to) against the UNMODIFIED
reference binary on random small transcriptomes with random technology layouts: barcode / UMI pieces anywhere in the
files, with and without a UMI, one sequence read or a pair with random start offsets, tag sequences of several lengths
(short ones must match exactly, src/ProcessReads.cpp:1517), strand modes, --num, reads that are too short for their
slices, Ns in barcodes, UMIs and tags.  The reference's results are stored in tests/golden/fuzz/ref_bus.npz (record
count and SHA-256 of the sorted records, EC sets, fragment lengths; `python -m tests.test_oracle_bus_fuzz` rewrites it
with oracle/_ref/kallisto after `python -m tests.test_oracle_fuzz` has stored the indices)."""
import hashlib
import os
import subprocess
import sys

import numpy as np
import pytest

from oracle import oracle as O
from tests.test_oracle_bus_paired import sorted_records
from tests.test_oracle_fuzz import FUZZ, make_case

SEEDS = range(16)
KS = [31, 21, 15, 27]
INDEX_CASES = [(50 + seed, KS[seed % 4], KS[seed % 4] + 2) for seed in SEEDS]     # (seed, k, read length) of make_case
REF_RESULTS = os.path.join(FUZZ, "ref_bus.npz")


def records_digest(rec):
    return hashlib.sha256(sorted_records(rec.copy()).tobytes()).hexdigest()


def layout(rng, paired, tag, no_umi):
    """Random technology: file 0 = barcode/UMI read (+ optionally the first sequence read), files 1.. = sequence reads."""
    a = int(rng.integers(0, 4))
    blen = int(rng.integers(4, 13))
    bc = [(0, a, a + blen)]
    if rng.random() < 0.4:                       # a second barcode piece further along
        b2 = a + blen + int(rng.integers(0, 5))
        bc.append((0, b2, b2 + int(rng.integers(2, 7))))
    end = bc[-1][2]
    taglen = len(tag) if tag else 0
    ulen = int(rng.integers(4, 11))
    u0 = end + int(rng.integers(0, 4))
    umi_user = None if no_umi else [(0, u0, u0 + taglen + ulen)]          # as the user writes it: tag + UMI
    pre = (umi_user[0][2] if umi_user else end) + int(rng.integers(0, 4))
    seq_in_0 = rng.random() < 0.5                # sequence read shares the barcode file (starts after the UMI)
    if paired:
        seq = (0, pre) if seq_in_0 else (1, int(rng.integers(0, 6)))
        seq2 = (2 if not seq_in_0 else 1, int(rng.integers(0, 9)))
    else:
        seq = (0, pre) if seq_in_0 else (1, int(rng.integers(0, 6)))
        seq2 = None
    nfiles = 1 + max(seq[0], seq2[0] if seq2 else 0)
    return bc, umi_user, seq, seq2, nfiles, pre


def tech_string(bc, umi_user, seq, seq2):
    t = lambda v: ",".join("%d,%d,%d" % x for x in v)
    s = [(seq[0], seq[1], 0)] + ([(seq2[0], seq2[1], 0)] if seq2 else [])
    return "%s:%s:%s" % (t(bc), t(umi_user) if umi_user else "-1,-1,-1", t(s))


def bus_case(seed, tmp_path):
    """Inputs of one random layout: -> dict(index, files as lists of sequences, their paths, layout, reference arguments)."""
    rng = np.random.default_rng(1000 + seed)
    paired = bool(seed & 1)
    tag = [None, None, b"ACGTTGCA", b"TTGCA", b"ATTGCGCAATG"][seed % 5]
    no_umi = tag is None and seed % 3 == 0
    strand = int(rng.integers(0, 3))
    num = bool(rng.random() < 0.3)
    k = KS[seed % 4]
    idx, r1, r2, _ = make_case(str(tmp_path), 50 + seed, k, int(rng.integers(k + 2, 90)), 1200)
    bc, umi_user, seq, seq2, nfiles, pre = layout(rng, paired, tag, no_umi)
    lut = np.frombuffer(b"ACGT", np.uint8)
    n = len(r1)
    cells = lut[rng.integers(0, 4, (5, pre))]
    head = []
    for i in range(n):
        h = bytearray(bytes(cells[int(rng.integers(0, 5))]))
        if umi_user:                              # a fresh UMI (and, for most reads, the tag in front of it)
            u0, u1 = umi_user[0][1], umi_user[0][2]
            h[u0:u1] = bytes(lut[rng.integers(0, 4, u1 - u0)])
            if tag and rng.random() < 0.6:
                tg = bytearray(tag)
                x = rng.random()
                if x < 0.15:
                    tg[int(rng.integers(0, len(tg)))] = ord("ACGT"[int(rng.integers(0, 4))])
                elif x < 0.2:
                    tg[int(rng.integers(0, len(tg)))] = ord("N")
                h[u0:u0 + len(tag)] = tg
        if rng.random() < 0.03:
            h[int(rng.integers(0, len(h)))] = ord("N")
        if rng.random() < 0.02:
            h = h[:int(rng.integers(0, len(h)))]     # too short for some slice: the set is skipped
        head.append(bytes(h))
    files = [None] * nfiles
    seqs = [r1, r2]
    si = 0
    for f in range(nfiles):
        if f == 0:
            if seq[0] == 0:
                files[0] = [head[i] + seqs[0][i] for i in range(n)]
                si = 1
            else:
                files[0] = head
        else:
            off = seq[1] if (seq[0] == f) else (seq2[1] if seq2 and seq2[0] == f else 0)
            files[f] = [bytes(lut[rng.integers(0, 4, off)]) + seqs[si][i] for i in range(n)]
            si += 1
    paths = []
    for f in range(nfiles):
        p = str(tmp_path / ("f%d.fq" % f))
        with open(p, "wb") as fo:
            for i, s in enumerate(files[f]):
                fo.write(b"@r%d\n%s\n+\n%s\n" % (i, s, b"I" * len(s)))
        paths.append(p)
    args = ["bus", "-i", idx, "-o", str(tmp_path / "o"), "-t", "1", "-x", tech_string(bc, umi_user, seq, seq2)]
    args += [["--unstranded"], ["--fr-stranded"], ["--rf-stranded"]][strand]
    if paired:
        args.append("--paired")
    if num:
        args.append("--num")
    if tag:
        args += ["--tag", tag.decode()]
    return dict(idx=idx, files=files, paths=paths, args=args, bc=bc, umi_user=umi_user, seq=seq, seq2=seq2, strand=strand,
                num=num, tag=tag, paired=paired)


def reference_bus(c, out):
    """-> {name: array}: the reference's record count and records digest, EC sets and fragment lengths."""
    r = subprocess.run([O.REF_BIN] + c["args"] + c["paths"], capture_output=True, text=True)
    assert r.returncode in (0, 1), r.stderr[-500:]          # 1: nothing pseudoaligned
    hdr, ref = O.read_bus(os.path.join(out, "output.bus"))
    ecs = O.read_matrix_ec(os.path.join(out, "matrix.ec")) if len(ref) else []
    res = {"n_records": np.array(len(ref)), "records_sha256": np.array(records_digest(ref)),
           "ec_offsets": np.cumsum([0] + [len(e) for e in ecs]), "ec_tids": np.array([t for e in ecs for t in e], np.int64)}
    if c["paired"]:
        res["flens"] = np.array(open(os.path.join(out, "flens.txt")).read().split(), np.uint32)
    return res


@pytest.mark.parametrize("seed", SEEDS)
def test_random_layout(seed, tmp_path):
    c = bus_case(seed, tmp_path)
    with np.load(REF_RESULTS) as z:
        ref = {name[len("seed%d_" % seed):]: z[name] for name in z.files if name.startswith("seed%d_" % seed)}
    tag, umi_user = c["tag"], c["umi_user"]
    taglen = len(tag) if tag else 0
    umi = None if umi_user is None else [(umi_user[0][0], umi_user[0][1] + taglen, umi_user[0][2])]
    ix = O.OracleIndex(c["idx"])
    m = O.bus_model(ix, c["files"], c["bc"], umi, c["seq"], c["seq2"], strand=c["strand"], num=c["num"], tag=tag)
    assert len(m["records"]) == int(ref["n_records"]), (c["args"], len(m["records"]), int(ref["n_records"]))
    assert records_digest(m["records"]) == str(ref["records_sha256"]), c["args"]
    offs, tids = ref["ec_offsets"], ref["ec_tids"]
    assert m["ecs"] == [tuple(int(t) for t in tids[offs[i]:offs[i + 1]]) for i in range(len(offs) - 1)]
    if c["paired"]:
        np.testing.assert_array_equal(m["flens"][0], ref["flens"])


if __name__ == "__main__":
    # rewrite tests/golden/fuzz/ref_bus.npz from the unmodified reference binary
    import pathlib
    import tempfile
    results = {}
    for seed in SEEDS:
        with tempfile.TemporaryDirectory() as td:
            c = bus_case(seed, pathlib.Path(td))
            for name, a in reference_bus(c, os.path.join(td, "o")).items():
                results["seed%d_%s" % (seed, name)] = a
    np.savez_compressed(REF_RESULTS, **results)
    sys.exit(0)
