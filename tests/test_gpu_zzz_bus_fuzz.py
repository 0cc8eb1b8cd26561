"""GPU: the CUDA BUS path (kb_bus_create / kb_bus_batch) on the random technology layouts of tests/test_oracle_bus_fuzz.py
-- barcode / UMI pieces anywhere, with and without UMI, one sequence read or a pair with random start offsets, tag
sequences, strand modes, --num, too-short reads, Ns -- against the BUS record model, which the CPU suite holds to the
unmodified reference binary on the very same cases.  (Written after the round's GPU budget was spent: first run is the
driver's.)"""
import numpy as np
import pytest

import kallisto_b200 as K
from oracle import oracle as O
from tests.test_oracle_bus_fuzz import layout
from tests.test_oracle_bus_paired import sorted_records
from tests.test_oracle_fuzz import make_case

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("seed", range(8))
def test_random_layout_cuda_vs_model(seed, tmp_path):
    rng = np.random.default_rng(1000 + seed)
    paired = bool(seed & 1)
    tag = [None, None, b"ACGTTGCA", b"TTGCA", b"ATTGCGCAATG"][seed % 5]
    no_umi = tag is None and seed % 3 == 0
    strand = int(rng.integers(0, 3))
    num = bool(rng.random() < 0.3)
    k = [31, 21, 15, 27][seed % 4]
    idx, r1, r2, _ = make_case(str(tmp_path), 50 + seed, k, int(rng.integers(k + 2, 90)), 1200)
    bc, umi_user, seq, seq2, nfiles, pre = layout(rng, paired, tag, no_umi)
    lut = np.frombuffer(b"ACGT", np.uint8)
    n = len(r1)
    cells = lut[rng.integers(0, 4, (5, pre))]
    head = []
    for i in range(n):
        h = bytearray(bytes(cells[int(rng.integers(0, 5))]))
        if umi_user:
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
            h = h[:int(rng.integers(0, len(h)))]
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
    taglen = len(tag) if tag else 0
    umi = None if umi_user is None else [(umi_user[0][0], umi_user[0][1] + taglen, umi_user[0][2])]
    m = O.bus_model(O.OracleIndex(idx), files, bc, umi, seq, seq2, strand=strand, num=num, tag=tag)

    tech = (nfiles, bc, umi_user if umi_user else [(-1, -1, -1)], (seq[0], seq[1], 0), 0)
    if seq2:
        tech = tech + ((seq2[0], seq2[1], 0),)
    ix = K.KmerIndex(idx, device=0)
    bp = K.BUSProcessor(ix, tech, strand={0: "unstranded", 1: "fr", 2: "rf"}[strand], num=num, tag=tag)
    parts = []
    for a, b in ((0, n // 3), (n // 3, n)):
        parts.append(bp.process_sets([O.to_batch(f[a:b]) for f in files]))
    rec = np.concatenate(parts)
    assert len(rec) == len(m["records"])
    assert rec.tobytes() == m["records"].tobytes()              # read order, EC ids of first occurrence
    st = bp.finalize()
    assert st["n_processed"] == n and st["n_pseudoaligned"] == len(rec)
    eo, et, ec, eh = bp.ec_table()
    from tests import util
    assert util.ec_sets(eo, et) == m["ecs"]
    if paired:
        np.testing.assert_array_equal(bp.flens, m["flens"][0])
    b_h, u_h = bp.lengths()
    np.testing.assert_array_equal(b_h, m["bc_hist"].astype(np.uint32))
    np.testing.assert_array_equal(u_h, m["umi_hist"].astype(np.uint32))
    bp.close()
    ix.close()
