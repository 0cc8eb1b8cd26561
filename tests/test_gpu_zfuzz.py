"""GPU: the CUDA path against the oracle on the random transcriptomes of tests/test_oracle_fuzz.py (other k, reads
barely longer than k, Ns, unrelated reads, all strand modes).  The oracle itself is pinned on the unmodified
reference for exactly these inputs by the CPU test; the indices are the reference's, stored in tests/golden/fuzz."""
import numpy as np
import pytest

import kallisto_b200 as K
from oracle import oracle as O
from tests import util
from tests.test_oracle_fuzz import make_case

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("seed,k,read_len", [(1, 31, 75), (2, 21, 50), (3, 15, 36), (4, 31, 33), (5, 27, 150)])
def test_random_transcriptome_gpu(seed, k, read_len, tmp_path):
    idx, r1, r2, _ = make_case(str(tmp_path), seed, k, read_len, 1500)
    oix = O.OracleIndex(idx)
    ix = K.KmerIndex(idx, device=0)
    for paired in (True, False):
        for strand in (0, 1, 2):
            bases, off = O.to_batch(r1, r2 if paired else None)
            orun = O.OracleRun(oix, paired, strand, True)
            want = orun.pseudoalign(bases, off)
            oo, ot, oc = orun.ec_table()
            mc = K.MinCollector(ix, paired=paired, strand=strand)
            h = mc.process_buffer(bases, off)
            eo, et, ec, eh = mc.ec_table()
            np.testing.assert_array_equal(util.handles_to_ids(h, eh), want)
            assert util.ec_sets(eo, et) == util.ec_sets(oo, ot)
            np.testing.assert_array_equal(ec, oc)
            if paired:
                np.testing.assert_array_equal(mc.flens, orun.flens())
            mc.close()
    ix.close()
