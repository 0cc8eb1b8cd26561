"""CPU: option validation of the kallisto_b200 command line against the unmodified reference binary
(CheckOptionsEM / CheckOptionsBus, src/main.cpp:1283-1805): same exit code and the same `Error:` lines for
invocations that are rejected before any device work.  The reference's answers are stored in
tests/golden/cli_errors.json (`python -m tests.test_cli_args_host` rewrites it with oracle/_ref/kallisto)."""
import json
import os
import subprocess
import sys

import pytest

from oracle import oracle as O
from tests import util

BIN = os.path.join(util.ROOT, "kallisto_b200", "kallisto_b200")
GOLDEN_ERRORS = os.path.join(util.GOLDEN, "cli_errors.json")
pytestmark = pytest.mark.skipif(not os.path.exists(BIN), reason="needs the kallisto_b200 CLI")

D = os.path.join(util.GOLDEN, "config1")
IDX, R1, R2 = (os.path.join(D, f) for f in ("transcripts.kidx", "reads_1.fastq.gz", "reads_2.fastq.gz"))
B1, B2 = (os.path.join(util.GOLDEN, "bus10x", f) for f in ("sc_reads_1.fastq.gz", "sc_reads_2.fastq.gz"))

CASES = [
    ["quant", "-i", "nope.kidx", "-o", "o", R1, R2],
    ["quant", "-i", IDX, "-o", "o", R1],
    ["quant", "-i", IDX, "-o", "o", "--single", R1],
    ["quant", "-i", IDX, "-o", "o", "--single", "-l", "200", R1],
    ["quant", "-i", IDX, "-o", "o", "--single", "-l", "-5", "-s", "20", R1],
    ["quant", "-i", IDX, "-o", "o", "--single", "-l", "200", "-s", "0", R1],
    ["quant", "-i", IDX, "-o", "o", "-t", "0", R1, R2],
    ["quant", "-i", IDX, "-o", "o", "missing_1.fq", "missing_2.fq"],
    ["quant", "-i", IDX, R1, R2],
    ["quant", "-o", "o", R1, R2],
    ["quant", "-i", IDX, "-o", "o", "-b", "-3", "--plaintext", R1, R2],
    ["quant", "-i", IDX, "-o", "o"],
    ["bus", "-i", "nope.kidx", "-o", "o", "-x", "10xv2", B1, B2],
    ["bus", "-i", IDX, "-o", "o", B1, B2],
    ["bus", "-i", IDX, "-o", "o", "-x", "10xv2", B1],
    ["bus", "-i", IDX, "-o", "o", "-x", "nosuchtech", B1, B2],
    ["bus", "-i", IDX, "-o", "o", "-x", "10xv2", "-t", "0", B1, B2],
    ["bus", "-i", IDX, "-x", "10xv2", B1, B2],
    ["bus", "-i", IDX, "-o", "o", "-x", "10xv2", "missing_1.fq", "missing_2.fq"],
    ["bus", "-i", IDX, "-o", "o", "-x", "0,0,16:0,16,26", B1, B2],
    ["bus", "-i", IDX, "-o", "o", "-x", "0,0,16:0,16,26:1,0,0:1,0,0", B1, B2],
    ["bus", "-i", IDX, "-o", "o", "-x", "0,0,16:0,16,26:1,0,0", B1],
    ["bus", "-o", "o", "-x", "10xv2", B1, B2],
    ["bus", "-i", IDX, "-o", "o", "-x", "bulk", "--paired", R1],
    ["bus", "-i", IDX, "-o", "o", "-x", "10xv2", "--paired", B1, B2],
    ["bus", "-i", IDX, "-o", "o", "-x", "STORM-seq", R1, R2],          # upper-cased before it is compared: not selectable (src/main.cpp:619,1358)
    ["bus", "-i", IDX, "-o", "o", "-x", "smartseq2", R1, R2],          # three files without --paired
    ["bus", "-i", IDX, "-o", "o", "-x", "0,0,8:1,0,8:1,22,0", "--tag", "ATTGCGCAATG", B1, B2],   # the UMI location must hold tag + UMI
    ["bus", "-i", IDX, "-o", "o", "-x", "bulk", "--tag", "ACGTAC", R1],
    ["bus", "-i", IDX, "-o", "o", "-x", "smartseq3", R1, R2],          # four files
    ["bus", "-i", IDX, "-o", "o", "-x", "10xv2", "--inleaved", B1, B2],
    ["bus", "-i", IDX, "-o", "o", "--batch", "nope.txt"],
    ["bus", "-i", IDX, "-o", "o", "--batch", IDX, R1],                 # read files next to a batch file
    ["quant", "-i", IDX, "-o", "o", "--single", "-l", "200", "-s", "20"],
    ["quant", "-i", IDX, "-o", "o", "-t", "-2", "--single", "-l", "200", "-s", "20", R1],
]


def errors(binary, args, cwd):
    r = subprocess.run([binary] + args, cwd=cwd, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=120)
    return r.returncode, [l.strip() for l in r.stderr.splitlines() if l.startswith("Error")]


def case_key(args):
    return " ".join(os.path.relpath(x, util.ROOT) if os.path.isabs(x) else x for x in args)


def reference_errors():
    with open(GOLDEN_ERRORS) as f:
        return {c["args"]: (c["exit_code"], c["errors"]) for c in json.load(f)}


@pytest.mark.parametrize("args", CASES, ids=lambda a: " ".join(os.path.basename(x) for x in a)[:60])
def test_rejected_like_the_reference(args, tmp_path):
    want = reference_errors()[case_key(args)]
    got = errors(BIN, args, str(tmp_path))
    assert want[0] != 0, "the reference accepts this invocation: not a validation case"
    assert got == want


if __name__ == "__main__":
    # rewrite the fixture from the unmodified reference binary
    import tempfile
    out = []
    for args in CASES:
        with tempfile.TemporaryDirectory() as td:
            rc, lines = errors(O.REF_BIN, args, td)
        out.append({"args": case_key(args), "exit_code": rc, "errors": lines})
    with open(GOLDEN_ERRORS, "w") as f:
        json.dump(out, f, indent=1)
        f.write("\n")
    sys.exit(0)
