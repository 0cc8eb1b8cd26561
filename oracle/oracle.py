"""ORACLE -- TEST INFRASTRUCTURE ONLY (see oracle/kb_oracle.cpp).

ctypes front-end of oracle/liboracle.so (the CPU restatement) plus helpers that run the
UNMODIFIED reference binary oracle/_ref/kallisto.  Imported only by tests/, bench.py's
cpu_baseline / --impl reference legs and __graft_entry__.smoke(); never by the product.
"""
import ctypes as C
import gzip
import os
import struct
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "liboracle.so")
REF_BIN = os.path.join(HERE, "_ref", "kallisto")


def build():
    """Compile the restatement (and, when /root/reference is present, the reference itself)."""
    src = os.path.join(HERE, "kb_oracle.cpp")
    if (not os.path.exists(LIB_PATH)) or os.path.getmtime(LIB_PATH) < os.path.getmtime(src):
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", src, "-o", LIB_PATH])
    if os.path.isdir("/root/reference/src") and not os.path.exists(REF_BIN):
        subprocess.check_call(["make", "-C", HERE, "-j8"], stdout=subprocess.DEVNULL)


_lib = None


def lib():
    global _lib
    if _lib is None:
        build()
        L = C.CDLL(LIB_PATH)
        L.oracle_index_load.restype = C.c_void_p
        L.oracle_index_load.argtypes = [C.c_char_p, C.c_char_p, C.c_int]
        L.oracle_index_free.argtypes = [C.c_void_p]
        for f in ("oracle_index_k", "oracle_index_n_targets", "oracle_index_n_unitigs"):
            getattr(L, f).argtypes = [C.c_void_p]
            getattr(L, f).restype = C.c_uint32
        for f in ("oracle_index_n_kmers", "oracle_index_n_blocks"):
            getattr(L, f).argtypes = [C.c_void_p]
            getattr(L, f).restype = C.c_uint64
        L.oracle_index_target_lens.argtypes = [C.c_void_p, C.c_void_p]
        L.oracle_index_target_name.argtypes = [C.c_void_p, C.c_uint32]
        L.oracle_index_target_name.restype = C.c_char_p
        L.oracle_run_create.restype = C.c_void_p
        L.oracle_run_create.argtypes = [C.c_void_p, C.c_int, C.c_int]
        L.oracle_run_free.argtypes = [C.c_void_p]
        L.oracle_run_set_fp.argtypes = [C.c_void_p, C.c_int]
        L.oracle_pseudoalign_batch.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32, C.c_int,
                                               C.c_void_p]
        L.oracle_n_ecs.argtypes = [C.c_void_p]
        L.oracle_n_ecs.restype = C.c_uint32
        L.oracle_n_ec_entries.argtypes = [C.c_void_p]
        L.oracle_n_ec_entries.restype = C.c_uint64
        L.oracle_n_find.argtypes = [C.c_void_p]
        L.oracle_n_find.restype = C.c_uint64
        L.oracle_ec_table.argtypes = [C.c_void_p] * 4
        L.oracle_get_flens.argtypes = [C.c_void_p, C.c_void_p]
        L.oracle_mean_fl_trunc.argtypes = [C.c_void_p, C.c_double, C.c_double, C.c_void_p]
        L.oracle_eff_lens.argtypes = [C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p]
        L.oracle_em.restype = C.c_int
        L.oracle_em.argtypes = [C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p,
                                C.c_int, C.c_int, C.c_void_p]
        L.oracle_tpm.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p]
        L.oracle_bootstrap_sample.argtypes = [C.c_void_p, C.c_uint32, C.c_uint64, C.c_int, C.c_void_p]
        _lib = L
    return _lib


def _p(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None else None


class OracleIndex:
    def __init__(self, path):
        err = C.create_string_buffer(256)
        self.h = lib().oracle_index_load(path.encode(), err, 256)
        if not self.h:
            raise RuntimeError(err.value.decode())
        L = lib()
        self.k = L.oracle_index_k(self.h)
        self.n_targets = L.oracle_index_n_targets(self.h)
        self.n_kmers = L.oracle_index_n_kmers(self.h)
        self.n_unitigs = L.oracle_index_n_unitigs(self.h)
        self.n_blocks = L.oracle_index_n_blocks(self.h)
        self.target_lens = np.zeros(self.n_targets, np.uint32)
        L.oracle_index_target_lens(self.h, _p(self.target_lens))
        self.target_names = [L.oracle_index_target_name(self.h, i).decode() for i in range(self.n_targets)]

    def __del__(self):
        if getattr(self, "h", None):
            lib().oracle_index_free(self.h)
            self.h = None


class OracleRun:
    """ReadProcessor::processBuffer + MasterProcessor::update, -t 1 semantics."""

    def __init__(self, index, paired=True, strand=0, collect_fld=True, fp_fl=-1):
        """fp_fl >= 0: the fragment-position filter of ProcessReads.cpp:1095-1136 ((int) of the -l value)."""
        self.index = index
        self.paired = paired
        self.collect_fld = collect_fld
        self.h = lib().oracle_run_create(index.h, int(paired), int(strand))
        if fp_fl >= 0:
            lib().oracle_run_set_fp(self.h, int(fp_fl))

    def __del__(self):
        if getattr(self, "h", None):
            lib().oracle_run_free(self.h)
            self.h = None

    def pseudoalign(self, bases, offsets=None, fixed_len=0):
        """bases: uint8 array; offsets: uint32 array (n_reads+1) or None with fixed_len."""
        bases = np.ascontiguousarray(bases, dtype=np.uint8)
        if offsets is not None:
            offsets = np.ascontiguousarray(offsets, dtype=np.uint32)
            n_reads = len(offsets) - 1
        else:
            n_reads = len(bases) // fixed_len
        n_frag = n_reads // 2 if self.paired else n_reads
        out = np.full(n_frag, -1, np.int32)
        lib().oracle_pseudoalign_batch(self.h, _p(bases), _p(offsets), n_reads, fixed_len, int(self.collect_fld), _p(out))
        return out

    def ec_table(self):
        L = lib()
        n = L.oracle_n_ecs(self.h)
        off = np.zeros(n + 1, np.uint64)
        tids = np.zeros(max(1, L.oracle_n_ec_entries(self.h)), np.uint32)
        counts = np.zeros(max(1, n), np.uint32)
        L.oracle_ec_table(self.h, _p(off), _p(tids), _p(counts))
        return off, tids[: int(off[n])], counts[:n]

    def flens(self):
        f = np.zeros(1000, np.uint32)
        lib().oracle_get_flens(self.h, _p(f))
        return f

    def n_find(self):
        return lib().oracle_n_find(self.h)


def mean_fl_trunc(flens, fld_mean=0.0, fld_sd=0.0):
    out = np.zeros(1000, np.float64)
    flens = np.ascontiguousarray(flens, np.uint32)
    lib().oracle_mean_fl_trunc(_p(flens), fld_mean, fld_sd, _p(out))
    return out


def eff_lens(target_lens, fl_trunc):
    target_lens = np.ascontiguousarray(target_lens, np.uint32)
    out = np.zeros(len(target_lens), np.float64)
    lib().oracle_eff_lens(_p(target_lens), len(target_lens), _p(fl_trunc), _p(out))
    return out


def em(off, tids, counts, eff, n_targets, counts_w=None, n_iter=10000, min_rounds=50):
    off = np.ascontiguousarray(off, np.uint64)
    tids = np.ascontiguousarray(tids, np.uint32)
    counts = np.ascontiguousarray(counts, np.uint32)
    cw = counts if counts_w is None else np.ascontiguousarray(counts_w, np.uint32)
    alpha = np.zeros(n_targets, np.float64)
    rounds = lib().oracle_em(len(counts), _p(off), _p(tids), _p(counts), _p(cw), n_targets, _p(eff), n_iter, min_rounds,
                             _p(alpha))
    return alpha, rounds


def tpm(est, eff):
    out = np.zeros(len(est), np.float64)
    lib().oracle_tpm(_p(np.ascontiguousarray(est)), _p(np.ascontiguousarray(eff)), len(est), _p(out))
    return out


def bootstrap_sample(counts, seed, b):
    counts = np.ascontiguousarray(counts, np.uint32)
    out = np.zeros(len(counts), np.uint32)
    lib().oracle_bootstrap_sample(_p(counts), len(counts), seed, b, _p(out))
    return out


def fmt_g6(x):
    """C++ default ostream formatting of a double (== printf %g with 6 significant digits)."""
    return "%g" % x


def abundance_tsv(names, lens, eff, est, tpm_):
    lines = ["target_id\tlength\teff_length\test_counts\ttpm"]
    for i in range(len(names)):
        lines.append("%s\t%d\t%s\t%s\t%s" % (names[i], lens[i], fmt_g6(eff[i]), fmt_g6(est[i]), fmt_g6(tpm_[i])))
    return "\n".join(lines) + "\n"


# ------------------------------------------------------------------------------------------
# FASTQ helpers (tests only; the product has its own reader)
# ------------------------------------------------------------------------------------------
def read_fastq(path):
    """-> list of sequences (bytes)."""
    op = gzip.open if path.endswith(".gz") else open
    seqs = []
    with op(path, "rb") as f:
        for i, line in enumerate(f):
            if i % 4 == 1:
                seqs.append(line.rstrip(b"\r\n"))
    return seqs


def to_batch(seqs1, seqs2=None):
    """-> (bases uint8, offsets uint32) with mates interleaved."""
    if seqs2 is not None:
        seqs = [s for pair in zip(seqs1, seqs2) for s in pair]
    else:
        seqs = list(seqs1)
    lens = np.fromiter((len(s) for s in seqs), dtype=np.int64, count=len(seqs))
    off = np.zeros(len(seqs) + 1, np.uint32)
    np.cumsum(lens, out=off[1:])
    bases = np.frombuffer(b"".join(seqs), dtype=np.uint8).copy()
    return bases, off


# ------------------------------------------------------------------------------------------
# the unmodified reference
# ------------------------------------------------------------------------------------------
def have_ref():
    return os.path.exists(REF_BIN)


def ref_run(args, cwd=None, check=True):
    return subprocess.run([REF_BIN] + list(args), cwd=cwd, check=check, stdout=subprocess.PIPE, stderr=subprocess.PIPE)


def ref_index(fasta, out, k=31, threads=1):
    # -T: the reference's scratch directory defaults to ./tmp, and the working directory may be read-only
    ref_run(["index", "-T", out + ".scratch", "-i", out, "-k", str(k), "-t", str(threads), fasta])
    return out


def index_unitig_kinds(path):
    """(n_long, n_short, n_abundant) from the GRAPH section of an index file (SURVEY.md 8b; ext/bifrost/src/IO.tcc:1635-1738)."""
    with open(path, "rb") as f:
        b = f.read()
    o = 16
    _magic, _k, _g, n_long = struct.unpack_from("<QiiQ", b, o)
    o += 24
    for _ in range(n_long):
        (ln,) = struct.unpack_from("<Q", b, o)
        o += 8 + (ln + 3) // 4
    (n_short,) = struct.unpack_from("<Q", b, o)
    o += 8 + 8 * n_short
    (n_abund,) = struct.unpack_from("<Q", b, o)
    return n_long, n_short, n_abund


def read_bus(path):
    """-> (header dict, structured array of records).  BUSData.h:30-38 / BUSTools.cpp:5-14"""
    with open(path, "rb") as f:
        magic = f.read(4)
        assert magic == b"BUS\0", magic
        version, bclen, umilen, tlen = struct.unpack("<IIII", f.read(16))
        text = f.read(tlen)
        dt = np.dtype([("barcode", "<u8"), ("umi", "<u8"), ("ec", "<i4"), ("count", "<u4"), ("flags", "<u4"),
                       ("pad", "<u4")])
        rec = np.frombuffer(f.read(), dtype=dt)
    return dict(version=version, bclen=bclen, umilen=umilen, text=text), rec


def read_matrix_ec(path):
    ecs = []
    with open(path) as f:
        for line in f:
            i, t = line.rstrip("\n").split("\t")
            assert int(i) == len(ecs)
            ecs.append(tuple(int(x) for x in t.split(",")))
    return ecs


def ref_ec_dump(index, outdir, files, paired=True, extra=()):
    """Per-fragment ECs from the unmodified reference: `kallisto bus -x bulk [--paired] -t 1`
    writes one BUS record per pseudoaligned fragment (flags = read number with --num), matrix.ec
    and flens.txt (SURVEY.md 8c)."""
    args = ["bus", "-x", "bulk", "-t", "1", "--num", "-i", index, "-o", outdir]
    if paired:
        args.append("--paired")
    args += list(extra) + list(files)
    ref_run(args)
    hdr, rec = read_bus(os.path.join(outdir, "output.bus"))
    ecs = read_matrix_ec(os.path.join(outdir, "matrix.ec"))
    flens = None
    fp = os.path.join(outdir, "flens.txt")
    if os.path.exists(fp):
        with open(fp) as f:
            flens = np.array([int(x) for x in f.read().split()], dtype=np.uint32)
    return rec, ecs, flens


# ------------------------------------------------------------------------------------------
# BUS records of a read set, restated (BUSProcessor::processBuffer, src/ProcessReads.cpp:1380-1832)
# ------------------------------------------------------------------------------------------
def string_to_binary(s):
    """stringToBinary (src/BUSData.cpp:8-36): 2-bit code of the first 32 letters + the N flag."""
    r, num_n, pos_n = 0, 0, 0
    for i, c in enumerate(s[:32]):
        x = (c & 4) >> 1
        if (c & 3) == 2:
            if num_n == 0:
                pos_n = i
            num_n += 1
        r = ((r << 2) | (x + ((x ^ (c & 2)) >> 1))) & 0xFFFFFFFFFFFFFFFF
    flag = 0
    if num_n > 0:
        flag = (min(num_n, 3) & 3) | ((pos_n & 31) << 2)
    return r, flag


def hamming(a, b, n):
    """hamming (src/BUSData.cpp:55-66): differing 2-bit symbols among the low n"""
    df = a ^ b
    return sum(1 for i in range(n) if (df >> (2 * i)) & 3)


def bus_model(index, files, bc, umi, seq, seq2=None, strand=0, num=False, samples=None, tag=None, sample_barcodes=None):
    """Records, EC sets, per-sample fragment-length histograms and barcode / UMI length histograms of `kallisto bus -t 1`.

    files: one list of sequences (bytes) per file of the technology; bc / umi: lists of (file, start, stop), bc == []
    = no barcode read (fake barcode: 0, or the sample's number), umi None = no UMI ("bulk_like", :1393); seq / seq2:
    (file, start) of the sequence read(s), seq2 given = busopt.paired; samples: list of (first set, end set) ranges that
    are samples of their own (`-x BULK`: barcode = sample number -- or sample_barcodes[i] for a --batch file whose lines
    share ids --, read numbers and fragment-length quota restart);
    tag: UMI tag sequence (`--tag`, SMARTSEQ3; umi[0].start already advanced by its length, src/main.cpp:1467-1468): a
    read set whose UMI is preceded by the tag (<= 1 mismatch when the tag is longer than 5) is a UMI read -- strand
    filter on, no fragment-length sampling; any other is an internal read -- UMI ~0, the whole read is sequence, no
    strand filter, fragment lengths sampled (:1497-1530,1545-1567).
    Records come out in read order (the reference writes the records of already-known ECs of a batch first,
    src/ProcessReads.cpp:1798-1812 + :603-612 -- compare sorted)."""
    n = len(files[0])
    paired = seq2 is not None
    by_sample = samples is not None
    samples = samples or [(0, n)]
    bc_hist = np.zeros(33, np.int64)
    umi_hist = np.zeros(33, np.int64)
    rec_bc, rec_umi, rec_fl, skip, notag = [0] * n, [0] * n, [0] * n, [False] * n, [False] * n
    taglen = len(tag) if tag else 0
    tag_bin = string_to_binary(tag)[0] if tag else 0

    def piece(i, f, a, b, back=0):          # :1505-1521 / :1592-1602: None = the slice does not fit
        l = len(files[f][i])
        ln = (l - a) if b == 0 else (b - a)
        if l < a + ln or ln <= 0:
            return None
        return files[f][i][a - back:a + ln]

    for si, (lo, hi) in enumerate(samples):
        for i in range(lo, hi):
            if umi is None:
                ulen, uval, uflag = 1, 0xFFFFFFFFFFFFFFFF, None
            else:
                parts = [piece(i, *u, back=(taglen if j == 0 else 0)) for j, u in enumerate(umi)]
                if any(p is None for p in parts):
                    skip[i] = True
                    continue
                us = b"".join(parts)
                ulen = len(us)
                uval, uflag = string_to_binary(us)
                if tag:
                    uflag = None                       # stringToBinary's flag of the UMI is dropped (local f, :1512-1513)
                    if hamming(tag_bin, uval >> (2 * (ulen - taglen)), taglen) <= (0 if taglen <= 5 else 1):
                        uval &= (1 << (2 * (ulen - taglen))) - 1
                        ulen -= taglen
                    else:
                        notag[i] = True
                        uval, ulen = 0xFFFFFFFFFFFFFFFF, 99
            if ulen <= 32:
                umi_hist[ulen] += 1
            if bc:
                parts = [piece(i, *b) for b in bc]
                if any(p is None for p in parts):
                    skip[i] = True
                    continue
                bs = b"".join(parts)
                blen = len(bs)
                bval, bflag = string_to_binary(bs)
            else:
                blen, bval, bflag = 16, ((sample_barcodes[si] if sample_barcodes else si) if by_sample else 0), 0
            if blen <= 32:
                bc_hist[blen] += 1
            if uflag is None:
                uflag = bflag       # no UMI / tag mode: stringToBinary ran once, for the barcode (:1736-1743)
            rec_bc[i], rec_umi[i] = bval, uval
            rec_fl[i] = (i - lo) if num else (bflag | (uflag << 8))

    # the sequence read(s): skipped sets have no sequence (they count as processed, :1372); an internal read of a tag
    # run starts where the tag would have started
    def seq_of(i, sq):
        if skip[i]:
            return b""
        st = sq[1]
        if notag[i] and umi[0][0] == sq[0]:
            st = umi[0][1] - taglen
        return files[sq[0]][i][st:]

    s1 = [seq_of(i, seq) for i in range(n)]
    s2 = [seq_of(i, seq2) for i in range(n)] if paired else None
    # groups of read sets that are pseudoaligned under different rules: (members, strand mode, samples fragment lengths)
    if tag:
        groups = [([not x for x in notag], strand, False), (list(notag), 0, True)]
    else:
        groups = [([True] * n, strand, True)]
    frag_set = [None] * n
    for members, smode, _ in groups:
        run = OracleRun(index, paired, smode, collect_fld=False)
        a1 = [s1[i] if members[i] else b"" for i in range(n)]
        a2 = [s2[i] if members[i] else b"" for i in range(n)] if paired else None
        bases, off = to_batch(a1, a2)
        frag = run.pseudoalign(bases, off)
        eo, et, ecn = run.ec_table()
        sets = [tuple(int(x) for x in et[int(eo[e]):int(eo[e + 1])]) for e in range(len(eo) - 1)]
        for i in range(n):
            if members[i] and frag[i] >= 0:
                frag_set[i] = sets[frag[i]]
    ids, ecs = {}, []
    for i in range(n):              # EC ids in order of first occurrence over the whole input
        if frag_set[i] is not None and frag_set[i] not in ids:
            ids[frag_set[i]] = len(ecs)
            ecs.append(frag_set[i])
    flens = []
    if paired:
        for lo, hi in samples:      # tlencounts[id]: 10 000 samples per sample (:486-493,1397-1400)
            f = np.zeros(1000, np.uint32)
            for members, smode, want in groups:
                if not want:
                    continue
                r = OracleRun(index, True, smode, collect_fld=True)
                b2, o2 = to_batch([s1[i] if members[i] else b"" for i in range(lo, hi)], [s2[i] if members[i] else b"" for i in range(lo, hi)])
                r.pseudoalign(b2, o2)
                f += r.flens()
            flens.append(f)
    dt = np.dtype([("barcode", "<u8"), ("umi", "<u8"), ("ec", "<i4"), ("count", "<u4"), ("flags", "<u4"), ("pad", "<u4")])
    keep = [i for i in range(n) if frag_set[i] is not None]
    rec = np.zeros(len(keep), dt)
    for j, i in enumerate(keep):
        rec[j] = (rec_bc[i], rec_umi[i], ids[frag_set[i]], 1, rec_fl[i] & 0xFFFFFFFF, 0)
    return dict(records=rec, ecs=ecs, flens=flens, bc_hist=bc_hist, umi_hist=umi_hist, n_processed=n)
