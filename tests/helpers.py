"""Shared test helpers: ctypes bindings for the oracle (oracle/liboracle.so), the compiled reference
(oracle/_ref/*), the workload generator (tools/libkjgen.so) and small workload builders.

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline leg may touch oracle/.
Nothing here reads /root/reference at run time (oracle/_ref holds prebuilt binaries).
"""
import ctypes as C
import os
import subprocess
import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ORACLE_DIR = os.path.join(ROOT, "oracle")
REF_DIR = os.path.join(ORACLE_DIR, "_ref")
TOOLS_DIR = os.path.join(ROOT, "tools")
GOLDEN_DIR = os.path.join(ROOT, "tests", "golden")


def have_ref():
    return all(os.path.exists(os.path.join(REF_DIR, f)) for f in ("kaiju", "kaiju-mkbwt", "kaiju-mkfmi", "libkaijuref.so"))


class KoParams(C.Structure):
    _fields_ = [("mode", C.c_int), ("min_fragment_length", C.c_uint32), ("mismatches", C.c_uint32),
                ("min_score", C.c_uint32), ("seed_length", C.c_uint32), ("use_evalue", C.c_int),
                ("min_evalue", C.c_double), ("seg", C.c_int), ("input_is_protein", C.c_int)]


class KoCounters(C.Structure):
    _fields_ = [(n, C.c_uint64) for n in ("reads", "initial_si", "update_si", "fmindex", "scanned_bytes", "get_suffix",
                                          "lf_steps", "seg_calls", "seg_hits", "fragments_initial", "fragments_searched",
                                          "bases", "classified")]

    def as_dict(self):
        return {n: int(getattr(self, n)) for n, _ in self._fields_}


def make_params(mode="mem", m=11, e=3, s=65, seed=7, E=0.01, seg=True, protein=False):
    greedy = mode == "greedy"
    return dict(mode=1 if greedy else 0, min_fragment_length=m, mismatches=e, min_score=s, seed_length=seed,
                use_evalue=1 if greedy else 0, min_evalue=E, seg=1 if seg else 0, input_is_protein=1 if protein else 0)


_oracle = None


def oracle_lib():
    global _oracle
    if _oracle is None:
        path = os.path.join(ORACLE_DIR, "liboracle.so")
        if not os.path.exists(path):
            subprocess.check_call(["make", "-C", ORACLE_DIR, "oracle"], stdout=subprocess.DEVNULL)
        L = C.CDLL(path)
        L.ko_index_load.restype = C.c_void_p; L.ko_index_load.argtypes = [C.c_char_p]
        L.ko_index_free.argtypes = [C.c_void_p]
        L.ko_index_bwtlen.restype = C.c_int64; L.ko_index_bwtlen.argtypes = [C.c_void_p]
        L.ko_index_alen.restype = C.c_int; L.ko_index_alen.argtypes = [C.c_void_p]
        L.ko_index_nseq.restype = C.c_int; L.ko_index_nseq.argtypes = [C.c_void_p]
        L.ko_index_seq_taxon.restype = C.c_uint64; L.ko_index_seq_taxon.argtypes = [C.c_void_p, C.c_int]
        L.ko_fmindex.restype = C.c_int64; L.ko_fmindex.argtypes = [C.c_void_p, C.c_int, C.c_int64]
        L.ko_get_suffix.argtypes = [C.c_void_p, C.c_int64, C.POINTER(C.c_int), C.POINTER(C.c_int64)]
        L.ko_tax_load.restype = C.c_void_p; L.ko_tax_load.argtypes = [C.c_char_p]
        L.ko_tax_free.argtypes = [C.c_void_p]
        L.ko_lca.restype = C.c_uint64; L.ko_lca.argtypes = [C.c_void_p, C.POINTER(C.c_uint64), C.c_int]
        L.ko_seg.restype = C.c_int; L.ko_seg.argtypes = [C.c_char_p, C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int), C.c_int]
        L.ko_lnfact.restype = C.c_double; L.ko_lnfact.argtypes = [C.c_int]
        L.ko_classify.restype = C.c_uint64
        L.ko_classify.argtypes = [C.c_void_p, C.c_void_p, C.POINTER(KoParams), C.c_char_p, C.c_int, C.c_char_p, C.c_int,
                                  C.POINTER(C.c_uint32), C.POINTER(C.c_uint64), C.POINTER(C.c_int), C.POINTER(KoCounters)]
        L.ko_classify_batch.argtypes = [C.c_void_p, C.c_void_p, C.POINTER(KoParams), C.c_void_p, C.c_void_p, C.c_void_p,
                                        C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p, C.POINTER(KoCounters)]
        L.ko_fragments.restype = C.c_int; L.ko_fragments.argtypes = [C.c_char_p, C.c_int, C.c_int, C.c_char_p, C.c_int]
        _oracle = L
    return _oracle


class Oracle:
    """CPU restatement (oracle/kaiju_oracle.c) bound to one index + taxonomy."""

    def __init__(self, fmi_path, nodes_path):
        self.L = oracle_lib()
        self.idx = self.L.ko_index_load(fmi_path.encode())
        assert self.idx, "oracle could not load " + fmi_path
        self.tax = self.L.ko_tax_load(nodes_path.encode())
        assert self.tax, "oracle could not load " + nodes_path

    def classify_batch(self, params, seq1, off1, seq2=None, off2=None, counters=None):
        n = len(off1) - 1
        P = KoParams(**params)
        tax = np.zeros(n, dtype=np.uint64); best = np.zeros(n, dtype=np.uint32)
        seq1 = np.ascontiguousarray(seq1, dtype=np.uint8); off1 = np.ascontiguousarray(off1, dtype=np.uint64)
        p2 = o2 = None
        if seq2 is not None:
            seq2 = np.ascontiguousarray(seq2, dtype=np.uint8); off2 = np.ascontiguousarray(off2, dtype=np.uint64)
            p2, o2 = seq2.ctypes.data, off2.ctypes.data
        self.L.ko_classify_batch(self.idx, self.tax, C.byref(P), seq1.ctypes.data, off1.ctypes.data, p2, o2, n,
                                 tax.ctypes.data, best.ctypes.data, C.byref(counters) if counters is not None else None)
        return tax, best

    def classify_one(self, params, s1, s2=None):
        P = KoParams(**params)
        best = C.c_uint32(0); ids = (C.c_uint64 * 64)(); nids = C.c_int(0)
        t = self.L.ko_classify(self.idx, self.tax, C.byref(P), s1, len(s1), s2, len(s2) if s2 is not None else 0,
                               C.byref(best), ids, C.byref(nids), None)
        return int(t), int(best.value), [int(ids[i]) for i in range(min(nids.value, 32))]


_kjgen = None


def kjgen_lib():
    global _kjgen
    if _kjgen is None:
        path = os.path.join(TOOLS_DIR, "libkjgen.so")
        if not os.path.exists(path):
            subprocess.check_call(["gcc", "-O2", "-fPIC", "-shared", "-fopenmp", "-o", path, os.path.join(TOOLS_DIR, "kjgen.c"), "-lm"])
        L = C.CDLL(path)
        L.kjgen_db_create.restype = C.c_void_p; L.kjgen_db_create.argtypes = [C.c_int64, C.c_uint64]
        L.kjgen_db_free.argtypes = [C.c_void_p]
        L.kjgen_db_nletters.restype = C.c_int64; L.kjgen_db_nletters.argtypes = [C.c_void_p]
        L.kjgen_db_write.restype = C.c_int; L.kjgen_db_write.argtypes = [C.c_void_p, C.c_char_p, C.c_char_p]
        L.kjgen_reads_packed.argtypes = [C.c_void_p, C.c_uint64, C.c_uint64, C.c_int64, C.c_int, C.c_int,
                                         C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        for fn in (L.kjgen_long_reads_packed, L.kjgen_protein_reads_packed):
            fn.argtypes = [C.c_void_p, C.c_uint64, C.c_uint64, C.c_int64, C.c_int, C.c_int, C.c_void_p, C.c_void_p]
        L.kjgen_reads_write_fastq.restype = C.c_int
        L.kjgen_reads_write_fastq.argtypes = [C.c_void_p, C.c_uint64, C.c_uint64, C.c_int64, C.c_int, C.c_int, C.c_char_p, C.c_char_p]
        _kjgen = L
    return _kjgen


class SynthDB:
    """Deterministic synthetic protein DB + taxonomy (tools/kjgen.c)."""

    def __init__(self, nprot, seed):
        self.L = kjgen_lib(); self.nprot = nprot; self.seed = seed
        self.h = self.L.kjgen_db_create(nprot, seed)

    def write(self, faa, nodes):
        assert self.L.kjgen_db_write(self.h, faa.encode(), nodes.encode()) == 0

    def reads(self, seed, first, n, readlen=150, paired=True):
        s1 = np.empty(n * readlen, dtype=np.uint8); o1 = np.empty(n + 1, dtype=np.uint64)
        s2 = np.empty(n * readlen if paired else 1, dtype=np.uint8); o2 = np.empty(n + 1, dtype=np.uint64)
        self.L.kjgen_reads_packed(self.h, seed, first, n, readlen, 1 if paired else 0,
                                  s1.ctypes.data, o1.ctypes.data, s2.ctypes.data, o2.ctypes.data)
        s1 = s1[:int(o1[n])]
        if paired:
            return s1, o1, s2[:int(o2[n])], o2
        return s1, o1, None, None

    def _varlen(self, fn, seed, first, n, minlen, maxlen):
        s = np.empty(n * maxlen, dtype=np.uint8); o = np.empty(n + 1, dtype=np.uint64)
        fn(self.h, seed, first, n, minlen, maxlen, s.ctypes.data, o.ctypes.data)
        return s[:int(o[n])].copy(), o

    def long_reads(self, seed, first, n, minlen, maxlen):
        """Variable-length DNA reads (segments of coding / random / low-complexity sequence), single-end."""
        return self._varlen(self.L.kjgen_long_reads_packed, seed, first, n, minlen, maxlen)

    def protein_reads(self, seed, first, n, minlen, maxlen):
        """Protein input for -p: residues plus the characters that split a read (X, *, B, Z, digits ...)."""
        return self._varlen(self.L.kjgen_protein_reads_packed, seed, first, n, minlen, maxlen)

    def write_fastq(self, seed, first, n, readlen, paired, fq1, fq2=None):
        assert self.L.kjgen_reads_write_fastq(self.h, seed, first, n, readlen, 1 if paired else 0, fq1.encode(),
                                              fq2.encode() if fq2 else None) == 0


def build_fmi(faa, prefix, threads=8, exponent=3):
    """Build <prefix>.fmi with the reference's own index tools (test-data tooling, SURVEY.md 8c)."""
    env = dict(os.environ)
    subprocess.check_call([os.path.join(REF_DIR, "kaiju-mkbwt"), "-n", str(threads), "-e", str(exponent), "-a",
                           "ACDEFGHIKLMNPQRSTVWY", "-o", prefix, faa], stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL, env=env)
    subprocess.check_call([os.path.join(REF_DIR, "kaiju-mkfmi"), prefix], stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL, env=env)
    for ext in (".bwt", ".sa"):
        try:
            os.remove(prefix + ext)
        except OSError:
            pass
    return prefix + ".fmi"


def run_ref_kaiju(nodes, fmi, fq1, fq2=None, mode="mem", m=11, e=3, s=65, E=None, seg=True, threads=1, verbose=True, out=None, protein=False):
    """Run the unmodified reference CLI; returns {name: (C/U, taxon, best, ids)}."""
    cmd = [os.path.join(REF_DIR, "kaiju"), "-t", nodes, "-f", fmi, "-i", fq1, "-a", mode, "-m", str(m), "-z", str(threads)]
    if fq2:
        cmd += ["-j", fq2]
    if mode == "greedy":
        cmd += ["-e", str(e), "-s", str(s)]
        if E is not None:
            cmd += ["-E", repr(E)]
    if not seg:
        cmd += ["-X"]
    if protein:
        cmd += ["-p"]
    if verbose:
        cmd += ["-v"]
    txt = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, check=True).stdout.decode()
    if out:
        with open(out, "w") as f:
            f.write(txt)
    return parse_kaiju_output(txt)


def parse_kaiju_output(txt):
    res = {}
    for line in txt.splitlines():
        p = line.split("\t")
        if len(p) < 3:
            continue
        best = int(p[3]) if len(p) > 3 and p[3] else 0
        ids = tuple(sorted(int(t) for t in p[4].split(",") if t)) if len(p) > 4 else ()
        res[p[1]] = (p[0], int(p[2]), best, ids)
    return res


def read_fastq_packed(path):
    """FASTQ -> (names, seq bytes, offsets) with kaiju.cpp:318-335 name trimming and strip()."""
    names, seqs = [], []
    with open(path) as f:
        while True:
            h = f.readline()
            if not h:
                break
            if not h.strip():
                continue
            s = f.readline().rstrip("\n"); f.readline(); f.readline()
            name = h[1:].rstrip("\n")
            for i, ch in enumerate(name):
                if ch in " /\t\r":
                    name = name[:i]; break
            names.append(name)
            seqs.append("".join(c for c in s if c.isalpha()))
    off = np.zeros(len(seqs) + 1, dtype=np.uint64)
    off[1:] = np.cumsum([len(s) for s in seqs])
    data = np.frombuffer("".join(seqs).encode(), dtype=np.uint8).copy()
    return names, data, off


def make_quirk_db(d, nprot=512, plen=255, seed=9, nreads=3000, build=False):
    """A DB whose BWT length is an exact multiple of 2^16 (nprot * (plen + 1) = 131072 rows by default): the case in which the
    reference's FM-index checkpoints misbehave for the last 129 positions (fmicommon.h:60-73, 88-89).  Returns (fmi, nodes, read
    strings).  The index of the default DB is committed (tests/golden/quirk_db.fmi, built by the reference's kaiju-mkbwt/-mkfmi);
    build=True builds it with oracle/_ref."""
    import random
    rnd = random.Random(seed); aa = "ACDEFGHIKLMNPQRSTVWY"
    assert (nprot * (plen + 1)) % 65536 == 0
    prots = ["".join(rnd.choice(aa) for _ in range(plen)) for _ in range(nprot)]
    with open(d + "/db.faa", "w") as f:
        for i, p in enumerate(prots):
            f.write(">P%d_%d\n%s\n" % (i, 100 + i % 7, p))
    with open(d + "/nodes.dmp", "w") as f:
        f.write("1\t|\t1\t|\tno rank\t|\n")
        for t in range(100, 107):
            f.write("%d\t|\t1\t|\tspecies\t|\n" % t)
    if build:
        fmi = build_fmi(d + "/db.faa", d + "/db", threads=2)
    else:
        assert (nprot, plen, seed) == (512, 255, 9), "only the default quirk DB has a committed index"
        fmi = os.path.join(GOLDEN_DIR, "quirk_db.fmi")
    codon = {'A': 'GCT', 'R': 'CGT', 'N': 'AAT', 'D': 'GAT', 'C': 'TGT', 'Q': 'CAA', 'E': 'GAA', 'G': 'GGT', 'H': 'CAT', 'I': 'ATT',
             'L': 'CTG', 'K': 'AAA', 'M': 'ATG', 'F': 'TTT', 'P': 'CCT', 'S': 'TCT', 'T': 'ACT', 'W': 'TGG', 'Y': 'TAT', 'V': 'GTT'}
    reads = []
    for i in range(nreads):
        p = rnd.choice(prots); s0 = rnd.randrange(0, len(p) - 50)
        dna = "".join(codon[c] for c in p[s0:s0 + 50])
        dna = "".join(ch if rnd.random() > 0.02 else rnd.choice("ACGT") for ch in dna)
        if rnd.random() < 0.5:
            dna = dna[::-1].translate(str.maketrans("ACGT", "TGCA"))
        reads.append(dna)
    return fmi, d + "/nodes.dmp", reads


def pack_reads(reads):
    seq = np.frombuffer("".join(reads).encode(), dtype=np.uint8)
    off = np.zeros(len(reads) + 1, np.uint64); off[1:] = np.cumsum([len(r) for r in reads])
    return seq, off
