#!/usr/bin/env python
"""Generates the committed golden fixtures by running the UNMODIFIED reference (oracle/_ref, built by
oracle/Makefile from /root/reference) on seeded synthetic inputs.  Run in the build container:

    make -C oracle ref && python tests/golden/make_golden.py

Outputs (all small, committed):
    db.fmi, nodes.dmp            index built by the reference's kaiju-mkbwt/kaiju-mkfmi (-e 3) from a seeded
                                 800-protein DB (tools/kjgen.c) + adversarial extras (see below)
    se100.fq.gz                  2,000 single-end 100 bp reads  (BASELINE.json configs[0] shape)
    pe150_1.fq.gz, pe150_2.fq.gz 1,500 paired 150 bp reads + hand-made adversarial reads
    expected_<cfg>.tsv.gz        reference `kaiju -v` output (status, name, taxon, best length/score, id set)
    fmindex_kat.npz              FMindex(c,k) for every letter at 4,000 positions + get_suffix at 2,000 rows,
                                 taken from the reference's own C functions (libkaijuref.so)
    seg_kat.json                 SeqBufferSeg regions of 300 sequences from the reference
"""
import ctypes as C
import gzip, json, os, random, subprocess, sys
import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
from helpers import SynthDB, build_fmi, run_ref_kaiju, REF_DIR, kjgen_lib   # noqa: E402

CONFIGS = {
    "mem_default": dict(mode="mem"),
    "mem_noseg": dict(mode="mem", seg=False),
    "mem_m5": dict(mode="mem", m=5),
    "greedy_default": dict(mode="greedy"),
    "greedy_e5": dict(mode="greedy", e=5),
    "greedy_e1_s40": dict(mode="greedy", e=1, s=40),
    "greedy_e0": dict(mode="greedy", e=0),
    "greedy_noseg": dict(mode="greedy", seg=False),
}
CODON = {'A': 'GCT', 'R': 'CGT', 'N': 'AAT', 'D': 'GAT', 'C': 'TGT', 'Q': 'CAA', 'E': 'GAA', 'G': 'GGT', 'H': 'CAT', 'I': 'ATT',
         'L': 'CTG', 'K': 'AAA', 'M': 'ATG', 'F': 'TTT', 'P': 'CCT', 'S': 'TCT', 'T': 'ACT', 'W': 'TGG', 'Y': 'TAT', 'V': 'GTT'}


def revcomp(s):
    return s[::-1].translate(str.maketrans("ACGTacgtN", "TGCAtgcaN"))


def write_db_faa(faa, nodes):
    """The golden DB as FASTA + nodes.dmp (the input of db.fmi); returns the DB, the random generator in its state after the DB and
    the adversarial proteins (capped, same, plain, zero, lowc)."""
    rnd = random.Random(20240607)
    db = SynthDB(800, 3)
    db.write(faa, nodes)
    node_ids = [int(l.split()[0]) for l in open(nodes)]
    leaves = [node_ids[5 + (i % (len(node_ids) - 5))] for i in range(200)]     # any node may carry proteins
    assert len(set(leaves[i] for i in range(30))) == 30
    # adversarial extras: one protein replicated over 30 taxa (21-id cap), one over 25 copies of ONE taxon (long interval,
    # one id), names without '_' (whole name is the taxon), a name with a non-numeric suffix (taxon 0), a taxon missing from nodes.dmp
    aa = "ACDEFGHIKLMNPQRSTVWY"
    capped = "".join(rnd.choice(aa) for _ in range(140))
    same = "".join(rnd.choice(aa) for _ in range(120))
    plain = "".join(rnd.choice(aa) for _ in range(90))
    zero = "".join(rnd.choice(aa) for _ in range(90))
    lowc = "".join(rnd.choice(aa) for _ in range(40)) + "QQQQQQQQQQQQQQQQQQ" + "".join(rnd.choice(aa) for _ in range(40)) + "SGSGSGSGSGSGSGSG" + "".join(rnd.choice(aa) for _ in range(30))
    with open(faa, "a") as f:
        for i in range(30):
            f.write(">CAP%d_%d\n%s\n" % (i, leaves[i], capped))
        for i in range(25):
            f.write(">SAME%d_%d\n%s\n" % (i, leaves[40], same))
        f.write(">%d\n%s\n" % (leaves[45], plain))
        f.write(">WEIRD_xyz\n%s\n" % zero)
        f.write(">MISSING_7777777\n%s\n" % zero[::-1])
        for i in range(3):
            f.write(">LOWC%d_%d\n%s\n" % (i, leaves[50 + i], lowc))
    return db, rnd, (capped, same, plain, zero, lowc)


def main():
    faa, nodes = os.path.join(HERE, "db.faa"), os.path.join(HERE, "nodes.dmp")
    db, rnd, (capped, same, plain, zero, lowc) = write_db_faa(faa, nodes)
    aa = "ACDEFGHIKLMNPQRSTVWY"
    fmi = build_fmi(faa, os.path.join(HERE, "db"), threads=4)
    os.remove(faa)

    def bt(p):
        return "".join(CODON[c] for c in p)

    adv = []   # (name, mate1, mate2)
    adv.append(("adv_cap", bt(capped[10:60]), revcomp(bt(capped[80:130]))))
    adv.append(("adv_cap_short", bt(capped[20:33]) + "TAA" + "ACGT" * 20, "ACGTTGCA" * 18))
    adv.append(("adv_same", bt(same[5:55]), revcomp(bt(same[60:110]))))
    adv.append(("adv_plain", bt(plain[3:53]), revcomp(bt(plain[30:80]))))
    adv.append(("adv_zero", bt(zero[3:53]), revcomp(bt(zero[30:80]))))
    adv.append(("adv_missing", bt(zero[::-1][3:53]), "A" * 150))
    adv.append(("adv_lowc1", bt(lowc[20:70]), revcomp(bt(lowc[70:120]))))
    adv.append(("adv_lowc2", "C" + bt(lowc[30:79]) + "AG", revcomp(bt(lowc[60:110]))))
    adv.append(("adv_homopolymer", "A" * 150, "T" * 150))
    adv.append(("adv_dinuc", "AG" * 75, "CT" * 75))
    adv.append(("adv_trinuc", "CAG" * 50, "GCA" * 50))
    adv.append(("adv_N", bt(capped[10:30]) + "N" + bt(capped[31:59])[1:], "N" * 150))
    adv.append(("adv_lower", bt(same[5:55]).lower(), revcomp(bt(same[60:110])).lower()))
    adv.append(("adv_iupac", bt(plain[3:30]) + "RYKM" + bt(plain[32:50]), "ACGU" * 37))
    adv.append(("adv_short_both", "ACGTACGTACGTACGTAC", "ACGTACGTAC"))
    adv.append(("adv_short_one", "ACGTACGTACGTACGTAC", revcomp(bt(capped[80:130]))))
    adv.append(("adv_len32", bt(capped[10:20]) + "AC", bt(capped[10:21])))
    adv.append(("adv_len33", bt(capped[10:21]), bt(capped[40:51])))
    adv.append(("adv_empty2", bt(capped[10:60]), ""))
    adv.append(("adv_stop_heavy", "TAATAGTGA" * 16, bt(capped[0:50])))
    # paired file
    L = kjgen_lib()
    tmp1, tmp2 = os.path.join(HERE, "_pe1.fq"), os.path.join(HERE, "_pe2.fq")
    db.write_fastq(5, 0, 1500, 150, True, tmp1, tmp2)
    with open(tmp1, "a") as f1, open(tmp2, "a") as f2:
        for name, a, b in adv:
            f1.write("@%s/1\n%s\n+\n%s\n" % (name, a, "I" * len(a)))
            f2.write("@%s/2\n%s\n+\n%s\n" % (name, b, "I" * len(b)))
    tmps = os.path.join(HERE, "_se.fq")
    db.write_fastq(9, 0, 2000, 100, False, tmps)
    with open(tmps, "a") as f1:
        for name, a, b in adv:
            f1.write("@%s\n%s\n+\n%s\n" % (name, a[:100], "I" * len(a[:100])))
    for cfg, kw in CONFIGS.items():
        for tag, args in (("pe150", (tmp1, tmp2)), ("se100", (tmps, None))):
            res = run_ref_kaiju(nodes, fmi, args[0], args[1], threads=1, **kw)
            names = [l[1:].split("/")[0].strip() for i, l in enumerate(open(args[0])) if i % 4 == 0]
            with gzip.open(os.path.join(HERE, "expected_%s_%s.tsv.gz" % (cfg, tag)), "wt") as f:
                for nm in names:
                    r = res[nm]
                    f.write("%s\t%s\t%d\t%d\t%s\n" % (r[0], nm, r[1], r[2], ",".join(map(str, r[3]))))
    for src, dst in ((tmp1, "pe150_1.fq.gz"), (tmp2, "pe150_2.fq.gz"), (tmps, "se100.fq.gz")):
        with open(src, "rb") as a, gzip.open(os.path.join(HERE, dst), "wb") as b:
            b.write(a.read())
        os.remove(src)

    # ---- function-level known answers from the reference's own C code
    R = C.CDLL(os.path.join(REF_DIR, "libkaijuref.so"))
    libc = C.CDLL(None)
    libc.fopen.restype = C.c_void_p; libc.fopen.argtypes = [C.c_char_p, C.c_char_p]
    R.readIndexes.restype = C.c_void_p; R.readIndexes.argtypes = [C.c_void_p]
    fp = libc.fopen(fmi.encode(), b"r")
    bwt = R.readIndexes(fp)

    class BWT(C.Structure):   # bwt/bwt.h:13-23
        _fields_ = [("len", C.c_long), ("nseq", C.c_int), ("bwt", C.c_void_p), ("alen", C.c_int), ("alphabet", C.c_char_p), ("f", C.c_void_p), ("s", C.c_void_p)]

    class FMI(C.Structure):   # bwt/compactfmi.h:10-19
        _fields_ = [("alen", C.c_int), ("bwtlen", C.c_long), ("bwt", C.c_void_p), ("N1", C.c_int), ("N2", C.c_int), ("index1", C.c_void_p), ("index2", C.c_void_p), ("startLcode", C.c_void_p)]
    b = BWT.from_address(bwt); fm = FMI.from_address(b.f)
    R.FMindex.restype = C.c_long; R.FMindex.argtypes = [C.c_void_p, C.c_ubyte, C.c_long]
    R.get_suffix.argtypes = [C.c_void_p, C.c_void_p, C.c_long, C.POINTER(C.c_int), C.POINTER(C.c_long)]
    n = fm.bwtlen
    ks = sorted(set([0, 1, 127, 128, 129, 255, 256, 257, 65535, 65536, 65537, n - 1, n] + [rnd.randrange(0, n + 1) for _ in range(4000)]))
    ks = [k for k in ks if 0 <= k <= n]
    fmv = np.array([[R.FMindex(b.f, c, k) for c in range(fm.alen)] for k in ks], dtype=np.int64)
    rows = sorted(set(rnd.randrange(0, n) for _ in range(2000)))
    iseq = C.c_int(); pos = C.c_long(); sfx = []
    for k in rows:
        R.get_suffix(b.f, b.s, k, C.byref(iseq), C.byref(pos)); sfx.append((iseq.value, pos.value))
    np.savez_compressed(os.path.join(HERE, "fmindex_kat.npz"), ks=np.array(ks, dtype=np.int64), fmindex=fmv,
                        rows=np.array(rows, dtype=np.int64), suffix=np.array(sfx, dtype=np.int64), bwtlen=n, alen=fm.alen)

    # SEG known answers
    class SSeqRange(C.Structure):
        _fields_ = [("left", C.c_int), ("right", C.c_int)]

    class BlastSeqLoc(C.Structure):
        pass
    BlastSeqLoc._fields_ = [("next", C.POINTER(BlastSeqLoc)), ("ssr", C.POINTER(SSeqRange))]
    R.SegParametersNewAa.restype = C.c_void_p
    R.SeqBufferSeg.argtypes = [C.c_char_p, C.c_int, C.c_int, C.c_void_p, C.POINTER(C.POINTER(BlastSeqLoc))]
    sp = R.SegParametersNewAa()

    class SegParameters(C.Structure):   # blast_seg.h
        _fields_ = [("window", C.c_int), ("locut", C.c_double), ("hicut", C.c_double), ("period", C.c_int), ("hilenmin", C.c_int),
                    ("overlaps", C.c_ubyte), ("maxtrim", C.c_int), ("maxbogus", C.c_int)]
    SegParameters.from_address(sp).overlaps = 1                      # Config.cpp:24-27
    tab = (C.c_ubyte * 128).in_dll(R, "AMINOACID_TO_NCBISTDAA")

    def ref_seg(s):
        conv = bytes(tab[ord(c)] for c in s); locs = C.POINTER(BlastSeqLoc)()
        R.SeqBufferSeg(conv, len(s), 0, sp, C.byref(locs)); out = []
        p = locs
        while p:
            out.append([p.contents.ssr.contents.left, p.contents.ssr.contents.right]); p = p.contents.next
        return out
    seqs = []
    for i in range(300):
        ln = rnd.choice([11, 12, 13, 20, 33, 49, 50, 50, 66, 100, 127])
        kind = i % 6
        if kind == 0:
            s = "".join(rnd.choice(aa) for _ in range(ln))
        elif kind == 1:
            s = "".join(rnd.choice(aa[:rnd.randint(1, 4)]) for _ in range(ln))
        elif kind == 2:
            a = rnd.randrange(0, max(1, ln - 15)); s = "".join(rnd.choice(aa) for _ in range(a)) + rnd.choice(aa) * 15 + "".join(rnd.choice(aa) for _ in range(ln))
            s = s[:ln]
        elif kind == 3:
            u = "".join(rnd.choice(aa) for _ in range(rnd.randint(1, 3))); s = ("".join(rnd.choice(aa) for _ in range(ln // 3)) + u * ln)[:ln]
        elif kind == 4:
            s = ("".join(rnd.choice(aa[:3]) for _ in range(ln // 2)) + "".join(rnd.choice(aa) for _ in range(ln // 4)) + "".join(rnd.choice(aa[5:7]) for _ in range(ln)))[:ln]
        else:
            s = "".join(rnd.choice(aa[:6]) for _ in range(ln))
        seqs.append(s)
    json.dump({"seqs": seqs, "regions": [ref_seg(s) for s in seqs], "lnfact": [float(x) for x in (C.c_double * 200).in_dll(R, "lnfact")]},
              open(os.path.join(HERE, "seg_kat.json"), "w"))
    print("golden fixtures written to", HERE)


if __name__ == "__main__":
    main()
