"""Seeded workloads whose reference answers are committed under tests/golden/ (tests/golden/make_golden_ref.py writes them).  The tests
and the generator build their inputs here, so both see the same reads, files and taxonomies."""
import ctypes as C
import gzip, hashlib, io, json, lzma, os, random
import numpy as np
from helpers import SynthDB, GOLDEN_DIR

GOLDEN_DB = (800, 3)         # SynthDB(nprot, seed) of the committed golden index (tests/golden/make_golden.py)


def golden_db():
    return SynthDB(*GOLDEN_DB)


def ref_answers():
    with open(os.path.join(GOLDEN_DIR, "ref_answers.npz.xz"), "rb") as f:
        return np.load(io.BytesIO(lzma.decompress(f.read())))


def k2t_reports():
    with gzip.open(os.path.join(GOLDEN_DIR, "kaiju2table_reports.json.gz"), "rt") as f:
        return json.load(f)


# ---- tests/test_oracle_vs_ref.py
CLI_CONFIGS = [dict(mode="mem"), dict(mode="mem", seg=False), dict(mode="greedy"), dict(mode="greedy", e=5, s=50), dict(mode="greedy", e=1, E=1e-6)]
LONG_CONFIGS = [dict(mode="mem"), dict(mode="mem", m=8, seg=False), dict(mode="greedy"), dict(mode="greedy", e=5, s=50), dict(mode="greedy", e=2, E=1e-9)]
PROTEIN_CONFIGS = [dict(mode="mem"), dict(mode="mem", m=6, seg=False), dict(mode="greedy"), dict(mode="greedy", e=4, s=40)]


def write_short_reads(d):
    """r1.fq/r2.fq: 3,000 PE150 pairs; s.fq: 3,000 SE100 reads."""
    db = golden_db()
    db.write_fastq(21, 0, 3000, 150, True, d + "/r1.fq", d + "/r2.fq")
    db.write_fastq(22, 0, 3000, 100, False, d + "/s.fq")


def _write_fasta(path, seq, off):
    with open(path, "w") as f:
        for i in range(len(off) - 1):
            f.write(">r%d\n%s\n" % (i, seq[int(off[i]):int(off[i + 1])].tobytes().decode()))


def write_long_and_protein_reads(d):
    """long.fa: 300 DNA reads of 400 bp - 12 kb (incl. >127-residue low-complexity runs); prot.fa: 1,500 protein reads for -p."""
    db = golden_db()
    ls, lo = db.long_reads(31, 0, 300, 400, 12000)
    ps, po = db.protein_reads(32, 0, 1500, 5, 1500)
    _write_fasta(d + "/long.fa", ls, lo); _write_fasta(d + "/prot.fa", ps, po)
    return (ls, lo), (ps, po)


# ---- FASTQ files with blank lines: the reference's reader rules (kaiju.cpp:288-289, 341-348)
def write_dirty_fastq(d):
    """From the first 400 pairs of r1.fq/r2.fq (write_short_reads): c1/c2.fq with every 37th record's sequence emptied, b1/b2.fq the same
    records with blank lines before the first record and between records and no final newline."""
    lines = open(d + "/r1.fq").read().split("\n")[:4 * 400]; lines2 = open(d + "/r2.fq").read().split("\n")[:4 * 400]
    def dirty(ls):
        out = ["", ""]                                                   # leading blank lines: the file type comes from the first non-empty line
        for r in range(0, len(ls), 4):
            rec = ls[r:r + 4]
            if (r // 4) % 37 == 5:
                rec = [rec[0], "", "+", ""]                               # empty sequence line: a line of the record
            out += rec
            if (r // 4) % 5 == 1:
                out += [""] * (1 + (r // 4) % 3)                          # blank lines between records
        return "\n".join(out)                                            # no newline at the end
    def clean(ls):
        out = []
        for r in range(0, len(ls), 4):
            rec = ls[r:r + 4]
            if (r // 4) % 37 == 5:
                rec = [rec[0], "", "+", ""]
            out += rec
        return "\n".join(out) + "\n"
    for name, fn, src in (("c1", clean, lines), ("c2", clean, lines2), ("b1", dirty, lines), ("b2", dirty, lines2)):
        open(d + "/" + name + ".fq", "w").write(fn(src))


def write_gpu_blank_line_fastq(d):
    """The files of test_gpu_parity.py::test_fastq_with_blank_lines: 500 PE150 pairs, clean (c1/c2.fq) and with blank lines (b1/b2.fq)."""
    rnd = random.Random(11); db = golden_db()
    s1, o1, s2, o2 = db.reads(93, 0, 500, 150, True)
    r1 = [s1[int(o1[i]):int(o1[i + 1])].tobytes().decode() for i in range(500)]; r2 = [s2[int(o2[i]):int(o2[i + 1])].tobytes().decode() for i in range(500)]
    def write(path, reads, blanks, mate):
        with open(path, "w") as f:
            if blanks:
                f.write("\n\n")                                              # the file type comes from the first non-empty line
            for i, sq in enumerate(reads):
                if blanks and i and rnd.random() < 0.2:
                    f.write("\n" * rnd.choice([1, 1, 2, 5]))
                if blanks and i % 97 == 5:
                    f.write("@r%d/%d\n\n+\n\n" % (i, mate))                  # an empty sequence line is a line of the record, not a skipped one
                    continue
                f.write("@r%d/%d\n%s\n+\n%s\n" % (i, mate, sq, "I" * len(sq)))
            if blanks:
                f.write("\n\n\n")
    r1c = [("" if i % 97 == 5 else x) for i, x in enumerate(r1)]; r2c = [("" if i % 97 == 5 else x) for i, x in enumerate(r2)]
    files = tuple(os.path.join(d, x) for x in ("c1.fq", "c2.fq", "b1.fq", "b2.fq"))
    write(files[0], r1c, False, 1); write(files[1], r2c, False, 2); write(files[2], r1, True, 1); write(files[3], r2, True, 2)
    return files


def blank_line_runs(d):
    """(key in ref_answers.npz.xz, (mate 1, mate 2), kaiju options) of the reference runs on files with blank lines."""
    write_dirty_fastq(d)
    yield "blank_pe", (d + "/b1.fq", d + "/b2.fq"), dict(mode="greedy")
    yield "blank_se", (d + "/b1.fq", None), dict(mode="mem")
    g = os.path.join(d, "gpu"); os.makedirs(g, exist_ok=True)
    c1, c2, b1, b2 = write_gpu_blank_line_fastq(g)
    yield "gpu_blank_pe", (b1, b2), dict(mode="greedy", e=3)
    yield "gpu_blank_se", (b1, None), dict(mode="greedy", e=3)


def stored_run(ans, key):
    """{name: (C/U, taxon, best, ids)} of a stored reference run, as helpers.parse_kaiju_output returns it."""
    return {str(n): (str(s), int(t), int(b), tuple(sorted(int(x) for x in str(i).split(",") if x)))
            for n, s, t, b, i in zip(ans[key + "_names"], ans[key + "_status"], ans[key + "_tax"], ans[key + "_best"], ans[key + "_ids"])}


# ---- kaiju2table (tests/test_table.py, test_gpu_parity.py::test_counts_table_equals_reference_kaiju2table)
TABLE_OPTS = [dict(rank="species"), dict(rank="genus", expand_viruses=True), dict(rank="family", filter_unclassified=True), dict(rank="phylum", min_percent=2.5),
              dict(rank="species", min_read_count=40), dict(rank="genus", full_path=True), dict(rank="species", rank_list="superkingdom,phylum,genus,species", expand_viruses=True),
              dict(rank="class", filter_unclassified=True, min_percent=0.5, expand_viruses=True)]
COUNTS_TABLE_OPTS = [(dict(rank="species"), ["-r", "species"]), (dict(rank="genus", filter_unclassified=True, full_path=True), ["-r", "genus", "-u", "-p"]),
                     (dict(rank="phylum", min_read_count=5), ["-r", "phylum", "-c", "5"])]


def make_taxonomy(d, rnd):
    """root 1 -> superkingdoms 2 (Bacteria), 10239 (Viruses) -> phylum -> class -> order -> family -> genus -> species, plus 'no rank' nodes."""
    ranks = ["superkingdom", "phylum", "class", "order", "family", "genus", "species"]
    nodes = {1: (1, "no rank")}; names = {1: "root"}; nxt = [20000]; leaves = []
    def grow(parent, depth, tag):
        if depth == len(ranks):
            leaves.append(parent); return
        for k in range(rnd.choice([1, 2, 2, 3])):
            nid = nxt[0]; nxt[0] += rnd.choice([1, 3, 7]); nodes[nid] = (parent, ranks[depth]); names[nid] = "%s %s%d" % (tag, ranks[depth][:3], nid)
            if depth == 3 and k == 0:                      # an unranked node in the lineage
                mid = nxt[0]; nxt[0] += 1; nodes[mid] = (nid, "no rank"); names[mid] = "%s clade%d" % (tag, mid); grow(mid, depth + 1, tag)
            else:
                grow(nid, depth + 1, tag)
    nodes[2] = (1, "superkingdom"); names[2] = "Bacteria"; nodes[10239] = (1, "superkingdom"); names[10239] = "Viruses"
    grow(2, 1, "Bac"); grow(10239, 1, "Vir")
    with open(d + "/nodes.dmp", "w") as f:
        for nid, (par, rk) in nodes.items():
            f.write("%d\t|\t%d\t|\t%s\t|\t\t|\n" % (nid, par, rk))
    with open(d + "/names.dmp", "w") as f:
        for nid, nm in names.items():
            if nid % 11 == 5:
                continue                                   # some taxa have no name -> "taxonid:<id>"
            f.write("%d\t|\t%s synonym\t|\t\t|\tsynonym\t|\n" % (nid, nm))
            f.write("%d\t|\t%s\t|\t\t|\tscientific name\t|\n" % (nid, nm))
    return nodes, leaves


def table_input(d, o):
    """nodes.dmp, names.dmp and a kaiju output file in.tsv: classified reads on leaves, inner nodes and a taxon that is missing from
    nodes.dmp; unclassified reads.  Returns (per-read taxa, the random generator in its state after the file)."""
    rnd = random.Random(11)
    nodes, leaves = make_taxonomy(d, rnd)
    pool = leaves + rnd.sample(sorted(nodes), 12) + [999999]
    weights = [rnd.choice([1, 1, 2, 5, 20, 80]) for _ in pool]
    reads = rnd.choices(pool, weights, k=6000) + [0] * 1500
    rnd.shuffle(reads)
    with open(d + "/in.tsv", "w") as f:
        for i, t in enumerate(reads):
            f.write("C\tr%d\t%d\n" % (i, t) if t else "U\tr%d\t0\n" % i)
    return reads, rnd


def table_flags(o):
    flags = ["-r", o["rank"]]
    flags += ["-e"] if o.get("expand_viruses") else []
    flags += ["-u"] if o.get("filter_unclassified") else []
    flags += ["-p"] if o.get("full_path") else []
    flags += ["-m", str(o["min_percent"])] if "min_percent" in o else []
    flags += ["-c", str(o["min_read_count"])] if "min_read_count" in o else []
    flags += ["-l", o["rank_list"]] if "rank_list" in o else []
    return flags


def ranked_golden_taxonomy(nodes_path, d):
    """The golden taxonomy has no ranks: d/nodes.dmp gives every node a rank by depth, d/names.dmp a name."""
    par = {}
    for l in open(nodes_path):
        p = l.split("\t|\t"); par[int(p[0])] = int(p[1])
    ranks = ["no rank", "superkingdom", "phylum", "class", "order", "family", "genus", "species"]
    def depth(x):
        k = 0
        while par[x] != x:
            x = par[x]; k += 1
        return k
    with open(d + "/nodes.dmp", "w") as f, open(d + "/names.dmp", "w") as g:
        for x in par:
            f.write("%d\t|\t%d\t|\t%s\t|\n" % (x, par[x], ranks[min(depth(x), 7)])); g.write("%d\t|\ttaxon %d\t|\t\t|\tscientific name\t|\n" % (x, x))


# ---- the bwtlen = 2^17 index of helpers.make_quirk_db (tests/golden/quirk_db.fmi)
QUIRK_CONFIGS = [dict(mode="mem"), dict(mode="greedy"), dict(mode="greedy", e=5, s=40), dict(mode="mem", m=5, seg=False)]


class RefBWT(C.Structure):   # the reference's bwt/bwt.h:13-23
    _fields_ = [("len", C.c_long), ("nseq", C.c_int), ("bwt", C.c_void_p), ("alen", C.c_int), ("alphabet", C.c_char_p), ("f", C.c_void_p), ("s", C.c_void_p)]


class RefFMI(C.Structure):   # the reference's bwt/compactfmi.h:10-19
    _fields_ = [("alen", C.c_int), ("bwtlen", C.c_long), ("bwt", C.c_void_p), ("N1", C.c_int), ("N2", C.c_int), ("index1", C.c_void_p), ("index2", C.c_void_p), ("startLcode", C.c_void_p)]


def quirk_probe_rows(n, nseq):
    """(positions k of the FMindex probes, rows of the get_suffix probes) on an index of n rows and nseq sequences."""
    ks = list(range(n - 400, n + 1)) + list(range(65536 - 200, 65536 + 200)) + list(range(0, n, 997))
    rows = list(range(n - 300, n)) + list(range(nseq, n, 511))          # rows below nseq are terminator suffixes: never inside a match interval
    return ks, rows


# ---- the golden DB with every protein K times (test_gpu_build.py::test_scaled_index_equals_reference_built_kfold_index)
KFOLD_COPIES = (2, 3, 7)
KFOLD_READS = (5, 0, 20000, 150)     # seed, first, pairs, read length


def kfold_reads():
    return golden_db().reads(*KFOLD_READS, True)


def kfold_fasta(src, dst, k):
    recs = []; cur = None
    for l in open(src).read().split("\n"):
        if l.startswith(">"):
            cur = [l, []]; recs.append(cur)
        elif cur is not None and l:
            cur[1].append(l)
    with open(dst, "w") as g:
        for h, s in recs:
            for _ in range(k):
                g.write(h + "\n" + "\n".join(s) + "\n")


def result_digest(tax, best):
    return hashlib.sha256(np.ascontiguousarray(tax, dtype=np.uint64).tobytes() + np.ascontiguousarray(best, dtype=np.uint32).tobytes()).hexdigest()
