#!/usr/bin/env python
"""Generates the committed answers of the UNMODIFIED reference that the comparison tests check against, on the committed golden
index (db.fmi, nodes.dmp) and reads drawn from its seeded DB (tools/kjgen.c).  Needs oracle/_ref (oracle/Makefile) once:

    make -C oracle ref && python tests/golden/make_golden_ref.py

Outputs (small, committed):
    ref_answers.npz.xz         taxon + best per read of `kaiju` for tests/test_oracle_vs_ref.py (short, long and protein reads),
                               the reference's records of the blank-line FASTQ files of test_gpu_parity.py::test_fastq_with_blank_lines
                               the SHA-256 of the reference's lnfact[0..10000] table, the reference's FMindex / get_suffix values
                               and CLI results on quirk_db.fmi, and for the golden DB repeated K = 2, 3, 7 times the checksums of
                               the index kaiju-mkbwt/-mkfmi build and a SHA-256 of the reference's results on it
    quirk_db.fmi               index of helpers.make_quirk_db (bwtlen = 2 * 2^16), built by kaiju-mkbwt/-mkfmi
    kaiju2table_reports.json.gz  `kaiju2table` reports for tests/test_table.py and test_gpu_parity.py::test_counts_table_...
                               (the input file name in the reports is written as {LABEL})
"""
import ctypes as C
import gzip, hashlib, io, json, lzma, os, shutil, subprocess, sys, tempfile, zipfile
import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
TESTS = os.path.dirname(HERE)
sys.path.insert(0, TESTS); sys.path.insert(0, os.path.dirname(TESTS))
from helpers import REF_DIR, Oracle, build_fmi, make_params, make_quirk_db, run_ref_kaiju, read_fastq_packed   # noqa: E402
import golden_workloads as gw                                     # noqa: E402


def ref_arrays(res, names):
    return (np.array([res[n][1] for n in names], dtype=np.uint64), np.array([res[n][2] for n in names], dtype=np.uint32))


def narrow(key, a):
    """taxon ids and best scores in the narrowest unsigned type that holds them (the tests compare values, not types)."""
    if key.endswith("_tax") and a.max(initial=0) < 2 ** 32:
        return a.astype(np.uint32)
    if key.endswith("_best") and a.max(initial=0) < 2 ** 16:
        return a.astype(np.uint16)
    return a


def quirk_answers(d, out):
    """The reference on the bwtlen = 2^17 index: FMindex(c, k) and get_suffix(k) of its own C code at the rows
    test_oracle_vs_ref.py::test_bwtlen_multiple_of_65536 probes, and its CLI results for gw.QUIRK_CONFIGS."""
    q = os.path.join(d, "quirk"); os.makedirs(q)
    fmi, nodes, reads = make_quirk_db(q, build=True)
    shutil.copyfile(fmi, os.path.join(HERE, "quirk_db.fmi"))
    R = C.CDLL(os.path.join(REF_DIR, "libkaijuref.so")); libc = C.CDLL(None)
    libc.fopen.restype = C.c_void_p; libc.fopen.argtypes = [C.c_char_p, C.c_char_p]
    R.readIndexes.restype = C.c_void_p; R.readIndexes.argtypes = [C.c_void_p]
    R.FMindex.restype = C.c_long; R.FMindex.argtypes = [C.c_void_p, C.c_ubyte, C.c_long]
    R.get_suffix.argtypes = [C.c_void_p, C.c_void_p, C.c_long, C.POINTER(C.c_int), C.POINTER(C.c_long)]
    b = gw.RefBWT.from_address(R.readIndexes(libc.fopen(fmi.encode(), b"r"))); fm = gw.RefFMI.from_address(b.f)
    ks, rows = gw.quirk_probe_rows(fm.bwtlen, b.nseq)
    out["quirk_fmindex"] = np.array([[R.FMindex(b.f, c, k) for c in range(fm.alen)] for k in ks], dtype=np.int64)
    iseq = C.c_int(); pos = C.c_long(); sfx = []
    for k in rows:
        R.get_suffix(b.f, b.s, k, C.byref(iseq), C.byref(pos)); sfx.append((iseq.value, pos.value))
    out["quirk_suffix"] = np.array(sfx, dtype=np.int64)
    with open(q + "/r.fa", "w") as f:
        for i, r in enumerate(reads):
            f.write(">r%d\n%s\n" % (i, r))
    for i, kw in enumerate(gw.QUIRK_CONFIGS):
        res = run_ref_kaiju(nodes, fmi, q + "/r.fa", None, threads=4, **kw)
        out["quirk%d_tax" % i], out["quirk%d_best" % i] = ref_arrays(res, ["r%d" % k for k in range(len(reads))])


def kfold_answers(d, out):
    """The golden DB with every protein K times, indexed by kaiju-mkbwt/-mkfmi: the checksums the host transcoder reports for that
    index and the SHA-256 of the reference's taxon + best on gw.kfold_reads() (MEM and Greedy)."""
    sys.path.insert(0, HERE)
    import kaiju_b200 as kb
    from make_golden import write_db_faa
    k = os.path.join(d, "kfold"); os.makedirs(k)
    write_db_faa(k + "/base.faa", k + "/nodes.dmp"); nodes = k + "/nodes.dmp"
    s1, o1, s2, o2 = gw.kfold_reads()
    gw.golden_db().write_fastq(*gw.KFOLD_READS, True, k + "/r1.fq", k + "/r2.fq")
    names = read_fastq_packed(k + "/r1.fq")[0]
    for copies in gw.KFOLD_COPIES:
        gw.kfold_fasta(k + "/base.faa", k + "/rep.faa", copies)
        rep = build_fmi(k + "/rep.faa", k + "/rep%d" % copies, threads=4)
        out["kfold%d_checksums" % copies] = kb.host_index_checksums(rep, nodes)
        orc = Oracle(rep, nodes)
        for mode in ("mem", "greedy"):
            tax, best = ref_arrays(run_ref_kaiju(nodes, rep, k + "/r1.fq", k + "/r2.fq", mode=mode, threads=8), names)
            otax, obest = orc.classify_batch(make_params(mode), s1, o1, s2, o2)
            assert np.array_equal(tax, otax) and np.array_equal(best, obest), (copies, mode)
            out["kfold%d_%s_sha256" % (copies, mode)] = np.array(gw.result_digest(tax, best))


def main():
    fmi, nodes = os.path.join(HERE, "db.fmi"), os.path.join(HERE, "nodes.dmp")
    d = tempfile.mkdtemp(prefix="kjgold_")
    out = {}
    # test_oracle_vs_ref.py: short reads (paired 150 bp, single 100 bp), long DNA reads, protein reads
    gw.write_short_reads(d)
    for i, kw in enumerate(gw.CLI_CONFIGS):
        for tag, fq1, fq2 in (("pe", d + "/r1.fq", d + "/r2.fq"), ("se", d + "/s.fq", None)):
            res = run_ref_kaiju(nodes, fmi, fq1, fq2, threads=4, **kw)
            out["cli%d_%s_tax" % (i, tag)], out["cli%d_%s_best" % (i, tag)] = ref_arrays(res, read_fastq_packed(fq1)[0])
    (ls, lo), (ps, po) = gw.write_long_and_protein_reads(d)
    for i, kw in enumerate(gw.LONG_CONFIGS):
        res = run_ref_kaiju(nodes, fmi, d + "/long.fa", None, threads=8, **kw)
        out["long%d_tax" % i], out["long%d_best" % i] = ref_arrays(res, ["r%d" % k for k in range(len(lo) - 1)])
    for i, kw in enumerate(gw.PROTEIN_CONFIGS):
        res = run_ref_kaiju(nodes, fmi, d + "/prot.fa", None, threads=8, protein=True, **kw)
        out["prot%d_tax" % i], out["prot%d_best" % i] = ref_arrays(res, ["r%d" % k for k in range(len(po) - 1)])
    # the reference's reader on FASTQ files with blank lines (test_oracle_vs_ref.py and test_gpu_parity.py)
    for key, files, kw in gw.blank_line_runs(d):
        res = run_ref_kaiju(nodes, fmi, files[0], files[1], threads=1, **kw)
        names = sorted(res)
        out[key + "_names"] = np.array(names); out[key + "_status"] = np.array([res[n][0] for n in names])
        out[key + "_tax"] = np.array([res[n][1] for n in names], dtype=np.uint64); out[key + "_best"] = np.array([res[n][2] for n in names], dtype=np.uint32)
        out[key + "_ids"] = np.array([",".join(map(str, res[n][3])) for n in names])
    tab = (C.c_double * 10001).in_dll(C.CDLL(os.path.join(REF_DIR, "libkaijuref.so")), "lnfact")
    out["lnfact_sha256"] = np.array(hashlib.sha256(np.array(tab[:], dtype=np.float64).tobytes()).hexdigest())
    quirk_answers(d, out)
    kfold_answers(d, out)
    npz = io.BytesIO()      # an uncompressed .npz with fixed member times, xz-compressed as a whole (the arrays repeat one another)
    with zipfile.ZipFile(npz, "w", zipfile.ZIP_STORED) as z:
        for key in sorted(out):
            buf = io.BytesIO(); np.save(buf, narrow(key, np.asarray(out[key]))); z.writestr(zipfile.ZipInfo(key + ".npy"), buf.getvalue())
    with open(os.path.join(HERE, "ref_answers.npz.xz"), "wb") as f:
        f.write(lzma.compress(npz.getvalue(), preset=9 | lzma.PRESET_EXTREME))

    # kaiju2table reports
    k2t = os.path.join(REF_DIR, "kaiju2table"); reports = {}
    def run_k2t(dd, inputs, flags):
        subprocess.run([k2t, "-t", dd + "/nodes.dmp", "-n", dd + "/names.dmp", "-o", dd + "/ref.tsv"] + flags + inputs, check=True, stderr=subprocess.DEVNULL)
        return open(dd + "/ref.tsv").read()
    for i, o in enumerate(gw.TABLE_OPTS):
        dd = tempfile.mkdtemp(prefix="kjk2t_", dir=d); gw.table_input(dd, o)
        flags = gw.table_flags(o); inp = dd + "/in.tsv"
        reports["table%d" % i] = run_k2t(dd, [inp], flags).replace(inp, "{LABEL}")
        reports["table%d_twice" % i] = run_k2t(dd, [inp, inp], flags).replace(inp, "{LABEL}")
    dd = tempfile.mkdtemp(prefix="kjk2t_", dir=d); gw.ranked_golden_taxonomy(nodes, dd)
    inp = dd + "/reads.tsv"
    with gzip.open(os.path.join(HERE, "expected_mem_default_pe150.tsv.gz"), "rt") as f, open(inp, "w") as g:
        for line in f:
            p = line.split("\t"); g.write("%s\t%s\t%s\n" % (p[0], p[1], p[2]))
    for i, (o, flags) in enumerate(gw.COUNTS_TABLE_OPTS):
        reports["counts%d" % i] = run_k2t(dd, [inp], flags).replace(inp, "{LABEL}")
    with open(os.path.join(HERE, "kaiju2table_reports.json.gz"), "wb") as raw, gzip.GzipFile(fileobj=raw, mode="wb", mtime=0) as f:
        f.write(json.dumps(reports, sort_keys=True).encode())          # mtime=0: the same reports give the same bytes
    print("reference answers written to", HERE)


if __name__ == "__main__":
    main()
