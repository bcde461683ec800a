"""Pins the oracle against the UNMODIFIED reference: its answers on seeded workloads over the committed golden index and the
reference-built bwtlen = 2^17 index (quirk_db.fmi) are stored in tests/golden/ref_answers.npz.xz (tests/golden/make_golden_ref.py).
CPU only."""
import hashlib, os, tempfile
import numpy as np
import pytest
import golden_workloads as gw
from helpers import Oracle, make_params, read_fastq_packed, make_quirk_db, pack_reads


@pytest.fixture(scope="module")
def answers():
    return gw.ref_answers()


@pytest.fixture(scope="module")
def work(built):
    d = tempfile.mkdtemp(prefix="kjref_")
    gw.write_short_reads(d)
    return d


def _assert_equal(ref_tax, ref_best, tax, best, label):
    bad = np.nonzero((ref_tax != tax) | (ref_best != best))[0]
    assert len(bad) == 0, [(label, int(i), int(ref_tax[i]), int(tax[i]), int(ref_best[i]), int(best[i])) for i in bad[:5]]


@pytest.mark.parametrize("kw", gw.CLI_CONFIGS)
def test_oracle_equals_reference_cli(work, golden, answers, kw):
    d = work; i = gw.CLI_CONFIGS.index(kw)
    orc = Oracle(golden.fmi, golden.nodes)
    for tag, fq1, fq2 in (("pe", d + "/r1.fq", d + "/r2.fq"), ("se", d + "/s.fq", None)):
        n1, s1, o1 = read_fastq_packed(fq1)
        s2 = o2 = None
        if fq2:
            _, s2, o2 = read_fastq_packed(fq2)
        tax, best = orc.classify_batch(make_params(**kw), s1, o1, s2, o2)
        _assert_equal(answers["cli%d_%s_tax" % (i, tag)], answers["cli%d_%s_best" % (i, tag)], tax, best, tag)


@pytest.fixture(scope="module")
def work_long(built):
    """Long DNA reads (400 bp - 12 kb, incl. >127-residue low-complexity runs) and protein reads for -p."""
    d = tempfile.mkdtemp(prefix="kjrefl_")
    return gw.write_long_and_protein_reads(d)


@pytest.mark.parametrize("kw", gw.LONG_CONFIGS)
def test_oracle_equals_reference_long_reads(work_long, golden, answers, kw):
    (ls, lo), _ = work_long; i = gw.LONG_CONFIGS.index(kw)
    tax, best = Oracle(golden.fmi, golden.nodes).classify_batch(make_params(**kw), ls, lo)
    _assert_equal(answers["long%d_tax" % i], answers["long%d_best" % i], tax, best, "long")
    assert (tax > 0).sum() > 100


@pytest.mark.parametrize("kw", gw.PROTEIN_CONFIGS)
def test_oracle_equals_reference_protein_input(work_long, golden, answers, kw):
    _, (ps, po) = work_long; i = gw.PROTEIN_CONFIGS.index(kw)
    tax, best = Oracle(golden.fmi, golden.nodes).classify_batch(make_params(protein=True, **kw), ps, po)
    _assert_equal(answers["prot%d_tax" % i], answers["prot%d_best" % i], tax, best, "protein")
    assert (tax > 0).sum() > 300


def test_lnfact_table_matches_reference(built, answers):
    """ko_lnfact reproduces every entry of the reference's lnfact[0..10000] (blast_seg.c:53-1306): the SHA-256 of the table, taken from
    oracle/_ref/libkaijuref.so, is stored in the golden answers."""
    from helpers import oracle_lib
    L = oracle_lib()
    tab = np.array([L.ko_lnfact(n) for n in range(10001)], dtype=np.float64)
    assert hashlib.sha256(tab.tobytes()).hexdigest() == str(answers["lnfact_sha256"])


def test_bwtlen_multiple_of_65536(built, answers):
    """SURVEY.md 8a exactness note (a): with bwtlen = m * 2^16 (m >= 2) the reference's FMindex resolves the last 129 positions to the
    index1 row that holds C[] instead of counts and returns values that are too small by a per-letter constant; matches that pass
    through those rows (e.g. every match ending in the last letter of the alphabet) behave differently from a "clean" FM index.
    The oracle reproduces that: function level (FMindex, get_suffix of the reference's own C code) and end to end (CLI), on the
    reference-built tests/golden/quirk_db.fmi against the reference's stored answers."""
    import ctypes as C
    from helpers import oracle_lib
    d = tempfile.mkdtemp(prefix="kjq_")
    fmi, nodes, reads = make_quirk_db(d)
    orc = Oracle(fmi, nodes); L = oracle_lib()
    n = L.ko_index_bwtlen(orc.idx); alen = L.ko_index_alen(orc.idx)
    assert n == 131072
    ks, rows = gw.quirk_probe_rows(n, L.ko_index_nseq(orc.idx))
    ref_fm, ref_sfx = answers["quirk_fmindex"], answers["quirk_suffix"]
    assert ref_fm.shape == (len(ks), alen) and len(ref_sfx) == len(rows)
    for k, want in zip(ks, ref_fm):
        for c in range(alen):
            assert L.ko_fmindex(orc.idx, c, k) == int(want[c]), (k, c)
    oseq = C.c_int(); opos = C.c_int64()
    for k, (es, ep) in zip(rows, ref_sfx):
        L.ko_get_suffix(orc.idx, k, C.byref(oseq), C.byref(opos))
        assert (oseq.value, opos.value) == (int(es), int(ep)), k
    seq, off = pack_reads(reads)
    for i, kw in enumerate(gw.QUIRK_CONFIGS):
        tax, best = orc.classify_batch(make_params(**kw), seq, off)
        _assert_equal(answers["quirk%d_tax" % i], answers["quirk%d_best" % i], tax, best, kw)


def test_reference_reader_rules_for_blank_lines(work, golden, answers):
    """What the device-side parser reproduces (kj_ingest.h, tests/test_gpu_parity.py::test_fastq_with_blank_lines), pinned on the reference itself:
    empty lines before the first record and between FASTQ records are skipped (kaiju.cpp:288-289, 341-348), an empty sequence line inside a
    record is the record's sequence, a missing final newline is fine.  The reference's output for the files with blank lines (stored) is the
    oracle's result for the records without them."""
    gw.write_dirty_fastq(work)
    orc = Oracle(golden.fmi, golden.nodes)
    for key, files, kw in (("blank_pe", ("c1.fq", "c2.fq"), dict(mode="greedy")), ("blank_se", ("c1.fq", None), dict(mode="mem"))):
        names, s1, o1 = read_fastq_packed(os.path.join(work, files[0]))
        s2 = o2 = None
        if files[1]:
            _, s2, o2 = read_fastq_packed(os.path.join(work, files[1]))
        P = make_params(**kw)
        tax, best = orc.classify_batch(P, s1, o1, s2, o2)
        ref = gw.stored_run(answers, key)
        assert len(names) == 400 and sorted(names) == sorted(ref)
        assert {nm: (ref[nm][1], ref[nm][2]) for nm in names} == {nm: (int(t), int(b)) for nm, t, b in zip(names, tax, best)}, key
        assert all(ref[nm][0] == ("C" if t else "U") for nm, t in zip(names, tax))
        for i, nm in enumerate(names):                                   # the id sets (column 5 of -v) of the classified records
            if tax[i]:
                a = bytes(s1[int(o1[i]):int(o1[i + 1])]); b = bytes(s2[int(o2[i]):int(o2[i + 1])]) if s2 is not None else None
                assert tuple(sorted(orc.classify_one(P, a, b)[2])) == ref[nm][3], (key, nm)
    assert sum(1 for v in gw.stored_run(answers, "blank_pe").values() if v[0] == "C") > 100
