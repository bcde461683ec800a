"""GPU parity: the CUDA path called through the C ABI (libkaijub200.so) vs the committed reference outputs, the oracle on
fresh seeded workloads, edge cases, and size-independent properties at large batch sizes.  Bit-exact (integer work)."""
import ctypes as C
import os
import numpy as np
import pytest
from conftest import GOLDEN_CONFIGS
import golden_workloads as gw
from helpers import Oracle, make_params, SynthDB

pytestmark = pytest.mark.gpu


def kb_params(kb, kw):
    return kb.make_params(kw.get("mode", "mem"), m=kw.get("m", 11), e=kw.get("e", 3), s=kw.get("s", 65), seed=kw.get("seed", 7), E=kw.get("E", 0.01), seg=kw.get("seg", True),
                          protein=kw.get("protein", False))


@pytest.fixture(scope="module")
def kb(built):
    import kaiju_b200
    return kaiju_b200


@pytest.fixture(scope="module")
def gclf(kb, golden):
    c = kb.Classifier(golden.fmi, golden.nodes, device=0, params=kb.make_params("mem"))
    yield c
    c.close()


@pytest.mark.parametrize("cfg", sorted(GOLDEN_CONFIGS))
@pytest.mark.parametrize("tag", ["pe150", "se100"])
def test_gpu_matches_reference_golden(kb, gclf, golden, cfg, tag):
    names, s1, o1, s2, o2 = golden.reads(tag)
    gclf.set_params(kb_params(kb, GOLDEN_CONFIGS[cfg]))
    tax, best = gclf.classify(s1, o1, s2, o2)
    etax, ebest, _ = golden.expected(cfg, tag)
    bad = np.nonzero((tax != etax) | (best != ebest))[0]
    assert len(bad) == 0, [(names[i], int(tax[i]), int(etax[i]), int(best[i]), int(ebest[i])) for i in bad[:5]]
    assert gclf.kernel_launches > 0


@pytest.fixture(scope="module")
def fresh(kb, golden):
    """Fresh seeded reads (tools/kjgen.c) from the DB of the committed golden index."""
    return gw.golden_db(), golden.fmi, golden.nodes


@pytest.mark.parametrize("kw", [dict(mode="mem"), dict(mode="mem", seg=False), dict(mode="mem", m=14), dict(mode="greedy"),
                                dict(mode="greedy", e=5), dict(mode="greedy", e=2, s=45, seg=False), dict(mode="greedy", E=1e-8)])
def test_gpu_matches_oracle_on_fresh_workload(kb, fresh, kw):
    db, fmi, nodes = fresh
    orc = Oracle(fmi, nodes)
    clf = kb.Classifier(fmi, nodes, device=0, params=kb_params(kb, kw))
    for paired, rl in ((True, 150), (False, 100), (True, 75)):
        s1, o1, s2, o2 = db.reads(31 + rl, 0, 6000, rl, paired)
        otax, obest = orc.classify_batch(make_params(**kw), s1, o1, s2, o2)
        tax, best = clf.classify(s1, o1, s2, o2)
        bad = np.nonzero((tax != otax) | (best != obest))[0]
        assert len(bad) == 0, (kw, paired, rl, [(int(i), int(tax[i]), int(otax[i]), int(best[i]), int(obest[i])) for i in bad[:5]])
    clf.close()


def test_edge_cases(kb, gclf, golden):
    gclf.set_params(kb.make_params("mem"))
    # empty batch
    t, b = gclf.classify(np.zeros(0, np.uint8), np.zeros(1, np.uint64))
    assert len(t) == 0
    # ragged batch: empty reads, reads shorter than 3m, one long read at the supported maximum
    rng = np.random.default_rng(3)
    reads = [b"", b"ACGT", b"ACGTACGTACGTACGTACGTACGTACGTACGT", bytes(rng.choice(list(b"ACGT"), 381).astype(np.uint8)), b"N" * 200, b"acgtn" * 30,
             bytes(rng.choice(list(b"ACGT"), 16383).astype(np.uint8)), b"GCA" * 5461]
    s = np.frombuffer(b"".join(reads), dtype=np.uint8); o = np.zeros(len(reads) + 1, np.uint64); o[1:] = np.cumsum([len(r) for r in reads])
    t, b = gclf.classify(s, o)
    orc = Oracle(golden.fmi, golden.nodes)
    ot, ob = orc.classify_batch(make_params("mem"), s, o)
    assert np.array_equal(t, ot) and np.array_equal(b, ob)
    # a read beyond KJ_MAX_READ_LEN is refused with an error code, not misclassified
    s2 = np.frombuffer(b"A" * 16384, dtype=np.uint8); o2 = np.array([0, 16384], np.uint64)
    with pytest.raises(kb.KaijuError):
        gclf.classify(s2, o2)
    # protein input takes one file only (kaiju.cpp:201) and at most KJ_MAX_PROTEIN_LEN residues
    gclf.set_params(kb.make_params("mem", protein=True))
    pr = np.frombuffer(b"MKV" * 40, dtype=np.uint8); po = np.array([0, 120], np.uint64)
    with pytest.raises(kb.KaijuError):
        gclf.classify(pr, po, pr, po)
    with pytest.raises(kb.KaijuError):
        gclf.classify(np.frombuffer(b"A" * 5462, dtype=np.uint8), np.array([0, 5462], np.uint64))
    gclf.set_params(kb.make_params("mem"))


def test_properties_at_scale(kb, fresh):
    """1 M pairs: (a) results do not depend on batch order/chunking (the persistent-kernel scheduler), (b) device-buffer
    and host-buffer entry points agree, (c) duplicated reads get identical results, (d) checksum of a subsample == oracle."""
    import torch
    db, fmi, nodes = fresh
    n = 1 << 20
    s1, o1, s2, o2 = db.reads(77, 0, n, 150, True)
    clf = kb.Classifier(fmi, nodes, device=0, params=kb.make_params("mem"))
    tax, best = clf.classify(s1, o1, s2, o2)
    # (a) reversed order
    perm = np.arange(n)[::-1]
    l1 = np.diff(o1).astype(np.int64); l2 = np.diff(o2).astype(np.int64)
    assert (l1[l1 != 150].size + l2[l2 != 150].size) < n // 100
    def gather(s, o, perm):
        ln = np.diff(o).astype(np.int64)[perm]; no = np.zeros(len(perm) + 1, np.uint64); no[1:] = np.cumsum(ln)
        idx = np.repeat(o[:-1].astype(np.int64)[perm] - no[:-1].astype(np.int64), ln) + np.arange(int(no[-1]))
        return s[idx], no
    rs1, ro1 = gather(s1, o1, perm); rs2, ro2 = gather(s2, o2, perm)
    rtax, rbest = clf.classify(rs1, ro1, rs2, ro2)
    assert np.array_equal(rtax[::-1], tax) and np.array_equal(rbest[::-1], best)
    # (b) device-resident entry point
    d = [torch.from_numpy(x.view(np.int64) if x.dtype == np.uint64 else x).cuda() for x in (s1, o1, s2, o2)]
    dt = torch.zeros(n, dtype=torch.int64, device="cuda"); dbst = torch.zeros(n, dtype=torch.int32, device="cuda")
    clf.classify_device(d[0].data_ptr(), d[1].data_ptr(), d[2].data_ptr(), d[3].data_ptr(), n, dt.data_ptr(), dbst.data_ptr())
    torch.cuda.synchronize(); clf.check_errors()
    assert np.array_equal(dt.cpu().numpy().view(np.uint64), tax) and np.array_equal(dbst.cpu().numpy().view(np.uint32), best)
    # (d) oracle on a strided subsample
    orc = Oracle(fmi, nodes); sub = np.arange(0, n, 257)[:3000]
    ss1, so1 = gather(s1, o1, sub); ss2, so2 = gather(s2, o2, sub)
    otax, obest = orc.classify_batch(make_params("mem"), ss1, so1, ss2, so2)
    assert np.array_equal(otax, tax[sub]) and np.array_equal(obest, best[sub])
    assert 0.55 < (tax != 0).mean() < 0.85          # ~70 % of the synthetic reads come from the DB
    clf.close()


def test_wide_index_kernels_and_no_kmer_table(kb, golden, monkeypatch):
    """The 64-bit-interval kernels (indexes >= 2^32 rows) and the table-free chain start, forced on the small golden index."""
    names, s1, o1, s2, o2 = golden.reads("pe150")
    for env in ({"KJ_FORCE_WIDE": "1"}, {"KJ_KMER_K": "0"}, {"KJ_KMER_K": "3"}):
        for k, v in env.items():
            monkeypatch.setenv(k, v)
        for cfg in ("mem_default", "greedy_default"):
            clf = kb.Classifier(golden.fmi, golden.nodes, device=0, params=kb_params(kb, GOLDEN_CONFIGS[cfg]))
            tax, best = clf.classify(s1, o1, s2, o2)
            etax, ebest, _ = golden.expected(cfg, "pe150")
            assert np.array_equal(tax, etax) and np.array_equal(best, ebest), (env, cfg)
            clf.close()
        for k in env:
            monkeypatch.delenv(k)


def test_cli_matches_reference_output_format(kb, golden, tmp_path):
    """kaiju-b200 (kj_cli.cpp) on the golden FASTQ files: same C/U lines as the reference, in input order."""
    import gzip, shutil, subprocess
    from conftest import ROOT
    cli = os.path.join(ROOT, "kaiju_b200", "kaiju-b200")
    assert os.path.exists(cli)
    gold = os.path.join(ROOT, "tests", "golden")
    fq = {}
    for name in ("pe150_1", "pe150_2"):
        fq[name] = str(tmp_path / (name + ".fq"))
        with gzip.open(os.path.join(gold, name + ".fq.gz"), "rb") as a, open(fq[name], "wb") as b:
            shutil.copyfileobj(a, b)
    for mode, cfg, extra in (("mem", "mem_default", []), ("greedy", "greedy_default", []), ("mem", "mem_noseg", ["-X"]), ("greedy", "greedy_e5", ["-e", "5"])):
        out = str(tmp_path / (cfg + ".tsv"))
        # gz input for mate 1 (zlib path), plain for mate 2; -z is accepted and ignored
        subprocess.check_call([cli, "-t", golden.nodes, "-f", golden.fmi, "-i", os.path.join(gold, "pe150_1.fq.gz"), "-j", fq["pe150_2"], "-a", mode, "-z", "4", "-v", "-o", out] + extra)
        etax, ebest, eids = golden.expected(cfg, "pe150"); names = golden.reads("pe150")[0]
        lines = open(out).read().splitlines()
        assert len(lines) == len(names)
        for ln, nm, t, b, ids in zip(lines, names, etax, ebest, eids):
            p = ln.split("\t")
            if t:      # columns 1-5 of the reference's -v output (ids: std::set order, each followed by a comma)
                assert p[:5] == ["C", nm, str(int(t)), str(int(b)), "".join("%d," % x for x in sorted(ids))] and len(p) == 7, (ln, nm, t, b, ids)
            else:
                assert p == ["U", nm, "0"], ln
    # error paths: -p with a second input file (kaiju.cpp:201), missing arguments: usage + non-zero exit
    assert subprocess.call([cli, "-t", golden.nodes, "-f", golden.fmi, "-i", fq["pe150_1"], "-j", fq["pe150_2"], "-p"], stderr=subprocess.DEVNULL) != 0
    assert subprocess.call([cli, "-f", golden.fmi], stderr=subprocess.DEVNULL) != 0


@pytest.mark.parametrize("cfg", ["mem_default", "mem_m5", "greedy_default", "greedy_e5"])
def test_verbose_id_sets_match_reference_column5(kb, gclf, golden, cfg):
    """kj_classify_verbose: the match-id set (column 5 of `kaiju -v`) incl. the 21-id cap case, ids missing from nodes.dmp, taxon 0."""
    names, s1, o1, s2, o2 = golden.reads("pe150")
    gclf.set_params(kb_params(kb, GOLDEN_CONFIGS[cfg]))
    tax, best, ids = gclf.classify_verbose(s1, o1, s2, o2)
    etax, ebest, eids = golden.expected(cfg, "pe150")
    assert np.array_equal(tax, etax) and np.array_equal(best, ebest)
    for i, nm in enumerate(names):
        assert ids[i] == (eids[i] if etax[i] else ()), (nm, ids[i], eids[i])
    assert max(len(x) for x in ids) == 21            # the capped read is in the fixture


LONG_CONFIGS = [dict(mode="mem"), dict(mode="mem", m=7, seg=False), dict(mode="greedy"), dict(mode="greedy", e=5, s=40, E=1e-3), dict(mode="greedy", e=1, s=100, seg=False, E=1e-30)]


@pytest.mark.parametrize("kw", LONG_CONFIGS)
def test_long_reads_match_oracle(kb, fresh, kw):
    """Reads of 0.3-16 kb (work space in global memory, >127-residue low-complexity runs, thousands of queued fragments) and the
    lengths around the shared-memory/global-memory switch, single-end and paired."""
    db, fmi, nodes = fresh
    orc = Oracle(fmi, nodes)
    clf = kb.Classifier(fmi, nodes, device=0, params=kb_params(kb, kw))
    for seed, n, lo, hi in ((41, 1500, 300, 16383), (42, 3000, 200, 700), (43, 3000, 380, 1200)):
        s, o = db.long_reads(seed, 0, n, lo, hi)
        otax, obest = orc.classify_batch(make_params(**kw), s, o)
        tax, best = clf.classify(s, o)
        bad = np.nonzero((tax != otax) | (best != obest))[0]
        assert len(bad) == 0, (kw, seed, [(int(i), int(tax[i]), int(otax[i]), int(best[i]), int(obest[i])) for i in bad[:5]])
        assert (tax != 0).mean() > 0.5
    # paired: a long mate 1 with a short mate 2 (mixed lengths inside one batch)
    s1, o1 = db.long_reads(44, 0, 1000, 150, 2500); s2, o2, _, _ = db.reads(45, 0, 1000, 150, False)
    otax, obest = orc.classify_batch(make_params(**kw), s1, o1, s2, o2)
    tax, best = clf.classify(s1, o1, s2, o2)
    assert np.array_equal(tax, otax) and np.array_equal(best, obest)
    clf.close()


@pytest.mark.parametrize("kw", [dict(mode="mem"), dict(mode="mem", m=6, seg=False), dict(mode="greedy"), dict(mode="greedy", e=4, s=40), dict(mode="greedy", e=8, s=30, m=9, seed=5, E=1e-9)])
def test_protein_input_matches_oracle(kb, fresh, kw):
    """-p: protein reads of 5-5461 residues, split at non-residue letters, lower case, long low-complexity runs."""
    db, fmi, nodes = fresh
    orc = Oracle(fmi, nodes)
    clf = kb.Classifier(fmi, nodes, device=0, params=kb_params(kb, dict(kw, protein=True)))
    for seed, n, lo, hi in ((51, 6000, 5, 400), (52, 2000, 100, 5461)):
        s, o = db.protein_reads(seed, 0, n, lo, hi)
        otax, obest = orc.classify_batch(make_params(protein=True, **kw), s, o)
        tax, best = clf.classify(s, o)
        bad = np.nonzero((tax != otax) | (best != obest))[0]
        assert len(bad) == 0, (kw, seed, [(int(i), int(tax[i]), int(otax[i]), int(best[i]), int(obest[i])) for i in bad[:5]])
        assert (tax != 0).mean() > 0.5
    clf.close()


def test_variant_ring_overflow_is_retried(kb, golden, monkeypatch):
    """Greedy -e 8 with a low score threshold on long reads that match nothing explores thousands of substituted variants per read;
    a full per-read ring is reported by the kernel, enlarged by the library and the call repeated -- the result equals the oracle's."""
    other = SynthDB(3000, 777)                                   # reads from proteins that are not in the golden index
    s, o = other.long_reads(61, 0, 120, 3000, 16383)
    kw = dict(mode="greedy", e=8, s=30, m=9, seed=5, E=1e-9)
    monkeypatch.setenv("KJ_VARIANT_CAP", "128")                  # test hook: start from a ring that is too small (the emulated test shows it overflows)
    clf = kb.Classifier(golden.fmi, golden.nodes, device=0, params=kb_params(kb, kw))
    tax, best = clf.classify(s, o)                               # overflow -> ring x4 -> repeated inside kj_classify
    otax, obest = Oracle(golden.fmi, golden.nodes).classify_batch(make_params(**kw), s, o)
    assert np.array_equal(tax, otax) and np.array_equal(best, obest)
    # the device-buffer entry point reports the overflow through kj_check_errors and succeeds when called again
    import torch
    clf2 = kb.Classifier(golden.fmi, golden.nodes, device=0, params=kb_params(kb, kw))
    ds = torch.from_numpy(s).cuda(); do = torch.from_numpy(o.view(np.int64)).cuda(); dt = torch.zeros(len(o) - 1, dtype=torch.int64, device="cuda")
    clf2.classify_device(ds.data_ptr(), do.data_ptr(), None, None, len(o) - 1, dt.data_ptr()); torch.cuda.synchronize()
    with pytest.raises(kb.KaijuError):
        clf2.check_errors()
    clf2.classify_device(ds.data_ptr(), do.data_ptr(), None, None, len(o) - 1, dt.data_ptr()); torch.cuda.synchronize(); clf2.check_errors()
    assert np.array_equal(dt.cpu().numpy().view(np.uint64), otax)
    clf.close(); clf2.close()


def test_cli_protein_and_verbose_columns(kb, golden, tmp_path):
    """kaiju-b200 -p -v: columns 1-5 equal the oracle's (name, taxon, best, ascending id set)."""
    import subprocess
    from conftest import ROOT
    db = SynthDB(800, 3)
    s, o = db.protein_reads(71, 0, 400, 5, 900)
    fa = tmp_path / "p.fa"
    with open(fa, "w") as f:
        for i in range(len(o) - 1):
            f.write(">q%d some description\n%s\n" % (i, s[int(o[i]):int(o[i + 1])].tobytes().decode()))
    out = subprocess.run([os.path.join(ROOT, "kaiju_b200", "kaiju-b200"), "-t", golden.nodes, "-f", golden.fmi, "-i", str(fa), "-p", "-v", "-a", "greedy", "-e", "2"],
                         capture_output=True, text=True, check=True).stdout.splitlines()
    orc = Oracle(golden.fmi, golden.nodes); P = make_params("greedy", e=2, protein=True)
    assert len(out) == len(o) - 1
    for i, line in enumerate(out):
        t, b, ids = orc.classify_one(P, s[int(o[i]):int(o[i + 1])].tobytes())
        exp = "C\tq%d\t%d\t%d\t%s" % (i, t, b, "".join("%d," % x for x in sorted(ids))) if t else "U\tq%d\t0" % i
        assert "\t".join(line.split("\t")[:5]) == exp, (i, line, exp)       # columns 6-7 (accessions, fragment strings) are pinned by test_gpu_frontends.py
    # kaiju-multi style: comma-separated lists of inputs and outputs against the index loaded once
    oa, ob = tmp_path / "a.tsv", tmp_path / "b.tsv"
    subprocess.run([os.path.join(ROOT, "kaiju_b200", "kaiju-b200"), "-t", golden.nodes, "-f", golden.fmi, "-i", "%s,%s" % (fa, fa), "-o", "%s,%s" % (oa, ob),
                    "-p", "-v", "-a", "greedy", "-e", "2"], check=True, stderr=subprocess.DEVNULL)
    assert open(oa).read().splitlines() == out and open(ob).read().splitlines() == out


def _expected_lines(orc, P, names, seqs1, seqs2=None, verbose=False):
    out = []
    for i, nm in enumerate(names):
        t, b, ids = orc.classify_one(P, seqs1[i], seqs2[i] if seqs2 else None)
        if t:
            out.append("C\t%s\t%d" % (nm, t) + ("\t%d\t%s" % (b, "".join("%d," % x for x in sorted(ids))) if verbose else ""))
        else:
            out.append("U\t%s\t0" % nm)
    return out


@pytest.mark.parametrize("chunk", ["4096", "65536", ""])
def test_file_ingest_on_device(kb, golden, tmp_path, monkeypatch, chunk):
    """kj_classify_files: FASTA (wrapped lines, CRLF, no final newline), FASTQ (gz), mixed file types for the two mates, name trimming
    at ' /\\t\\r', stripping of non-letters -- parsed, classified and formatted on the device, across many chunk boundaries."""
    import gzip, random
    if chunk:
        monkeypatch.setenv("KJ_INGEST_CHUNK", chunk)
    rnd = random.Random(5); db = SynthDB(800, 3)
    s1, o1, s2, o2 = db.reads(91, 0, 700, 150, True)
    ls, lo = db.long_reads(92, 0, 60, 300, 9000)
    r1 = [s1[int(o1[i]):int(o1[i + 1])].tobytes() for i in range(700)]; r2 = [s2[int(o2[i]):int(o2[i + 1])].tobytes() for i in range(700)]
    lr = [ls[int(lo[i]):int(lo[i + 1])].tobytes() for i in range(60)]
    orc = Oracle(golden.fmi, golden.nodes)
    # --- paired: mate 1 as gzipped FASTQ with decorated names, mate 2 as wrapped FASTA with CRLF and dirt inside the sequence lines
    names = ["read%d" % i for i in range(700)]
    deco1 = [" 1:N:0:ACGT", "/1", "\tx", "", " desc/1"]; deco2 = [" 2:N:0:ACGT", "/2", "\ty", "", " other"]
    f1 = tmp_path / "m1.fq.gz"; f2 = tmp_path / "m2.fa"
    with gzip.open(f1, "wt") as f:
        for i, nm in enumerate(names):
            f.write("@%s%s\n%s\n+\n%s\n" % (nm, deco1[i % 5], r1[i].decode(), "I" * len(r1[i])))
    with open(f2, "wb") as f:
        for i, nm in enumerate(names):
            sq = r2[i].decode(); w = rnd.choice([40, 60, 70, 200]); body = "\r\n".join(sq[k:k + w] for k in range(0, len(sq), w))
            if i % 7 == 0:
                body = body[:10] + " 12-*" + body[10:]                        # strip() removes everything that is not a letter
            f.write((">%s%s\r\n%s%s" % (nm, deco2[i % 5], body, "" if i == 699 else "\r\n")).encode())      # no newline at the end of the file
    clf = kb.Classifier(golden.fmi, golden.nodes, device=0, params=kb.make_params("greedy", e=2))
    out = tmp_path / "pe.tsv"
    n, k = clf.classify_files(str(f1), str(f2), str(out), verbose=True)
    exp = _expected_lines(orc, make_params("greedy", e=2), names, r1, r2, verbose=True)
    got = open(out).read().splitlines()
    assert n == 700 and got == exp and k == sum(1 for l in exp if l[0] == "C")
    # --- single-end long reads as FASTA, MEM
    f3 = tmp_path / "long.fa"
    with open(f3, "w") as f:
        for i, sq in enumerate(lr):
            f.write(">L%d some text\n%s\n" % (i, "\n".join(sq.decode()[k:k + 80] for k in range(0, len(sq), 80))))
    clf.set_params(kb.make_params("mem"))
    out3 = tmp_path / "long.tsv"
    n, k = clf.classify_files(str(f3), None, str(out3))
    assert n == 60 and open(out3).read().splitlines() == _expected_lines(orc, make_params("mem"), ["L%d" % i for i in range(60)], lr)
    # --- errors mirror the reference's front end
    bad = tmp_path / "bad.fq"; bad.write_text("ACGT\n")
    with pytest.raises(kb.KaijuError, match="Auto-detection"):
        clf.classify_files(str(bad), None, str(tmp_path / "x.tsv"))
    f4 = tmp_path / "m2_renamed.fa"
    f4.write_bytes(open(f2, "rb").read().replace(b">read350", b">readX350"))
    with pytest.raises(kb.KaijuError, match="not identical"):
        clf.classify_files(str(f1), str(f4), str(tmp_path / "x.tsv"))
    f5 = tmp_path / "m2_short.fa"
    f5.write_bytes(open(f2, "rb").read().split(b">read600")[0])
    with pytest.raises(kb.KaijuError, match="contains more reads"):
        clf.classify_files(str(f1), str(f5), str(tmp_path / "x.tsv"))
    n, k = clf.classify_files(str(f5), None, str(tmp_path / "y.tsv"))           # the truncated file alone is fine
    assert n == 600
    clf.close()


@pytest.mark.parametrize("chunk", ["1024", "20000", ""])
def test_fastq_with_blank_lines(kb, golden, tmp_path, monkeypatch, chunk):
    """Empty lines between FASTQ records (and at the end of the file) are skipped where the reference's reader skips them (kaiju.cpp:288-289,
    341-348); empty lines inside a record count as the record's lines.  Output == the output for the clean files == the reference binary's
    (stored in tests/golden/ref_answers.npz.xz)."""
    if chunk:
        monkeypatch.setenv("KJ_INGEST_CHUNK", chunk)
    clean1, clean2, b1, b2 = gw.write_gpu_blank_line_fastq(str(tmp_path))
    clf = kb.Classifier(golden.fmi, golden.nodes, device=0, params=kb.make_params("greedy", e=3))
    outs = []
    for a, b in ((clean1, clean2), (b1, b2), (b1, clean2), (clean1, None), (b1, None)):
        o = str(tmp_path / "o.tsv"); n, k = clf.classify_files(a, b, o, verbose=True)
        assert n == 500
        outs.append(open(o).read())
    assert outs[0] == outs[1] == outs[2] and outs[3] == outs[4] and outs[0].count("C\t") > 200
    clf.close()
    from helpers import parse_kaiju_output
    ans = gw.ref_answers()                                                   # the reference binary's output for b1 (+ b2), stored
    assert parse_kaiju_output(outs[1]) == gw.stored_run(ans, "gpu_blank_pe")
    assert parse_kaiju_output(outs[4]) == gw.stored_run(ans, "gpu_blank_se")


def test_per_taxon_counts(kb, golden, tmp_path, monkeypatch):
    """The dense per-taxon count vector in HBM (kaiju2table's input): equals a histogram of the per-read results for the host-buffer,
    device-buffer and file entry points; a call repeated after a variant-ring overflow is counted once."""
    import torch
    names, s1, o1, s2, o2 = golden.reads("pe150"); n = len(names)
    clf = kb.Classifier(golden.fmi, golden.nodes, device=0, params=kb.make_params("mem"))
    def hist(t):
        u, c = np.unique(t, return_counts=True); return dict(zip(u.tolist(), c.tolist()))
    tax, _ = clf.classify(s1, o1, s2, o2)
    ids, cnt = clf.counts()
    assert dict(zip(ids.tolist(), cnt.tolist())) == hist(tax) and int(cnt.sum()) == n
    tax2, _ = clf.classify(s1, o1)                                  # a second call accumulates
    ids, cnt = clf.counts(); exp = hist(np.concatenate([tax, tax2]))
    assert dict(zip(ids.tolist(), cnt.tolist())) == exp
    clf.counts_reset()
    d = [torch.from_numpy(x.view(np.int64) if x.dtype == np.uint64 else x).cuda() for x in (s1, o1, s2, o2)]
    dt = torch.zeros(n, dtype=torch.int64, device="cuda")
    clf.classify_device(d[0].data_ptr(), d[1].data_ptr(), d[2].data_ptr(), d[3].data_ptr(), n, dt.data_ptr()); torch.cuda.synchronize(); clf.check_errors()
    assert int(clf.counts()[1].sum()) == 0                          # the device entry point leaves counting to the caller
    clf.counts_add_device(dt.data_ptr(), n); ids, cnt = clf.counts()
    assert dict(zip(ids.tolist(), cnt.tolist())) == hist(tax)
    # the count vector is a plain device array: torch (and therefore NCCL all-reduce) can address it in place
    from kaiju_b200.sharding import _DevArray
    ptr, m = clf.counts_device_ptr
    view = torch.as_tensor(_DevArray(ptr, m, "<i8"), device="cuda:0")
    assert int(view.sum().item()) == n
    # files
    clf.counts_reset()
    gold = os.path.dirname(golden.fmi)
    k, _ = clf.classify_files(os.path.join(gold, "pe150_1.fq.gz"), os.path.join(gold, "pe150_2.fq.gz"), str(tmp_path / "o.tsv"))
    ids, cnt = clf.counts()
    assert k == n and dict(zip(ids.tolist(), cnt.tolist())) == hist(tax)
    clf.close()
    # overflow + retry counts once
    other = SynthDB(3000, 777); s, o = other.long_reads(61, 0, 120, 3000, 16383)
    monkeypatch.setenv("KJ_VARIANT_CAP", "128")
    clf = kb.Classifier(golden.fmi, golden.nodes, device=0, params=kb.make_params("greedy", m=9, e=8, s=30, seed=5, E=1e-9))
    t, _ = clf.classify(s, o); ids, cnt = clf.counts()
    assert int(cnt.sum()) == 120 and dict(zip(ids.tolist(), cnt.tolist())) == hist(t)
    clf.close()


def test_native_index_file(kb, golden, tmp_path):
    """A context created from the device-native index file classifies exactly like one created from .fmi + nodes.dmp (API and CLI)."""
    import subprocess
    from conftest import ROOT
    native = str(tmp_path / "db.kjb")
    kb.write_native_index(golden.fmi, golden.nodes, native)
    names, s1, o1, s2, o2 = golden.reads("pe150")
    for cfg in ("mem_default", "greedy_default"):
        clf = kb.Classifier(native, None, device=0, params=kb_params(kb, GOLDEN_CONFIGS[cfg]))
        tax, best = clf.classify(s1, o1, s2, o2)
        etax, ebest, _ = golden.expected(cfg, "pe150")
        assert np.array_equal(tax, etax) and np.array_equal(best, ebest)
        clf.close()
    cli = os.path.join(ROOT, "kaiju_b200", "kaiju-b200"); gold = os.path.dirname(golden.fmi)
    native2 = str(tmp_path / "db2.kjb")
    subprocess.check_call([cli, "-t", golden.nodes, "-f", golden.fmi, "-w", native2])
    assert open(native, "rb").read() == open(native2, "rb").read()
    out = str(tmp_path / "o.tsv")
    subprocess.check_call([cli, "-f", native2, "-i", os.path.join(gold, "pe150_1.fq.gz"), "-j", os.path.join(gold, "pe150_2.fq.gz"), "-a", "mem", "-o", out])
    etax, _, _ = golden.expected("mem_default", "pe150")
    got = [l.split("\t") for l in open(out).read().splitlines()]
    assert [int(p[2]) for p in got] == [int(t) for t in etax] and [p[1] for p in got] == list(names)
    with pytest.raises(kb.KaijuError):
        kb.Classifier(golden.fmi, None, device=0, params=kb.make_params("mem"))        # a reference .fmi is not a native index


def test_index_with_bwtlen_multiple_of_65536(kb, tmp_path):
    """The reference's FM-index checkpoint quirk for bwtlen = m * 2^16 is reproduced on the GPU (oracle pinned to the reference for this
    case in tests/test_oracle_vs_ref.py), for the 32-bit, 64-bit and table-free kernels and through the device-native index file."""
    from helpers import make_quirk_db, pack_reads
    fmi, nodes, reads = make_quirk_db(str(tmp_path))
    seq, off = pack_reads(reads); orc = Oracle(fmi, nodes)
    native = str(tmp_path / "q.kjb"); kb.write_native_index(fmi, nodes, native)
    for kw in (dict(mode="mem"), dict(mode="greedy"), dict(mode="greedy", e=5, s=40)):
        otax, obest = orc.classify_batch(make_params(**kw), seq, off)
        for src in ((fmi, nodes), (native, None)):
            clf = kb.Classifier(src[0], src[1], device=0, params=kb_params(kb, kw))
            tax, best = clf.classify(seq, off)
            assert np.array_equal(tax, otax) and np.array_equal(best, obest), (kw, src)
            clf.close()


def test_counts_table_equals_reference_kaiju2table(kb, golden, tmp_path):
    """reads -> per-taxon counts in HBM -> kaiju2table report (kj_counts_table) == the reference's kaiju2table run on the per-read output file
    (the reference's reports are stored in tests/golden/kaiju2table_reports.json.gz)."""
    gold = os.path.dirname(golden.fmi); d = str(tmp_path)
    gw.ranked_golden_taxonomy(golden.nodes, d)
    reports = gw.k2t_reports()
    clf = kb.Classifier(golden.fmi, golden.nodes, device=0, params=kb.make_params("mem"))
    out = d + "/reads.tsv"
    clf.classify_files(os.path.join(gold, "pe150_1.fq.gz"), os.path.join(gold, "pe150_2.fq.gz"), out)
    for i, (o, flags) in enumerate(gw.COUNTS_TABLE_OPTS):
        clf.counts_table(d + "/nodes.dmp", d + "/names.dmp", out, d + "/ours.tsv", **o)
        assert open(d + "/ours.tsv").read() == reports["counts%d" % i].replace("{LABEL}", out), o
    clf.close()
