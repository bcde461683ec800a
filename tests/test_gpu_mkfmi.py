"""GPU tests of the index construction (kj_mkfmi / kaiju_b200.build_index / kaiju-b200 -M mkfmi): the .fmi built on the device must be
byte for byte the file kaiju-mkbwt + kaiju-mkfmi write -- against the committed reference-built indexes, the stored checksums of the
reference's K-fold indexes, and (when oracle/_ref holds the reference tools) the reference run on seeded adversarial FASTAs."""
import os
import random
import subprocess
import numpy as np
import pytest
import golden_workloads as gw
from helpers import GOLDEN_DIR, REF_DIR, make_quirk_db

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CLI = os.path.join(ROOT, "kaiju_b200", "kaiju-b200")
AA = "ACDEFGHIKLMNPQRSTVWY"


@pytest.fixture(scope="module")
def kb(built):
    import kaiju_b200
    return kaiju_b200


def _bytes(p):
    with open(p, "rb") as f:
        return f.read()


def _golden_faa(d):
    import sys
    sys.path.insert(0, GOLDEN_DIR)
    from make_golden import write_db_faa
    write_db_faa(d + "/db.faa", d + "/nodes.dmp")
    return d + "/db.faa", d + "/nodes.dmp"


def test_golden_db_equals_committed_index(kb, tmp_path):
    faa, _ = _golden_faa(str(tmp_path))
    st = kb.build_index(faa, str(tmp_path / "db"), exponent=3)
    assert _bytes(str(tmp_path / "db.fmi")) == _bytes(os.path.join(GOLDEN_DIR, "db.fmi"))
    assert st["nseq"] > 800 and st["sort_rounds"] >= 2 and st["round_items"][0] == st["bwtlen"] - st["nseq"]
    assert not os.path.exists(str(tmp_path / "db.bwt"))


def test_quirk_db_equals_committed_index(kb, tmp_path):
    """bwtlen = 2 * 2^16: the index1 / index2 tables of the reference's checkpoint quirk come out as the reference writes them"""
    make_quirk_db(str(tmp_path))
    st = kb.build_index(str(tmp_path / "db.faa"), str(tmp_path / "q"), exponent=3)
    assert st["bwtlen"] == 2 * 65536
    assert _bytes(str(tmp_path / "q.fmi")) == _bytes(os.path.join(GOLDEN_DIR, "quirk_db.fmi"))


@pytest.mark.parametrize("copies", list(gw.KFOLD_COPIES))
def test_kfold_db_equals_reference_checksums(kb, tmp_path, copies):
    """every protein K times (identical sequences ordered by their terminators only): the host transcoder's checksums of the result
    equal those of the index kaiju-mkbwt / kaiju-mkfmi built for the same FASTA"""
    faa, nodes = _golden_faa(str(tmp_path))
    gw.kfold_fasta(faa, str(tmp_path / "rep.faa"), copies)
    kb.build_index(str(tmp_path / "rep.faa"), str(tmp_path / "rep"), exponent=3)
    got = kb.host_index_checksums(str(tmp_path / "rep.fmi"), nodes)
    assert np.array_equal(got, gw.ref_answers()["kfold%d_checksums" % copies]), got


# ---- seeded adversarial FASTAs against the reference tools
def _rand(rnd, n, letters=AA):
    return "".join(rnd.choice(letters) for _ in range(n))


def adversarial_faa(path, kind, seed):
    rnd = random.Random(seed * 1000 + sum(map(ord, kind)))
    recs = []                                            # (header line without '>', sequence text as written)
    if kind == "duplicates":
        base = [_rand(rnd, rnd.randint(5, 80)) for _ in range(6)]
        for i in range(400):
            recs.append(("D%d_%d" % (i, 100 + i % 9), rnd.choice(base)))
    elif kind == "prefixes":
        for i in range(60):
            p = _rand(rnd, rnd.randint(20, 120))
            for k in sorted(rnd.sample(range(1, len(p) + 1), 4)) + [len(p)]:
                recs.append(("P%d_%d" % (len(recs), k), p[:k]))
        rnd.shuffle(recs)
    elif kind == "homopolymers":
        for i in range(40):
            a = rnd.choice(AA); n = rnd.choice([30, 200, 1500])
            recs.append(("H%d" % i, rnd.choice(["", _rand(rnd, 3)]) + a * n + rnd.choice(["", _rand(rnd, 2), a])))
            recs.append(("R%d" % i, (_rand(rnd, 2) * rnd.randint(20, 300))))
        recs.append(("W", "W" * 3000)); recs.append(("W2", "W" * 2999))
    elif kind == "short_and_empty":
        for i in range(300):
            r = rnd.random()
            s = "" if r < 0.1 else _rand(rnd, 1) if r < 0.3 else _rand(rnd, rnd.randint(2, 40))
            recs.append(("S%d" % i, s))
        recs.append(("E_last", ""))
    elif kind == "letters":
        for i in range(200):
            s = _rand(rnd, rnd.randint(10, 90), AA + AA.lower() + "XXBZUJOx-.0123 ")
            recs.append(("L%d desc with\tspace" % i, s))
    elif kind == "layout":
        for i in range(150):
            s = _rand(rnd, rnd.randint(10, 200))
            recs.append(("C%d %s" % (i, "d" * rnd.randint(0, 30)), s))
        recs.append(("x" * 1200, _rand(rnd, 50)))       # an id line longer than the 999 bytes read of it
        recs.append(("y" * 300 + " d", _rand(rnd, 50)))  # an id longer than the 255 bytes stored
    elif kind == "many":
        n = 12000 if seed % 2 else 150
        for i in range(n):
            recs.append(("M%d_%d" % (i, i % 50), _rand(rnd, rnd.randint(1, 30))))
    with open(path, "wb") as f:
        if kind == "layout":
            f.write(b"text before the first record\n")
        nl = b"\r\n" if kind == "layout" else b"\n"
        for h, s in recs:
            f.write(b">" + h.encode() + nl)
            width = rnd.choice([60, 7, 1000]) if kind in ("layout", "letters") else 80
            for k in range(0, len(s), width):
                f.write(s[k:k + width].encode() + nl)
            if kind == "layout" and rnd.random() < 0.2:
                f.write(nl)
    return path


def _ref_build(faa, prefix, e, alphabet, with_fmi):
    mb = os.path.getsize(faa) * 2 / 1e6 + 1
    subprocess.check_call([os.path.join(REF_DIR, "kaiju-mkbwt"), "-n", "4", "-l", "%.3f" % mb, "-e", str(e), "-a", alphabet, "-o", prefix, faa],
                          stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
    if with_fmi:
        subprocess.check_call([os.path.join(REF_DIR, "kaiju-mkfmi"), prefix], stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)


KINDS = ["duplicates", "prefixes", "homopolymers", "short_and_empty", "letters", "layout", "many"]


@pytest.mark.skipif(not os.path.exists(os.path.join(REF_DIR, "kaiju-mkbwt")), reason="reference tools not built (oracle/_ref)")
@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("e,alphabet", [(3, AA), (5, AA), (0, AA), (3, "protein")])
def test_equals_reference_tools(kb, tmp_path, kind, e, alphabet):
    """.bwt, .sa and .fmi bytes equal kaiju-mkbwt + kaiju-mkfmi on the same FASTA (kaiju-mkfmi fails at -e 0, so there .bwt and .sa only)"""
    for seed in (1, 2):
        faa = adversarial_faa(str(tmp_path / ("%s%d.faa" % (kind, seed))), kind, seed)
        ref, got = str(tmp_path / "ref"), str(tmp_path / "got")
        _ref_build(faa, ref, e, alphabet, with_fmi=e > 0)
        kb.build_index(faa, got, exponent=e, alphabet=alphabet, write_bwt_sa=True)
        for ext in (".bwt", ".sa") + ((".fmi",) if e > 0 else ()):
            assert _bytes(got + ext) == _bytes(ref + ext), (kind, seed, ext)


def test_refused_inputs(kb, tmp_path):
    import kaiju_b200 as k
    p = tmp_path / "a.faa"
    p.write_text(">a\nMKV*LL\n")
    with pytest.raises(k.KaijuError, match="-5"):
        kb.build_index(str(p), str(tmp_path / "o"))
    p.write_text("no record here\n")
    with pytest.raises(k.KaijuError, match="-5"):
        kb.build_index(str(p), str(tmp_path / "o"))
    with pytest.raises(k.KaijuError, match="-2"):
        kb.build_index(str(tmp_path / "missing.faa"), str(tmp_path / "o"))
    with pytest.raises(k.KaijuError, match="-5"):
        kb.build_index(str(p), str(tmp_path / "o"), alphabet="ABCDEFGHIJKLMNOPQRSTUVWXY")


def test_cli_mkfmi(kb, tmp_path):
    faa, nodes = _golden_faa(str(tmp_path))
    r = subprocess.run([CLI, "-M", "mkfmi", "-i", faa, "-o", str(tmp_path / "c"), "-e", "3", "-d", "0", "-t", nodes, "-w", str(tmp_path / "c.kjx")],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    assert _bytes(str(tmp_path / "c.fmi")) == _bytes(os.path.join(GOLDEN_DIR, "db.fmi"))
    assert _bytes(str(tmp_path / "c.kjx"))[:8] == b"KJB200IX"
    r = subprocess.run([CLI, "-M", "mkfmi", "-i", faa, "-o", str(tmp_path / "p"), "-a", "protein"], capture_output=True, text=True)
    assert r.returncode == 0 and os.path.exists(str(tmp_path / "p.fmi")), r.stderr
    for bad, msg in ((["-o", str(tmp_path / "x")], "needs the protein FASTA"), (["-i", faa], "needs the protein FASTA"),
                     (["-i", faa, "-o", str(tmp_path / "x"), "-e", "17"], "0..16"),
                     (["-i", faa, "-o", str(tmp_path / "x"), "-a", "ABCDEFGHIJKLMNOPQRSTUVWXY"], "at most 24"),
                     (["-i", faa, "-o", str(tmp_path / "x"), "-a", "DNA"], "not supported"),
                     (["-i", faa, "-o", str(tmp_path / "x"), "-w", str(tmp_path / "n")], "needs nodes.dmp"),
                     (["-i", str(tmp_path / "nope.faa"), "-o", str(tmp_path / "x")], "could not open")):
        r = subprocess.run([CLI, "-M", "mkfmi"] + bad, capture_output=True, text=True)
        assert r.returncode == 1 and msg in r.stderr, (bad, r.stderr)
