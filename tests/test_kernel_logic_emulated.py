"""The product's kernel source (kaiju_b200/csrc/kj_core*.h) executed on the CPU warp emulator (tests/emu) against the
golden reference outputs and the oracle.  This checks the device LOGIC without a GPU; the `gpu` tests check the real thing."""
import ctypes as C
import os
import numpy as np
import pytest
from conftest import GOLDEN_CONFIGS, ROOT
from helpers import Oracle, make_params, SynthDB


class KjParams(C.Structure):
    _fields_ = [("mode", C.c_int32), ("min_fragment_length", C.c_uint32), ("mismatches", C.c_uint32), ("min_score", C.c_uint32),
                ("seed_length", C.c_uint32), ("use_evalue", C.c_int32), ("min_evalue", C.c_double), ("seg", C.c_int32), ("input_is_protein", C.c_int32), ("name_mode", C.c_int32)]


@pytest.fixture(scope="module")
def emu(built):
    E = C.CDLL(os.path.join(ROOT, "tests", "emu", "libkjemu.so"))
    E.kjemu_create.restype = C.c_void_p; E.kjemu_create.argtypes = [C.c_char_p, C.c_char_p, C.POINTER(KjParams)]
    E.kjemu_destroy.argtypes = [C.c_void_p]
    E.kjemu_classify.argtypes = [C.c_void_p] + [C.c_void_p] * 4 + [C.c_uint64, C.c_void_p, C.c_void_p, C.c_int]
    return E


def emu_classify(E, fmi, nodes, P, s1, o1, s2, o2):
    kp = KjParams(**P); h = E.kjemu_create(fmi.encode(), nodes.encode(), C.byref(kp)); assert h
    n = len(o1) - 1; tax = np.zeros(n, dtype=np.uint64); best = np.zeros(n, dtype=np.uint32)
    rc = E.kjemu_classify(h, s1.ctypes.data, o1.ctypes.data, s2.ctypes.data if s2 is not None else None, o2.ctypes.data if s2 is not None else None,
                          n, tax.ctypes.data, best.ctypes.data, 4)
    E.kjemu_destroy(h); assert rc == 0
    return tax, best


@pytest.mark.parametrize("cfg", sorted(GOLDEN_CONFIGS))
@pytest.mark.parametrize("tag", ["pe150", "se100"])
def test_emulated_kernel_matches_reference_golden(emu, golden, cfg, tag):
    names, s1, o1, s2, o2 = golden.reads(tag)
    tax, best = emu_classify(emu, golden.fmi, golden.nodes, make_params(**GOLDEN_CONFIGS[cfg]), s1, o1, s2, o2)
    etax, ebest, _ = golden.expected(cfg, tag)
    bad = np.nonzero((tax != etax) | (best != ebest))[0]
    assert len(bad) == 0, [(names[i], int(tax[i]), int(etax[i]), int(best[i]), int(ebest[i])) for i in bad[:5]]


@pytest.mark.parametrize("cfg", [c for c in sorted(GOLDEN_CONFIGS) if c.startswith("greedy")])
def test_emulated_two_kernel_greedy_matches_reference_golden(emu, golden, cfg, monkeypatch):
    """Greedy as the GPU runs it: front end -> per-item record (queue, translated arrays; SEG class scan done there) -> work space wiped -> search."""
    monkeypatch.setenv("KJ_EMU_SPLIT", "1")
    for tag in ("pe150", "se100"):
        names, s1, o1, s2, o2 = golden.reads(tag)
        tax, best = emu_classify(emu, golden.fmi, golden.nodes, make_params(**GOLDEN_CONFIGS[cfg]), s1, o1, s2, o2)
        etax, ebest, _ = golden.expected(cfg, tag)
        bad = np.nonzero((tax != etax) | (best != ebest))[0]
        assert len(bad) == 0, [(names[i], int(tax[i]), int(etax[i]), int(best[i]), int(ebest[i])) for i in bad[:5]]


def test_emulated_kernel_matches_oracle_on_random_parameters(emu, golden):
    """Seeded sweep over the CLI parameter space (-a, -m, -e, -s, -E, -x/-X): kernel logic (emulated) == oracle (pinned to the reference)."""
    import random
    rnd = random.Random(7)
    names, s1, o1, s2, o2 = golden.reads("pe150")
    orc = Oracle(golden.fmi, golden.nodes)
    for trial in range(10):
        mode = rnd.choice(["mem", "greedy"])
        kw = dict(mode=mode, m=rnd.choice([3, 6, 9, 11, 12, 15, 25]), seg=rnd.random() < 0.7)
        if mode == "greedy":
            kw.update(e=rnd.choice([0, 1, 2, 3, 4, 6, 8]), s=rnd.choice([20, 40, 65, 80, 110]), E=rnd.choice([10.0, 0.01, 1e-5, 1e-12]))
        P = make_params(**kw)
        otax, obest = orc.classify_batch(P, s1, o1, s2, o2)
        tax, best = emu_classify(emu, golden.fmi, golden.nodes, P, s1, o1, s2, o2)
        bad = np.nonzero((tax != otax) | (best != obest))[0]
        assert len(bad) == 0, (kw, [(names[i], int(tax[i]), int(otax[i]), int(best[i]), int(obest[i])) for i in bad[:5]])


def emu_classify_rc(E, fmi, nodes, P, s1, o1):
    kp = KjParams(**P); h = E.kjemu_create(fmi.encode(), nodes.encode(), C.byref(kp)); assert h
    n = len(o1) - 1; tax = np.zeros(n, dtype=np.uint64); best = np.zeros(n, dtype=np.uint32)
    rc = E.kjemu_classify(h, s1.ctypes.data, o1.ctypes.data, None, None, n, tax.ctypes.data, best.ctypes.data, 4)
    E.kjemu_destroy(h)
    return rc, tax, best


@pytest.mark.parametrize("kw", [dict(mode="mem"), dict(mode="greedy"), dict(mode="mem", m=7, seg=False), dict(mode="greedy", e=5, s=40, E=1e-3)])
def test_emulated_kernel_long_reads_and_protein_input(emu, golden, kw):
    """Reads up to KJ_MAX_READ_LEN (16383 bases) and protein input (-p, up to 5461 residues): kernel logic (emulated) == oracle."""
    db = SynthDB(800, 3); orc = Oracle(golden.fmi, golden.nodes)
    for prot, (s, o) in ((False, db.long_reads(41, 0, 250, 300, 16383)), (True, db.protein_reads(42, 0, 1200, 5, 5461))):
        P = make_params(protein=prot, **kw)
        otax, obest = orc.classify_batch(P, s, o)
        rc, tax, best = emu_classify_rc(emu, golden.fmi, golden.nodes, P, s, o)
        bad = np.nonzero((tax != otax) | (best != obest))[0]
        assert rc == 0 and len(bad) == 0, (kw, prot, rc, [(int(i), int(tax[i]), int(otax[i]), int(best[i]), int(obest[i])) for i in bad[:5]])
        assert (otax != 0).mean() > 0.5


def test_emulated_kernel_reports_variant_ring_overflow(emu, golden, monkeypatch):
    """A full Greedy variant ring is flagged (never silently truncated); the library reacts by enlarging the ring (GPU test)."""
    s, o = SynthDB(3000, 777).long_reads(61, 0, 120, 3000, 16383)
    P = make_params(mode="greedy", e=8, s=30, m=9, seed=5, E=1e-9)
    monkeypatch.setenv("KJ_VARIANT_CAP", "128")           # test hook: a ring of 128 entries is too small for these reads
    rc, _, _ = emu_classify_rc(emu, golden.fmi, golden.nodes, P, s, o)
    assert rc == -406                                     # KJ_ERR_OVERFLOW - 100 * flag 4
    monkeypatch.setenv("KJ_VARIANT_CAP", "512")
    rc, tax, best = emu_classify_rc(emu, golden.fmi, golden.nodes, P, s, o)
    otax, obest = Oracle(golden.fmi, golden.nodes).classify_batch(P, s, o)
    assert rc == 0 and np.array_equal(tax, otax) and np.array_equal(best, obest)


def test_native_index_file_roundtrip(emu, golden, tmp_path, monkeypatch):
    """Device-native index file (kj_native_index_write / kj_create_from_native): every array survives write + read bit for bit,
    for the 32-bit and the 64-bit interval layouts; truncated or foreign files are refused."""
    emu.kjemu_native_roundtrip.argtypes = [C.c_char_p] * 3; emu.kjemu_native_read.argtypes = [C.c_char_p]
    p = str(tmp_path / "db.kjb")
    assert emu.kjemu_native_roundtrip(golden.fmi.encode(), golden.nodes.encode(), p.encode()) == 0
    assert os.path.getsize(p) > 1000
    blob = open(p, "rb").read()
    open(p + ".trunc", "wb").write(blob[:len(blob) // 2]); open(p + ".long", "wb").write(blob + b"x"); open(p + ".bad", "wb").write(b"NOTANIDX" + blob[8:])
    for suffix in (".trunc", ".long", ".bad"):
        assert emu.kjemu_native_read((p + suffix).encode()) != 0
    assert emu.kjemu_native_read(golden.fmi.encode()) != 0            # a reference .fmi is not a native index
    monkeypatch.setenv("KJ_FORCE_WIDE", "1")
    assert emu.kjemu_native_roundtrip(golden.fmi.encode(), golden.nodes.encode(), p.encode()) == 0


def test_emulated_kernel_on_index_with_bwtlen_multiple_of_65536(emu, built, tmp_path, monkeypatch):
    """The reference's checkpoint quirk (tests/test_oracle_vs_ref.py::test_bwtlen_multiple_of_65536) is reproduced by the device code:
    rank correction for the last 129 rows, in the k-mer table, in the SA walk, and the general 'recorded match' rule of maxMatches."""
    from helpers import make_quirk_db, pack_reads
    fmi, nodes, reads = make_quirk_db(str(tmp_path))
    seq, off = pack_reads(reads); orc = Oracle(fmi, nodes)
    for env in ({}, {"KJ_FORCE_WIDE": "1"}, {"KJ_KMER_K": "0"}):
        for k, v in env.items():
            monkeypatch.setenv(k, v)
        for kw in (dict(mode="mem"), dict(mode="greedy"), dict(mode="greedy", e=5, s=40)):
            P = make_params(**kw); otax, obest = orc.classify_batch(P, seq, off)
            rc, tax, best = emu_classify_rc(emu, fmi, nodes, P, seq, off)
            assert rc == 0 and np.array_equal(tax, otax) and np.array_equal(best, obest), (env, kw)
        for k in env:
            monkeypatch.delenv(k)


def test_evalue_break_points_equal_the_reference_expression(emu):
    """The E-value gate on the device = number of break points below the query length.  For every score k and query lengths around and
    far from the break points, that integer threshold must agree with the reference's expression (ConsumerThread.cpp:500-513)
    evaluated directly: Evalue = db_length * query_len * 2^-((0.3176 * k + 2.009915479) / 0.6931471805) > min_Evalue -> rejected."""
    import math, random
    emu.kjemu_evalue_breaks.argtypes = [C.c_double, C.c_double, C.POINTER(C.c_double), C.c_int]
    rnd = random.Random(3)
    def rejected(db, q, k, E):
        bitscore = (0.3176 * k - (-2.009915479)) / 0.6931471805
        return db * q * math.pow(2, -1 * bitscore) > E
    for E in (10.0, 0.01, 1e-5, 1e-12, 1e-30):
        for db in (8.2e5, 1.99e8, 2.7e10):
            buf = (C.c_double * 4096)(); n = emu.kjemu_evalue_breaks(E, db, buf, 4096); assert 0 < n <= 4096
            br = [buf[i] for i in range(n)]
            assert all(br[i] <= br[i + 1] for i in range(n - 1))
            qs = [a / 3.0 + b / 3.0 for a in (33, 100, 150, 151, 301, 5000, 16383) for b in (0, 149, 150, 16383)] + [float(x) for x in (11, 300, 5461)]
            for k in range(0, min(n, 400), 7):        # doubles right at a break point
                if 0 < br[k] < 1e11:
                    qs += [br[k], math.nextafter(br[k], math.inf), math.nextafter(br[k], 0.0)]
            for q in qs:
                thr = sum(1 for x in br if x < q)                       # what the device computes
                ks = sorted(set([max(0, thr - 2), max(0, thr - 1), thr, thr + 1, thr + 5] + [rnd.randrange(0, 2000) for _ in range(6)]))
                for k in ks:
                    assert (k >= thr) == (not rejected(db, q, k, E)), (E, db, q, k, thr)


XP_CONFIGS = {"mem_default": dict(mode="mem"), "mem_m5_noseg": dict(mode="mem", m=5, seg=False), "greedy_default": dict(mode="greedy"),
              "greedy_e5_s40": dict(mode="greedy", e=5, s=40), "greedy_e0": dict(mode="greedy", e=0)}


@pytest.mark.parametrize("cfg", sorted(XP_CONFIGS))
def test_emulated_name_frontend_matches_reference_kaijux(emu, golden, cfg):
    """kaijux semantics (name_mode: sequences numbered under one root, MEM matches in maxMatches order) on the emulated kernel logic ==
    the committed output of the reference's own kaijux binary (tests/golden/make_golden_xp.py), line by line."""
    import gzip
    import kaiju_b200 as kb
    from conftest import GOLD
    L = kb.lib(); L.kj_fmi_seq_name.restype = C.c_char_p; L.kj_fmi_seq_name.argtypes = [C.c_void_p, C.c_int32]
    f = C.c_void_p(); assert L.kj_fmi_load(golden.fmi.encode(), C.byref(f)) == 0
    emu.kjemu_classify_ids.argtypes = [C.c_void_p] + [C.c_void_p] * 4 + [C.c_uint64] + [C.c_void_p] * 4 + [C.c_int]
    kw = XP_CONFIGS[cfg]
    for tag in ("se100", "pe150"):
        names, s1, o1, s2, o2 = golden.reads(tag)
        P = make_params(**kw); P["name_mode"] = 1
        kp = KjParams(**P); h = emu.kjemu_create(golden.fmi.encode(), None, C.byref(kp)); assert h
        n = len(o1) - 1; tax = np.zeros(n, np.uint64); best = np.zeros(n, np.uint32); ids = np.zeros((n, 21), np.uint64); nids = np.zeros(n, np.uint8)
        rc = emu.kjemu_classify_ids(h, s1.ctypes.data, o1.ctypes.data, s2.ctypes.data if s2 is not None else None, o2.ctypes.data if s2 is not None else None,
                                    n, tax.ctypes.data, best.ctypes.data, ids.ctypes.data, nids.ctypes.data, 4)
        emu.kjemu_destroy(h); assert rc == 0
        want = gzip.open(os.path.join(GOLD, "expected_x_%s_%s.tsv.gz" % (cfg, tag)), "rt").read().split("\n")
        m3 = 3 * kw.get("m", 11); bad = []
        for i in range(n):
            l1 = int(o1[i + 1] - o1[i]); gate = l1 < m3 if s2 is None else (l1 < m3 and int(o2[i + 1] - o2[i]) < m3)
            if gate:
                line = "U\t%s\t0" % names[i]
            elif not tax[i] or not nids[i]:
                line = "U\t%s" % names[i]
            else:
                line = "C\t%s\t%d\t%s,\t" % (names[i], best[i], ",".join(L.kj_fmi_seq_name(f, int(x) - 2).decode() for x in ids[i, :nids[i]]))
            if line != want[i]:
                bad.append((line[:120], want[i][:120]))
        assert not bad, bad[:3]
    L.kj_fmi_free(f)


@pytest.mark.parametrize("cfg", ["mem_default", "mem_m5_noseg", "greedy_default", "greedy_e5_s40"])
def test_emulated_verbose_columns_match_reference(emu, golden, cfg):
    """All seven columns of `kaiju -v` (taxon, best, id set, accession set, fragment strings) from the emulated kernel logic == the raw output of the
    reference binary (tests/golden/expected_v7_*)."""
    import gzip
    import kaiju_b200 as kb
    from conftest import GOLD
    L = kb.lib(); L.kj_fmi_accession.restype = C.c_char_p; L.kj_fmi_accession.argtypes = [C.c_void_p, C.c_uint32]
    f = C.c_void_p(); assert L.kj_fmi_load(golden.fmi.encode(), C.byref(f)) == 0
    emu.kjemu_classify_v2.argtypes = [C.c_void_p] + [C.c_void_p] * 4 + [C.c_uint64] + [C.c_void_p] * 7 + [C.c_uint32, C.c_void_p, C.c_int]
    kw = XP_CONFIGS[cfg]; ST = 2048
    for tag in ("se100", "pe150"):
        names, s1, o1, s2, o2 = golden.reads(tag)
        kp = KjParams(**make_params(**kw)); h = emu.kjemu_create(golden.fmi.encode(), golden.nodes.encode(), C.byref(kp)); assert h
        n = len(o1) - 1; tax = np.zeros(n, np.uint64); best = np.zeros(n, np.uint32); ids = np.zeros((n, 21), np.uint64); nids = np.zeros(n, np.uint8)
        acc = np.zeros((n, 20), np.uint32); nacc = np.zeros(n, np.uint8); frag = np.zeros((n, ST), np.uint8); flen = np.zeros(n, np.uint32)
        rc = emu.kjemu_classify_v2(h, s1.ctypes.data, o1.ctypes.data, s2.ctypes.data if s2 is not None else None, o2.ctypes.data if s2 is not None else None, n,
                                   tax.ctypes.data, best.ctypes.data, ids.ctypes.data, nids.ctypes.data, acc.ctypes.data, nacc.ctypes.data, frag.ctypes.data, ST, flen.ctypes.data, 4)
        emu.kjemu_destroy(h); assert rc == 0
        want = gzip.open(os.path.join(GOLD, "expected_v7_%s_%s.tsv.gz" % (cfg, tag)), "rt").read().split("\n"); bad = []
        for i in range(n):
            line = "U\t%s\t0" % names[i] if not tax[i] else "C\t%s\t%d\t%d\t%s,\t%s\t%s" % (
                names[i], tax[i], best[i], ",".join(str(int(x)) for x in ids[i, :nids[i]]),
                "".join(L.kj_fmi_accession(f, int(a)).decode() + "," for a in acc[i, :nacc[i]]), bytes(frag[i, :flen[i]]).decode())
            if line != want[i]:
                bad.append((line[:160], want[i][:160]))
        assert not bad, bad[:3]
    L.kj_fmi_free(f)
