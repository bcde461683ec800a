"""GPU tests of the index construction on the device (kj_build.h): array for array against the host transcoder, the scaled (K-fold) index
against the index the reference's own kaiju-mkbwt/-mkfmi build for the K-fold FASTA (stored answers), the dense-index output, and a
genuinely wide index."""
import os
import numpy as np
import pytest
import golden_workloads as gw
from golden_workloads import golden_db
from helpers import Oracle, make_params, make_quirk_db

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def kb(built):
    import kaiju_b200
    return kaiju_b200


@pytest.mark.parametrize("force_wide", [False, True])
def test_device_build_equals_host_transcoder(kb, golden, monkeypatch, force_wide):
    """rank records, packed letters, taxon-reduced SA, sequence taxa and the k-mer table built by the kernels == the host transcoder's,
    for the narrow (64-row) and the wide (192-row) layout."""
    if force_wide:
        monkeypatch.setenv("KJ_FORCE_WIDE", "1")
    want = kb.host_index_checksums(golden.fmi, golden.nodes)
    clf = kb.Classifier(golden.fmi, golden.nodes, device=0, params=kb.make_params("mem"))
    got = clf.debug_index_checksums()
    assert int(got[6]) == (1 if force_wide else 0)
    assert np.array_equal(got, want), (got, want)
    monkeypatch.setenv("KJ_HOST_BUILD", "1")              # the upload path of the host transcoder gives the same context
    clf2 = kb.Classifier(golden.fmi, golden.nodes, device=0, params=kb.make_params("mem"))
    assert np.array_equal(clf2.debug_index_checksums(), want)
    names, s1, o1, s2, o2 = golden.reads("pe150")
    a = clf.classify(s1, o1, s2, o2); b = clf2.classify(s1, o1, s2, o2)
    assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1])
    clf.close(); clf2.close()


def test_device_build_quirk_index(kb, tmp_path):
    """bwtlen = m * 2^16: the reference's checkpoint quirk constants and the k-mer table come out of the device build as on the host"""
    fmi, nodes, reads = make_quirk_db(str(tmp_path))
    want = kb.host_index_checksums(fmi, nodes)
    clf = kb.Classifier(fmi, nodes, device=0, params=kb.make_params("mem"))
    assert np.array_equal(clf.debug_index_checksums(), want)
    clf.close()


@pytest.mark.parametrize("copies", list(gw.KFOLD_COPIES))
def test_scaled_index_equals_reference_built_kfold_index(kb, golden, copies):
    """kj_create_scaled(copies = K) == the index kaiju-mkbwt / kaiju-mkfmi build for the FASTA that holds every protein of the golden DB
    K times: same arrays in HBM (the host transcoder's checksums of the reference-built index are stored), the reference's classification
    on that index (MEM and Greedy, stored as a digest); and MEM results equal those on the base index."""
    ans = gw.ref_answers()
    big = kb.Classifier(golden.fmi, golden.nodes, device=0, params=kb.make_params("mem"), copies=copies)
    got = big.debug_index_checksums(); want = ans["kfold%d_checksums" % copies]
    # the sampled-SA arrays differ in length by the reference's dropped last entry only: compare everything else exactly, the SA through results
    assert np.array_equal(got[[0, 1, 3, 4, 5, 6]], want[[0, 1, 3, 4, 5, 6]]), (got, want)
    small = kb.Classifier(golden.fmi, golden.nodes, device=0, params=kb.make_params("mem"))
    s1, o1, s2, o2 = gw.kfold_reads()
    for mode in ("mem", "greedy"):
        for c in (big, small):
            c.set_params(kb.make_params(mode))
        a = big.classify(s1, o1, s2, o2)
        assert gw.result_digest(*a) == str(ans["kfold%d_%s_sha256" % (copies, mode)]), mode
        if mode == "mem":
            c0 = small.classify(s1, o1, s2, o2)
            assert np.array_equal(a[0], c0[0]) and np.array_equal(a[1], c0[1])
    assert (a[0] != 0).mean() > 0.4
    for c in (big, small):
        c.close()


def test_dense_taxon_indices(kb, golden):
    """kj_classify2 / kj_classify_device2: the uint32 dense indices map back to the 64-bit taxon ids through the counts' id list"""
    import torch
    names, s1, o1, s2, o2 = golden.reads("pe150")
    n = len(o1) - 1
    clf = kb.Classifier(golden.fmi, golden.nodes, device=0, params=kb.make_params("mem"))
    tax, best = clf.classify(s1, o1, s2, o2)
    pin = lambda a: torch.from_numpy(a.view(np.int64) if a.dtype == np.uint64 else a)
    h = [pin(np.ascontiguousarray(x)) for x in (s1, o1, s2, o2)]
    d = [x.cuda() for x in h]
    d_comp = torch.zeros(n, dtype=torch.int32, device="cuda"); d_tax = torch.zeros(n, dtype=torch.int64, device="cuda")
    clf.classify_device2(d[0].data_ptr(), d[1].data_ptr(), d[2].data_ptr(), d[3].data_ptr(), n, d_tax.data_ptr(), None, d_comp.data_ptr(), 0, 0, None)
    torch.cuda.synchronize(); clf.check_errors()
    ids = clf.compact_ids(); comp = d_comp.cpu().numpy().view(np.uint32)
    mapped = np.where(comp == 0xffffffff, np.uint64(0), ids[np.minimum(comp, len(ids) - 1)])
    assert np.array_equal(mapped, tax) and np.array_equal(d_tax.cpu().numpy().view(np.uint64), tax)
    # taxon output omitted, dense indices only
    d_comp2 = torch.zeros(n, dtype=torch.int32, device="cuda")
    clf.classify_device2(d[0].data_ptr(), d[1].data_ptr(), d[2].data_ptr(), d[3].data_ptr(), n, None, None, d_comp2.data_ptr(), 150, 150, None)
    torch.cuda.synchronize(); assert torch.equal(d_comp, d_comp2)
    # host buffers in, host taxa + device dense indices out
    h_tax = np.zeros(n, dtype=np.uint64); d_comp3 = torch.zeros(n, dtype=torch.int32, device="cuda")
    clf.classify2_ptrs(h[0].data_ptr(), h[1].data_ptr(), h[2].data_ptr(), h[3].data_ptr(), n, h_tax.ctypes.data, None, d_comp3.data_ptr())
    assert np.array_equal(h_tax, tax) and torch.equal(d_comp, d_comp3)
    clf.close()


def test_index_beyond_2_pow_32_rows(kb, golden):
    """A genuinely wide index (>= 2^32 BWT rows, not KJ_FORCE_WIDE): the committed golden index scaled past 2^32 rows (~20 GB in HBM);
    MEM results must equal the base index's, which are checked against the oracle."""
    import torch
    if torch.cuda.mem_get_info()[0] < (40 << 30):
        pytest.skip("needs 40 GB of free HBM")
    db = golden_db(); fmi, nodes = golden.fmi, golden.nodes
    small = kb.Classifier(fmi, nodes, device=0, params=kb.make_params("mem"))
    copies = (1 << 32) // small.bwtlen + 2
    big = kb.Classifier(fmi, nodes, device=0, params=kb.make_params("mem"), copies=copies)
    assert big.bwtlen >= (1 << 32)
    s1, o1, s2, o2 = db.reads(9, 0, 200000, 150, True)
    a = small.classify(s1, o1, s2, o2); b = big.classify(s1, o1, s2, o2)
    assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1])
    otax, obest = Oracle(fmi, nodes).classify_batch(make_params("mem"), s1[:int(o1[5000])], o1[:5001], s2[:int(o2[5000])], o2[:5001])
    assert np.array_equal(a[0][:5000], otax) and np.array_equal(a[1][:5000], obest)
    assert (a[0] != 0).mean() > 0.5
    small.close(); big.close()


def test_classify_multi_and_cli_device_list(kb, golden, tmp_path):
    """Several contexts in one process (kj_classify_multi: contiguous shards, one host thread per context) give the single-context result;
    the CLI hands the data sets of its -i/-j/-o lists to the devices of -d (here: every visible device, or device 0 twice over the ABI)."""
    import gzip, shutil, subprocess
    from conftest import ROOT
    if not hasattr(kb.lib(), "kj_classify_multi"):
        pytest.skip("library build without kj_classify_multi")
    names, s1, o1, s2, o2 = golden.reads("pe150")
    nd = max(1, kb.device_count())
    one = kb.Classifier(golden.fmi, golden.nodes, device=0, params=kb.make_params("greedy"))
    want = one.classify(s1, o1, s2, o2)
    ctxs = [kb.Classifier(golden.fmi, golden.nodes, device=d % nd, params=kb.make_params("greedy")) for d in range(3)]
    got = kb.classify_multi(ctxs, s1, o1, s2, o2)
    assert np.array_equal(got[0], want[0]) and np.array_equal(got[1], want[1])
    for c in ctxs + [one]:
        c.close()
    g = os.path.dirname(golden.fmi); d = str(tmp_path)
    def plain(src, dst):
        with gzip.open(src, "rb") as f, open(dst, "wb") as h:
            shutil.copyfileobj(f, h)
        return dst
    a = plain(g + "/pe150_1.fq.gz", d + "/a.fq"); b = plain(g + "/pe150_2.fq.gz", d + "/b.fq"); c1 = plain(g + "/se100.fq.gz", d + "/c.fq")
    cli = os.path.join(ROOT, "kaiju_b200", "kaiju-b200")
    base = [cli, "-t", golden.nodes, "-f", golden.fmi, "-a", "mem"]
    subprocess.run(base + ["-i", ",".join([a, c1, a]), "-o", ",".join([d + "/o1", d + "/o2", d + "/o3"]), "-d", "all"], check=True, stderr=subprocess.DEVNULL)
    subprocess.run(base + ["-i", a, "-o", d + "/r1", "-d", "0"], check=True, stderr=subprocess.DEVNULL)
    subprocess.run(base + ["-i", c1, "-o", d + "/r2"], check=True, stderr=subprocess.DEVNULL)
    assert open(d + "/o1").read() == open(d + "/r1").read() == open(d + "/o3").read() and open(d + "/o2").read() == open(d + "/r2").read()


def test_kmer_table_k7(kb, golden, monkeypatch):
    """The 7-mer interval table (the MEM kernels use it on indexes of >= 5e7 rows; forced here for both modes on the small golden index):
    results equal the oracle's and the default table's."""
    names, s1, o1, s2, o2 = golden.reads("pe150")
    ref = kb.Classifier(golden.fmi, golden.nodes, device=0, params=kb.make_params("mem"))
    monkeypatch.setenv("KJ_KMER_K", "7")
    clf = kb.Classifier(golden.fmi, golden.nodes, device=0, params=kb.make_params("mem"))
    orc = Oracle(golden.fmi, golden.nodes)
    for mode in ("mem", "greedy"):
        ref.set_params(kb.make_params(mode)); clf.set_params(kb.make_params(mode))
        a = clf.classify(s1, o1, s2, o2); b = ref.classify(s1, o1, s2, o2)
        assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1]), mode
        otax, obest = orc.classify_batch(make_params(mode), s1, o1, s2, o2)
        assert np.array_equal(a[0], otax) and np.array_equal(a[1], obest), mode
    clf.set_params(kb.make_params("mem", m=7)); ref.set_params(kb.make_params("mem", m=7))      # the shortest fragment length the table serves
    a = clf.classify(s1, o1, s2, o2); b = ref.classify(s1, o1, s2, o2)
    assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1])
    clf.close(); ref.close()
