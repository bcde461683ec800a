"""kj_table_write (kaiju2table's report from per-taxon counts) against the UNMODIFIED reference kaiju2table, byte for byte: its reports
for these inputs are stored in tests/golden/kaiju2table_reports.json.gz (tests/golden/make_golden_ref.py).  CPU only."""
import random
import numpy as np
import pytest
import golden_workloads as gw
from golden_workloads import make_taxonomy


@pytest.mark.parametrize("o", gw.TABLE_OPTS)
def test_table_equals_reference_kaiju2table(built, tmp_path, o):
    import kaiju_b200 as kb
    d = str(tmp_path); i = gw.TABLE_OPTS.index(o); reports = gw.k2t_reports()
    reads, rnd = gw.table_input(d, o)
    label = d + "/in.tsv"
    ids, cnt = np.unique(np.array(reads, dtype=np.uint64), return_counts=True)
    perm = rnd.sample(range(len(ids)), len(ids))          # the order of the count vector must not matter
    kb.write_table(ids[perm], cnt[perm], d + "/nodes.dmp", d + "/names.dmp", label, d + "/ours.tsv", **o)
    assert open(d + "/ours.tsv").read() == reports["table%d" % i].replace("{LABEL}", label)
    # two data sets in one report (kaiju2table in1 in2): second call appends
    kb.write_table(ids, cnt, d + "/nodes.dmp", d + "/names.dmp", label, d + "/ours.tsv", append=True, **o)
    assert open(d + "/ours.tsv").read() == reports["table%d_twice" % i].replace("{LABEL}", label)


def test_table_argument_errors(built, tmp_path):
    import kaiju_b200 as kb
    d = str(tmp_path); make_taxonomy(d, random.Random(1))
    ids = np.array([0], dtype=np.uint64); cnt = np.array([3], dtype=np.uint64)
    for bad in (dict(rank="kingdom"), dict(rank="species", min_percent=1.0, min_read_count=2), dict(rank="genus", full_path=True, rank_list="genus"),
                dict(rank="genus", rank_list="phylum,species"), dict(rank="species", min_percent=101.0)):
        with pytest.raises(kb.KaijuError):
            kb.write_table(ids, cnt, d + "/nodes.dmp", d + "/names.dmp", "x", d + "/o.tsv", **bad)
