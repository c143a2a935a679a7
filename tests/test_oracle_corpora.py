"""tests/corpora.rs restated for the oracle: round trip + exact byte accounting on the reference's
fixtures, plus the SURVEY.md Appendix B.2 size/SHA cross-check.  The fixtures come from
tests/golden/corpora/corpora.tar.xz, byte-identical to the reference's resources/ (its MANIFEST.json holds
their SHA-256, checked by tests/test_corpora_fixture.py)."""
import hashlib
import json
import os

import pytest

import corpora_fixture as cf
import oracle_lib as o

TABLE = json.load(open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "corpus_table.json")))
SMALL = [r for r in TABLE if r["raw"] <= 150000]


@pytest.mark.parametrize("triple", ["8,14,16", "8,22,24", "8,30,32"])
def test_corpus_table_tree(triple):
    """Every fixture <= 150 kB: size + sha prefix equal the independent B.2 table, round trip exact,
    decoder consumes exactly the compressed length (tests/corpora.rs:40-41,59,61)."""
    p = tuple(int(x) for x in triple.split(","))
    for row in SMALL:
        data = cf.corpora()[row["file"]]
        assert len(data) == row["raw"]
        rc, comp, ic, oc = o.compress(data, o.TREE, p)
        assert rc == o.OK and ic == len(data) and oc == len(comp)
        assert len(comp) == row[triple][0], row["file"]
        assert hashlib.sha256(comp).hexdigest()[:16] == row[triple][1], row["file"]
        rc, dec, ic, oc = o.decompress(comp, o.TREE, p, out_cap=len(data) + 16)
        assert rc == o.OK and dec == data and ic == len(comp) and oc == len(data)


def test_corpus_linear_equals_tree_small():
    """AdaptiveLinearModel and AdaptiveTreeModel give identical bytes (config 2's claim)."""
    for row in [r for r in TABLE if r["raw"] <= 60000]:
        data = cf.corpora()[row["file"]]
        for p in ((8, 14, 16), (8, 30, 32)):
            a = o.compress(data, o.LINEAR, p)
            b = o.compress(data, o.TREE, p)
            assert a == b, row["file"]
            d = o.decompress(a[1], o.LINEAR, p, out_cap=len(data) + 16)
            assert d[0] == o.OK and d[1] == data


def test_book1_cli_parameters():
    """Config 1: calgary/book1, Tree, (8,30,32) (src/main.rs:108)."""
    row = [r for r in TABLE if r["file"] == "calgary/book1"][0]
    data = cf.corpora()["calgary/book1"]
    rc, comp, ic, oc = o.compress(data, o.TREE, (8, 30, 32))
    assert (rc, ic, oc) == (o.OK, 768771, 435400)
    assert hashlib.sha256(comp).hexdigest()[:16] == row["8,30,32"][1]
    rc, dec, ic, oc = o.decompress(comp, o.TREE, (8, 30, 32), out_cap=len(data) + 16)
    assert rc == o.OK and dec == data and ic == 435400
