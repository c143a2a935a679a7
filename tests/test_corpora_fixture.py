"""The corpora fixture is the reference's own data: every member matches the manifest (size and SHA-256 of every
file of the reference's resources/), and the oracle's compressed size + SHA-256 prefix of every file equals
SURVEY.md's B.2 table (tests/golden/corpus_table.json) -- for all 36 files as one batch."""
import hashlib
import os

import numpy as np
import pytest

import corpora_fixture as cf
import oracle_lib as o


def test_fixture_matches_manifest_and_table():
    files = cf.corpora()
    man = cf.manifest()
    assert len(man) == 36 and sorted(files) == sorted(r["file"] for r in man)
    for r in man:
        assert len(files[r["file"]]) == r["raw"] and hashlib.sha256(files[r["file"]]).hexdigest() == r["sha256"]
    table = {r["file"]: r for r in cf.corpus_table()}
    assert sorted(table) == sorted(files)
    assert all(table[f]["raw"] == len(files[f]) for f in files)
    assert sum(len(v) for k, v in files.items() if k.startswith(("calgary/", "canterbury/"))) == 6040451   # config 2


@pytest.mark.parametrize("triple", ["8,14,16", "8,22,24", "8,30,32"])
def test_oracle_reproduces_the_table_from_the_fixture(triple):
    """All 36 files as one batch through the oracle (one stream per file, all host threads): size and SHA prefix
    of every compressed stream equal the independent table; Linear gives the same bytes as Tree."""
    p = tuple(int(x) for x in triple.split(","))
    files = cf.corpora()
    names = sorted(files)
    data = np.frombuffer(b"".join(files[n] for n in names), dtype=np.uint8)
    off = np.zeros(len(names) + 1, dtype=np.uint64)
    np.cumsum([len(files[n]) for n in names], out=off[1:])
    table = {r["file"]: r for r in cf.corpus_table()}
    threads = min(len(os.sched_getaffinity(0)), 16)
    outs = {}
    for kind in (o.TREE, o.LINEAR) if triple == "8,14,16" else (o.TREE,):
        rc, slots, slot_off, out_len, status = o.compress_batch(data, off, kind, p, threads)
        assert rc == 0 and (status == 0).all()
        outs[kind] = [slots[int(slot_off[i]):int(slot_off[i]) + int(out_len[i])].tobytes() for i in range(len(names))]
    for i, n in enumerate(names):
        comp = outs[o.TREE][i]
        assert len(comp) == table[n][triple][0], n
        assert hashlib.sha256(comp).hexdigest()[:16] == table[n][triple][1], n
    if o.LINEAR in outs:
        small = [i for i, n in enumerate(names)]
        assert all(outs[o.LINEAR][i] == outs[o.TREE][i] for i in small)


def test_ecoli_stand_in_is_deterministic():
    d = cf.ecoli_stand_in()
    assert len(d) == cf.ECOLI_LEN and set(d) == set(b"acgt")
    assert hashlib.sha256(d).hexdigest()[:16] == "3f2cc99a6d154e97"
