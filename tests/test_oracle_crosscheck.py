"""The two independent CPU restatements (oracle/pyoracle.py, oracle/blu_oracle.cpp) must agree byte for
byte on the canonical JSONL (incl. serde_json float formatting) and on which inputs are data errors."""
import random

import pytest

import pyoracle as po
from helpers import CUTOFFS_16S, random_blast, random_taxonomy
from oracle_ffi import Oracle, OracleDataError


@pytest.mark.parametrize("seed", range(60))
def test_crosscheck(seed):
    rng = random.Random(seed)
    units = random_taxonomy(rng, n_leaves=rng.choice([5, 20, 60]), shared_root=rng.random() < 0.9)
    text = random_blast(rng, units, n_queries=rng.choice([1, 10, 40]), contiguous=rng.random() < 0.7,
                        low_pident=rng.choice([60.0, 45.0]))
    n_ok = 0
    for taxon in ("bacteria", "fungi", "custom"):
        for strat in ("cautious", "relaxed"):
            for use_taxid in (False, True):
                custom = None
                if taxon == "custom":
                    custom = CUTOFFS_16S if seed % 3 else {"domain": 50, "species": 99, "genus": 95}
                tax = {u["taxid"]: (u["numericLineage"] if use_taxid else u["textLineage"]) for u in units}
                try:
                    a = po.results_to_jsonl(po.build_consensus_identities(text, tax, taxon, strat, custom))
                except po.DataError:
                    a = None
                try:
                    o = Oracle([u["taxid"] for u in units], [tax[u["taxid"]] for u in units], taxon, strat, custom, threads=3)
                    b = o.run_raw(text)[0].decode()
                except OracleDataError:
                    b = None
                assert (a is None) == (b is None)
                if a is not None:
                    assert a == b
                    n_ok += 1


@pytest.mark.parametrize("bad", [b"", b"q\tacc\t1\t99.0\t10\t0\t0\t1\t10\t1\t10\t0.0\n", b"q\tacc\tN/A\t99.0\t10\t0\t0\t1\t10\t1\t10\t0.0\t50\n",
                                 b"q\tacc\t1\t99.0\t10\t0\t0\t1\t10\t1\t10\t0.0\t50\textra\n", b"q\t\"acc\t1\t99.0\t10\t0\t0\t1\t10\t1\t10\t0.0\t50\n",
                                 b"q\tacc\t1\t99.0\t10\t0\t0\t1\t10\t1\t10\t0.0\t50\r\n", b"q\tacc\t1\t9x\t10\t0\t0\t1\t10\t1\t10\t0.0\t50\n",
                                 b"q\tacc\t2\t99.0\t10\t0\t0\t1\t10\t1\t10\t0.0\t50\n",  # unmapped taxid in top group
                                 b"\n\n"])
def test_data_errors(bad):
    tax = {1: "d__a;p__b"}
    with pytest.raises(po.DataError):
        po.build_consensus_identities(bad, tax, "bacteria", "cautious")
    o = Oracle([1], ["d__a;p__b"], "bacteria", "cautious")
    with pytest.raises(OracleDataError):
        o.run_raw(bad)


def test_headers_without_hits():
    tax = {1: "d__a;p__b"}
    text = b"q2\tacc\t1\t99.0\t10\t0\t0\t1\t10\t1\t10\t0.0\t50\n"
    a = po.build_consensus_identities(text, tax, "bacteria", "cautious", headers=["q1", "q2", "q3"])
    assert [r["query"] for r in a] == ["q1", "q2", "q3"] and a[0]["taxon"] is None and a[2]["taxon"] is None
    o = Oracle([1], ["d__a;p__b"], "bacteria", "cautious")
    assert o.run(text, headers=["q1", "q2", "q3"]) == a
