"""The variant tables of tests/consensus_variants.py -- top groups of 9..1000 rows, bit scores beyond int32 -- through the three
CPU implementations of the path: oracle/pyoracle.py, oracle/blu_oracle.cpp and the product's device core compiled for the host.
They agree byte for byte, and on which inputs are data errors, for all four taxa and both strategies.  The GPU test of the same
variants (tests/test_gpu_consensus_classes.py) compares the kernels with the C++ oracle; this pins that oracle to the other two
on groups of these sizes."""
from hypothesis import HealthCheck, given, settings
from hypothesis import strategies as st

import consensus_variants as V
from generators import _text, _three_ways


@settings(max_examples=40, derandomize=True, database=None, deadline=None, suppress_health_check=[HealthCheck.too_slow, HealthCheck.data_too_large])
@given(st.data())
def test_consensus_variants_three_ways(data):
    tax = data.draw(V.lineage_maps())
    queries = data.draw(V.tables(tax))
    tax, var = data.draw(V.variants(tax, queries))
    taxon, strategy = data.draw(st.sampled_from(V.CONFIGS))
    custom = V.custom_cutoffs(data.draw) if taxon == "custom" else None
    if _three_ways(tax, _text([(qid, rows) for qid, rows, _k, _c in var]), taxon, strategy, custom=custom) is None:
        # a query that aborts hides the results of the others: then one query at a time
        for qid, rows, _k, _c in var:
            _three_ways(tax, _text([(qid, rows)]), taxon, strategy, custom=custom)


def test_variants_reach_every_class():
    """The variants of a two-row query whose top group has one row, and the class the dispatch rule gives each."""
    rows = [("A.1", 7, "99.5", 300, "850.3"), ("B.1", 7, "98", 300, "700")]
    assert V.expected_class(rows) == "narrow"
    assert V.lift(rows) == [("A.1", 7, "99.5", 300, "3000000850.3"), ("B.1", 7, "98", 300, "3000000700")]
    assert V.expected_class(V.lift(rows)) == "block"
    for size, cls in [(9, "warp32"), (32, "warp32"), (33, "block"), (1000, "block")]:
        for fresh in (False, True):
            g = V.grow(rows, size, fresh)
            assert V.expected_class(g) == cls and V.expected_class(V.lift(g)) == "block"
            top = [r for r in g if r[4] == "850.3"]
            assert len(top) == size and len({r[0] for r in top}) == (size if fresh else 1)
            assert g.count(rows[1]) == 1 and 0 < g.index(rows[1]) < size  # the lower row stays, among the top rows
            twins = [r[1] for r in V.grow(rows, size, fresh, twins=True)]
            assert twins.count(7 + V.TWIN) == size // 2 and twins.count(7) == size + 1 - size // 2
