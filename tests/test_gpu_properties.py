"""The generated cases of tests/generators.py through the CUDA path (C ABI): lineage maps with non-Linnaean levels,
unequal lengths, rank names that occur twice and fully tied beans; hit groups that tie on the truncated bit score; custom cutoff
tables; rows with odd fields.  Derandomised: every run draws the same cases.

These cases have top groups of 1..4 rows nearly always, so they reach the 8-lane consensus only; the same cases rewritten into
top groups of 9..1000 rows and bit scores beyond int32 (the 32-lane and the block-parallel consensus) are in
tests/test_gpu_consensus_classes.py."""
import pytest
from hypothesis import given, settings
from hypothesis import strategies as st

import generators as P
from generators import GPU
from helpers import engine
from oracle_ffi import Oracle, OracleDataError

pytestmark = pytest.mark.gpu


def _gpu_equals_oracle(tax, text, taxon, strategy, custom=None, loud_limits=False):
    from blutils_b200 import ConsensusPanic, Unsupported

    ids = list(tax)
    lin = [tax[i] for i in ids]
    try:
        want = Oracle(ids, lin, taxon, strategy, custom, threads=2).run_raw(text)[0]
    except OracleDataError:
        want = None
    eng = engine(taxon, strategy, False, custom)
    try:
        eng.load_taxonomy_arrays(ids, lin)
        try:
            got = eng.run_host(text).jsonl()
        except ConsensusPanic:
            got = None
        except Unsupported:
            if loud_limits and want is not None:
                return  # a documented loud limit (DESIGN.md section 5), never a different result
            raise
        assert got == want
    finally:
        eng.close()


@settings(**GPU)
@given(st.data())
def test_generated_lineages_and_hit_groups(data):
    tax = data.draw(P.lineage_maps())
    queries = data.draw(P.tables(tax))
    taxon = data.draw(st.sampled_from(["bacteria", "fungi", "eukaryotes", "custom"]))
    custom = None
    if taxon == "custom":
        custom = {"domain": data.draw(st.integers(0, 100)), "species": data.draw(st.integers(0, 100))}
        for k in ["kingdom", "phylum", "class", "order", "family", "genus"]:
            custom[k] = data.draw(st.one_of(st.none(), st.integers(0, 100)))
    _gpu_equals_oracle(tax, P._text(queries), taxon, data.draw(st.sampled_from(["cautious", "relaxed"])), custom)


@settings(**GPU)
@given(st.data())
def test_generated_rows_with_odd_fields(data):
    tax = {7: "d__bac;p__p1;c__c1", 12: "d__bac;p__p1;c__c2", 1500: "d__bac;p__p2"}
    text = data.draw(P.grammar_rows(sorted(tax)))
    _gpu_equals_oracle(tax, text, "bacteria", data.draw(st.sampled_from(["cautious", "relaxed"])), loud_limits=True)
