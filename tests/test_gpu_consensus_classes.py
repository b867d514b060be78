"""The generated cases of tests/generators.py, rewritten by tests/consensus_variants.py, through all three
consensus implementations of the GPU: cons_compute<8> (top groups of 1..8 rows), cons_compute<32> (9..32 rows) and the
long-run kernel's long_consensus / consensus_single (more than 32 rows, or a bit score beyond int32).  Lineage maps with
non-Linnaean levels, rank names that occur twice at one level (fully tied beans), unequal depths; fungi, eukaryote and custom
cutoff tables with missing levels; both strategies.

Per case, the C++ oracle first runs every variant query alone in each of the eight configurations.  A query that aborts in any
of them leaves the batch (an aborted query would hide the results of the others); a few of them per class are run alone and
must fail the same way on the GPU.  The rest, all classes mixed in one table, runs once through the eight configurations in one
pass and once through the drawn configuration alone; every result equals the oracle's byte for byte.  The wrapper counts what
was compared per class and asserts floors afterwards, so that a generator that stops reaching a class fails loudly instead of
passing vacuously."""
import json
from collections import Counter

import pytest
from hypothesis import given, settings
from hypothesis import strategies as st

import consensus_variants as V
from generators import GPU, _text
from helpers import engine
from oracle_ffi import Oracle, OracleDataError

pytestmark = pytest.mark.gpu

PANICS_PER_CLASS = 3  # aborting queries per case and class that are run alone on the GPU

# Floors of the counts over the 150 derandomised cases: about half of what the draws and the C++ oracle give.  They depend on
# nothing the GPU computes (with the oracle standing in for the GPU, the counts were the ones in the comments).
COMPARED_FLOOR = {"narrow": 1300, "warp32": 1700, "block": 4800}  # (query, configuration) pairs compared byte for byte: 2600 / 3480 / 9560
PANIC_FLOOR = {"narrow": 400, "warp32": 100, "block": 530}  # (query, configuration) pairs that failed alone as the oracle does: 806 / 208 / 1070
TIED_FLOOR = {"warp32": 170, "block": 400}  # compared results with two fully tied beans: 352 / 800


@pytest.fixture(scope="module")
def fixed_engines():
    """One context per configuration with fixed cutoffs (the six of bacteria, fungi, eukaryotes); every case loads its own
    taxonomy into them."""
    engines = {(taxon, strategy): engine(taxon, strategy) for taxon, strategy in V.CONFIGS if taxon != "custom"}
    yield engines
    for e in engines.values():
        e.close()


def has_tied_beans(line: bytes) -> bool:
    """Two beans of one result with equal identifier and occurrences: an order the rank names alone decide."""
    beans = json.loads(line)["taxon"]["consensusBeans"] or []
    keys = [(b["identifier"], b["occurrences"]) for b in beans]
    return len(set(keys)) < len(keys)


def plan(tax, var, custom):
    """The oracle's side of a case: (the batch [(qid, rows, class)], its JSONL per configuration, the aborting queries to
    run alone [(qid, rows, class, [configurations where the oracle aborts])])."""
    ids = list(tax)
    lin = [tax[i] for i in ids]
    oracles = [Oracle(ids, lin, taxon, strategy, custom if taxon == "custom" else None, threads=1) for taxon, strategy in V.CONFIGS]
    batch, panics, per_class = [], [], Counter()
    for qid, rows, _kind, cls in var:
        text = _text([(qid, rows)])
        aborts = []
        for k, orc in enumerate(oracles):
            try:
                orc.run_raw(text)
            except OracleDataError:
                aborts.append(k)
        if not aborts:
            batch.append((qid, rows, cls))
        elif per_class[cls] < PANICS_PER_CLASS:
            per_class[cls] += 1
            panics.append((qid, rows, cls, aborts))
    want = None
    if batch:
        text = _text([(qid, rows) for qid, rows, _c in batch])
        want = [orc.run_raw(text)[0] for orc in oracles]
    for orc in oracles:
        orc.close()
    return batch, want, panics


def _engines_for(fixed, tax, custom):
    ids = list(tax)
    lin = [tax[i] for i in ids]
    engines, own = [], []
    for taxon, strategy in V.CONFIGS:
        if taxon == "custom":
            eng = engine(taxon, strategy, custom=custom)
            own.append(eng)
        else:
            eng = fixed[(taxon, strategy)]
        eng.load_taxonomy_arrays(ids, lin)
        engines.append(eng)
    return engines, own


def test_generated_variants_through_every_consensus_class(fixed_engines):
    from blutils_b200 import ConsensusPanic, run_host_configs

    compared, panicked, tied = Counter(), Counter(), Counter()

    @settings(**GPU)
    @given(st.data())
    def case(data):
        tax = data.draw(V.lineage_maps())
        tax, var = data.draw(V.variants(tax, data.draw(V.tables(tax))))
        custom = V.custom_cutoffs(data.draw)
        drawn = data.draw(st.integers(0, len(V.CONFIGS) - 1))
        batch, want, panics = plan(tax, var, custom)
        engines, own = _engines_for(fixed_engines, tax, custom)
        try:
            # aborting queries, alone: the GPU fails the configurations the oracle fails
            for qid, rows, cls, aborts in panics:
                for k in aborts:
                    with pytest.raises(ConsensusPanic):
                        engines[k].run_host(_text([(qid, rows)]))
                    panicked[cls] += 1
            if not batch:
                return
            text = _text([(qid, rows) for qid, rows, _c in batch])
            deferred = sum(cls == "block" for _q, _r, cls in batch)
            outs = run_host_configs(engines, text)
            assert int(engines[0].timings()["n_deferred_runs"]) >= deferred  # the long-run kernel took every block-class query
            got = [o.jsonl() for o in outs]
            for o in outs:
                o.close()
            classes = {qid: cls for qid, _r, cls in batch}
            for k, (g, w) in enumerate(zip(got, want)):
                assert g == w, f"configuration {V.CONFIGS[k]}"
                for line in g.splitlines():
                    cls = classes[json.loads(line)["query"]]
                    compared[cls] += 1
                    tied[cls] += has_tied_beans(line)
            single = engines[drawn].run_host(text)
            assert int(engines[drawn].timings()["n_deferred_runs"]) >= deferred
            assert single.jsonl() == want[drawn], f"configuration {V.CONFIGS[drawn]} alone"
            single.close()
        finally:
            for e in own:
                e.close()

    case()
    for cls in V.CLASSES:
        assert compared[cls] >= COMPARED_FLOOR[cls], (cls, compared)
        assert panicked[cls] >= PANIC_FLOOR[cls], (cls, panicked)
    for cls, floor in TIED_FLOOR.items():
        assert tied[cls] >= floor, (cls, tied)
