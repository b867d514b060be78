"""Property tests (hypothesis; SURVEY section 4) over generated lineage maps and hit groups, on the CPU:

* three implementations of the path agree byte for byte on the canonical JSONL -- and on WHICH inputs are data errors:
  oracle/pyoracle.py, oracle/blu_oracle.cpp and the product's device core compiled for the host (tests/csrc/sim_harness.cpp:
  the same parse / top-group / consensus / cutoff functions the CUDA kernels call);
* metamorphic properties the domain offers (build_consensus_identities/mod.rs:104-128 is an order-free per-query map, and only the
  top bit-score group of a query is ever looked at, find_single_query_consensus.rs:17-173):
    - the result of a query depends on its own rows only: queries can be reordered, tables can be cut at query boundaries and the
      pieces' results concatenated;
    - rows below the query's top bit score can be dropped, duplicated, permuted or given any mapped / unmapped taxid;
    - a consensus taxonomy consists of levels of one of the top group's lineages, in order, from the root, cut in front of the first level -- among those every top lineage has -- at which two top rows
      name different taxa, and a single-row top group is a single match.
"""
import json

import pytest
from hypothesis import HealthCheck, given, settings
from hypothesis import strategies as st

import pyoracle as po
import sim_ffi
from generators import _text, _three_ways, grammar_rows, lineage_maps, tables

def _by_query(jsonl: bytes):
    return {json.loads(line)["query"]: line for line in jsonl.decode().splitlines()}


# Derandomised by default (the suite draws the same cases on every run); BLU_HYP_RANDOM=1 explores new ones (optionally with
# --hypothesis-seed=N and BLU_HYP_EXAMPLES=N), which is how the properties were exercised while they were written.
COMMON = dict(max_examples=int(__import__("os").environ.get("BLU_HYP_EXAMPLES", "120")), derandomize=not __import__("os").environ.get("BLU_HYP_RANDOM"),
              database=None, deadline=None, suppress_health_check=[HealthCheck.too_slow, HealthCheck.data_too_large])


@settings(**COMMON)
@given(st.data())
def test_three_implementations_agree(data):
    tax = data.draw(lineage_maps())
    queries = data.draw(tables(tax))
    taxon = data.draw(st.sampled_from(["bacteria", "fungi", "eukaryotes", "custom"]))
    strategy = data.draw(st.sampled_from(["cautious", "relaxed"]))
    custom = None
    if taxon == "custom":  # CustomTaxon (taxon.rs:14-65): domain and species required, the others optional
        custom = {"domain": data.draw(st.integers(0, 100)), "species": data.draw(st.integers(0, 100))}
        for k in ["kingdom", "phylum", "class", "order", "family", "genus"]:
            custom[k] = data.draw(st.one_of(st.none(), st.integers(0, 100)))
    # ParallelBlastOutput.headers (mod.rs:84-102): ids without hits become NoConsensusFound; ids with hits change nothing
    headers = None
    if data.draw(st.booleans()):
        headers = data.draw(st.lists(st.one_of(st.sampled_from([q for q, _ in queries]), st.sampled_from(["nohit_1", "nohit 2", "é"])), max_size=5, unique=True))
    _three_ways(tax, _text(queries), taxon, strategy, custom=custom, headers=headers or None)


@settings(**COMMON)
@given(st.data())
def test_a_query_depends_on_its_own_rows_only(data):
    tax = data.draw(lineage_maps())
    queries = data.draw(tables(tax))
    strategy = data.draw(st.sampled_from(["cautious", "relaxed"]))
    whole = _three_ways(tax, _text(queries), "bacteria", strategy)
    if whole is None:
        return
    whole_q = _by_query(whole)
    # any order of the queries; any cut at a query boundary, results concatenated (SURVEY 8e: shard invariance)
    perm = data.draw(st.permutations(queries))
    assert _by_query(_three_ways(tax, _text(perm), "bacteria", strategy)) == whole_q
    cut = data.draw(st.integers(0, len(queries)))
    pieces = {}
    for part in (queries[:cut], queries[cut:]):
        if part:
            pieces.update(_by_query(_three_ways(tax, _text(part), "bacteria", strategy)))
    assert pieces == whole_q


@settings(**COMMON)
@given(st.data())
def test_only_the_top_bit_score_group_matters(data):
    tax = data.draw(lineage_maps())
    queries = data.draw(tables(tax))
    strategy = data.draw(st.sampled_from(["cautious", "relaxed"]))
    whole = _three_ways(tax, _text(queries), "bacteria", strategy)
    if whole is None:
        return
    changed = []
    for qid, rows in queries:
        top = max(int(float(r[4])) for r in rows)  # (the reference compares the TRUNCATED bit score, mod.rs:162,184)
        keep, low = [r for r in rows if int(float(r[4])) == top], [r for r in rows if int(float(r[4])) != top]
        mode = data.draw(st.sampled_from(["drop", "double", "permute", "unmapped"]))
        if mode == "drop":
            low = []
        elif mode == "double":
            low = low + low
        elif mode == "permute":
            low = list(data.draw(st.permutations(low)))
        else:
            low = [(a, 999_999, p, ln, b) for a, _t, p, ln, b in low]  # not in the map: only top-group rows are ever joined
        # rows below the top score may sit anywhere among the top rows, whose own order stays
        merged, ki, li = [], 0, 0
        while ki < len(keep) or li < len(low):
            take_low = li < len(low) and (ki >= len(keep) or data.draw(st.booleans()))
            if take_low:
                merged.append(low[li]); li += 1
            else:
                merged.append(keep[ki]); ki += 1
        changed.append((qid, merged))
    assert _by_query(_three_ways(tax, _text(changed), "bacteria", strategy)) == _by_query(whole)


@settings(**COMMON)
@given(st.data())
def test_shape_of_a_consensus(data):
    tax = data.draw(lineage_maps())
    queries = data.draw(tables(tax))
    strategy = data.draw(st.sampled_from(["cautious", "relaxed"]))
    out = _three_ways(tax, _text(queries), "bacteria", strategy)
    if out is None:
        return
    res = {json.loads(line)["query"]: json.loads(line) for line in out.decode().splitlines()}
    assert sorted(res) == sorted(q for q, _ in queries)
    for qid, rows in queries:
        t = res[qid]["taxon"]
        assert t is not None
        top = max(int(float(r[4])) for r in rows)
        group = [r for r in rows if int(float(r[4])) == top]
        assert t["bitScore"] == float(top)
        assert t["singleMatch"] == (len(group) == 1)
        lineages = [tax[r[1]].replace("species group", "species-group").replace("no rank", "no-rank").split(";") for r in group]  # (ranks are slugified)
        if t["taxonomy"] != "":  # ("" when the identity is below every cutoff: nothing of the lineage is kept)
            got = t["taxonomy"].split(";")
            # the levels of one of the top group's lineages, in order, that pass the identity filter (linnaean_ranks.rs:194-212
            # filters level by level: a level can be dropped between two kept ones when a rank name occurs twice in a lineage)
            def subsequence(a, l):
                it = iter(l)
                return all(x in it for x in a)
            assert any(subsequence(got, l) and got[0] == l[0] for l in lineages), (got, lineages)
        got = t["taxonomy"].split(";") if t["taxonomy"] else []
        if len(group) > 1:
            # Levels are compared only as deep as the SHORTEST top lineage reaches (find_multi_taxa_consensus.rs:137-214: a
            # take_while over the length-ascending list ends at the first lineage that has ended).  A disagreement inside that
            # range bounds the consensus; without one the reference lineage is kept as far as the identity allows.
            shortest = min(len(l) for l in lineages)
            i0 = next((i for i in range(shortest) if len({l[i] for l in lineages}) > 1), None)
            if i0 is not None:
                assert len(got) <= i0, (got, lineages)
            beans = t["consensusBeans"]
            assert beans is not None and sum(b["occurrences"] for b in beans) <= len(group)
            keys = [(-b["occurrences"], b["identifier"]) for b in beans]
            assert keys == sorted(keys)  # folded beans: occurrences descending, then identifier (consensus_result.rs:60-89)


# ---- the input grammar: every implementation accepts and rejects the same rows -----------------------------------------------
@settings(**COMMON)
@given(st.data())
def test_the_input_grammar_three_ways(data):
    """Rows with clean and with odd fields (number shapes, empty fields, non-ASCII, quotes, field counts, CRLF, blank lines, no final
    newline): the two oracles and the product's parsers (the lean mask parser with the full grammar behind it, compiled for the
    host) accept the same tables, reject the same tables, and give the same results."""
    tax = {7: "d__bac;p__p1;c__c1", 12: "d__bac;p__p1;c__c2", 1500: "d__bac;p__p2"}
    text = data.draw(grammar_rows(sorted(tax)))
    _three_ways(tax, text, "bacteria", data.draw(st.sampled_from(["cautious", "relaxed"])), loud_limits=True)


# ---- a9: the cutoff interpolation, the only floating-point arithmetic of the path -----------------------------------------------
RANK_NAMES = ["d", "domain", "k", "kingdom", "p", "c", "class", "o", "order", "f", "g", "genus", "s", "species", "u", "clade", "species group", "species-group",
              "strain", "no rank", "subspecies", "Subspecies", "superkingdom", "Forma  specialis", "serotype", " genus ", "GENUS", "x"]


@settings(**COMMON)
@given(st.lists(st.sampled_from(RANK_NAMES), min_size=1, max_size=24), st.sampled_from(["bacteria", "fungi", "eukaryotes", "custom"]),
       st.lists(st.one_of(st.none(), st.integers(0, 100)), min_size=6, max_size=6), st.integers(0, 100), st.integers(0, 100))
def test_cutoff_interpolation_matches_the_oracle(names, taxon, optional6, dom, spe):
    """Rank vectors of any shape -- repeated names, ranks out of order, non-Linnaean names first / last / in runs, the NaN and
    infinity cases of a zero-width window -- through the product's interpolate_cutoffs (host, f64), the C++ oracle and the Python
    restatement of InterpolatedIdentity::interpolate_identities (linnaean_ranks.rs:220-383): bit-identical f64 values."""
    import math

    custom = None
    if taxon == "custom":  # domain and species are required (taxon.rs:14-65), the six between them optional
        keys = ["kingdom", "phylum", "class", "order", "family", "genus"]
        custom = dict({"domain": dom, "species": spe}, **dict(zip(keys, optional6)))
    want = po.interpolate([po.rank_from_str(n) for n in names], po.backbone_for(taxon, custom))
    from oracle_ffi import interpolate as cpp_oracle_interpolate

    for got in (sim_ffi.interpolate(names, taxon, custom), cpp_oracle_interpolate(names, taxon, custom)):
        assert len(got) == len(want)
        for g, w in zip(got, want):
            assert (math.isnan(g) and math.isnan(w)) or (g == w and math.copysign(1.0, g) == math.copysign(1.0, w)), (names, taxon, custom, got, want)


# ---- the writers: JSON / JSONL / YAML / TSV bytes of tables whose strings need escaping ------------------------------------------
ODD = st.text(alphabet=st.sampled_from(list("abZ09 _-.;:#'\"\\/|&*!%@`?[]{},>~=") + ["é", "ß", "漢", "\U0001d518", " ", " ", "﻿", "\x7f", "\x01", "\x1b"]),
              min_size=1, max_size=10)
LOOKS_LIKE = st.sampled_from(["null", "~", "true", "False", "yes", "NO", "on", "0x1F", "0o17", "1e3", "-.inf", ".NaN", "007", "12", "-3", "+4", "1.5", "- x", "a: b", "x #y",
                              " lead", "trail ", "---", "...", "? k", ": v", "[a]", "{b}", "&a", "*a", "!t", "|", ">", "%", "@", "`"])


@settings(**COMMON)
@given(st.data())
def test_the_writers_escape_like_the_oracle(tmp_path_factory, data):
    """Query ids and accessions made of quotes, backslashes, control characters, non-ASCII and astral characters, YAML indicators and
    things that read as null / booleans / numbers: the product's pretty JSON, JSONL, YAML (serde_yaml 0.9 quoting) and build-tabular
    TSV writers against the oracle's, byte for byte, on a table that goes through the whole host-compiled path."""
    tax = {7: "d__bac;p__p1;c__c1", 12: "d__bac;p__p1;c__c2"}
    ids = list(tax)
    lin = [tax[i] for i in ids]
    word = st.one_of(ODD, LOOKS_LIKE).filter(lambda w: "\t" not in w and "\n" not in w and "\r" not in w and '"' not in w)
    n_q = data.draw(st.integers(1, 4))
    qids = data.draw(st.lists(word, min_size=n_q, max_size=n_q, unique=True))
    rows = []
    for q in qids:
        for h in range(data.draw(st.integers(1, 3))):
            rows.append(f"{q}\t{data.draw(word)}\t{data.draw(st.sampled_from(ids))}\t{data.draw(st.sampled_from(['97.5', '100', '88.125']))}\t300\t0\t0\t1\t300\t1\t300\t1e-50\t640\n")
    text = "".join(rows).encode("utf-8")
    try:
        res = po.build_consensus_identities(text, tax, "bacteria", "relaxed", None)
    except po.DataError:
        return  # (e.g. an id that is only blanks: the grammar property covers agreement on rejections)
    run_id = "0b0e3c55-7a2f-4a61-9d4e-5f1c2a7b8c9d"
    doc = {"results": [dict([("runId", run_id)] + list(r.items())) for r in res], "config": None}
    want = {"json": po.to_json_pretty(doc), "jsonl": "null\n" + po.results_to_jsonl(res, run_id),  # (the config line, write_blutils_output.rs:165-175)
            "yaml": po.results_to_yaml(res, run_id),
            "tsv": po.results_to_tabular(res, run_id, to_stdout=False)}
    d = tmp_path_factory.mktemp("w")
    for fmt, expected in want.items():
        path = str(d / ("out." + ("tsv" if fmt == "tsv" else fmt)))
        rc = sim_ffi.run_write(ids, lin, "bacteria", "relaxed", text, path, fmt, run_id)
        assert rc == 0, (fmt, rc)
        got = open(path, "rb").read().decode("utf-8")
        assert got == expected, (fmt, qids)


# ---- a3: the `.blutils.json` reader (hand-written pull parser) against Python's json ---------------------------------------------
JSON_TEXT = st.text(alphabet=st.one_of(st.sampled_from(list("ab;_ -\"\\/\b\f\n\r\t{}[]:,") + ["é", "漢", "\U0001d518", "\x00", "\x1f", "\x7f", "퟿", "", "￿"]),
                                       st.characters(blacklist_categories=("Cs",))), max_size=12)
JUNK = st.recursive(st.one_of(st.none(), st.booleans(), st.integers(-10 ** 20, 10 ** 20), st.floats(allow_nan=False, allow_infinity=False), JSON_TEXT),
                    lambda c: st.one_of(st.lists(c, max_size=3), st.dictionaries(JSON_TEXT, c, max_size=3)), max_leaves=8)


@settings(**COMMON)
@given(st.data())
def test_taxonomy_json_reader_matches_python_json(tmp_path_factory, data):
    """Schema-conforming `.blutils.json` documents (taxonomies_map.rs:6-32) with arbitrary strings -- every escape json.dumps can
    produce, raw UTF-8, astral characters, control characters --, unknown fields holding arbitrary JSON at every level, keys in
    any order, any whitespace: the product's reader (blu_taxonomy.cpp, the parser the GPU path's taxonomy comes through) yields
    the (taxid, lineage) pairs Python's json module reads from the same bytes."""
    import random as _random

    rnd = _random.Random(data.draw(st.integers(0, 2 ** 32)))

    def shuffled(d):
        items = list(d.items())
        rnd.shuffle(items)
        return dict(items)

    taxa = []
    for _ in range(data.draw(st.integers(0, 5))):
        t = {"taxid": data.draw(st.integers(0, 2 ** 53)), "rank": data.draw(JSON_TEXT), "numericLineage": data.draw(JSON_TEXT), "textLineage": data.draw(JSON_TEXT),
             "accessions": [shuffled(dict({"accession": data.draw(JSON_TEXT), "oid": data.draw(JSON_TEXT)}, **data.draw(st.dictionaries(st.sampled_from(["x", "y"]), JUNK, max_size=1))))
                            for _ in range(data.draw(st.integers(0, 2)))]}
        if data.draw(st.booleans()):
            t["futureField"] = data.draw(JUNK)
        taxa.append(shuffled(t))
    doc = {"blutilsVersion": data.draw(JSON_TEXT), "ignoreTaxids": data.draw(st.one_of(st.none(), st.lists(st.integers(0, 2 ** 40), max_size=3))),
           "replaceRank": data.draw(st.one_of(st.none(), st.dictionaries(JSON_TEXT, JSON_TEXT, max_size=2))), "dropNonLinnaeanTaxonomies": data.draw(st.one_of(st.none(), st.booleans())),
           "sourceDatabase": data.draw(JSON_TEXT), "taxonomies": taxa}
    if data.draw(st.booleans()):
        doc["somethingNew"] = data.draw(JUNK)
    doc = shuffled(doc)
    text = json.dumps(doc, ensure_ascii=data.draw(st.booleans()), indent=data.draw(st.sampled_from([None, 0, 2])),
                      separators=data.draw(st.sampled_from([None, (",", ":"), (" , ", " : ")])))
    path = str(tmp_path_factory.mktemp("j") / "t.blutils.json")
    with open(path, "w", encoding="utf-8") as fh:
        fh.write(text)
    back = json.loads(text)
    for use_taxid in (False, True):
        want = [(t["taxid"], t["numericLineage" if use_taxid else "textLineage"]) for t in back["taxonomies"]]
        if any("\x00" in lin for _, lin in want):
            continue  # (the harness hands strings over NUL-separated)
        assert sim_ffi.dump_taxonomy_json(path, use_taxid) == want
    # a required field missing anywhere is an error, as it is for serde (mod.rs:261: from_str::<TaxonomiesMap>)
    if taxa:
        victim = data.draw(st.sampled_from(["taxid", "rank", "numericLineage", "textLineage", "accessions"]))
        broken = json.loads(text)
        del broken["taxonomies"][data.draw(st.integers(0, len(taxa) - 1))][victim]
        with open(path, "w", encoding="utf-8") as fh:
            json.dump(broken, fh)
        with pytest.raises(IOError):
            sim_ffi.dump_taxonomy_json(path)
