"""The result writers (blu_decode.h, blu_tabular.h) on the CPU, through the host-compiled path (tests/csrc/sim_harness.cpp):
every format, to a file, to stdout and to a pipe, byte for byte against the oracle (pyoracle.to_json_pretty / to_json_compact /
results_to_jsonl / results_to_yaml / results_to_tabular).  The tables reach what the small hypothesis cases do not: hit-less
headers, a maxAllowedRank whose rank is not in the cutoff backbone (printed by its display name), results in two parts or
already in query order, and ~20 000 queries, enough for ordered_parallel_write's threads (pwrite to a regular file, the in-order
writer to a pipe).  A metamorphic check closes the loop: build-tabular of the written JSON or YAML is the TSV written straight
from the records."""
import os
import random
import re
import threading

import pytest

import pyoracle as po
import sim_ffi
from helpers import random_blast, random_taxonomy

RUN_ID = "0b0e3c55-7a2f-4a61-9d4e-5f1c2a7b8c9d"
FORMATS = ["json", "jsonl", "yaml", "tsv"]
LAYOUTS = {"one-part": dict(), "two-parts": dict(two_parts=True), "sorted-two-parts": dict(sorted_records=True, two_parts=True)}


def _table(seed, n_queries, max_hits):
    rng = random.Random(seed)
    units = random_taxonomy(rng, n_leaves=40)
    # a kingdom under every domain: a default rank the bacteria backbone does not have, so a maxAllowedRank there is "k"
    tax = {u["taxid"]: re.sub(r"(d__dom\d+)", r"\1;k__kng", u["textLineage"]) for u in units}
    text = random_blast(rng, units, n_queries=n_queries, max_hits=max_hits, low_pident=60.0)
    present = sorted({line.split("\t", 1)[0] for line in text.decode().splitlines()})
    # hit-less headers that sort before, between and after the ids, and a few ids that do have hits (those are not repeated)
    headers = ["A0", "zz_last", "q00000a", "SRR1.1_size_3 "] + [f"nohit_{i}" for i in range(n_queries // 10)] + present[::max(1, len(present) // 5)]
    rng.shuffle(headers)
    res = po.build_consensus_identities(text, tax, "bacteria", "relaxed", headers=headers)
    assert any(r["taxon"] and r["taxon"]["maxAllowedRank"] == "k" for r in res)
    assert any(r["taxon"] is None for r in res)
    return dict(ids=list(tax), lin=list(tax.values()), text=text, headers=headers, res=res)


@pytest.fixture(scope="module", params=[(20261021, 300, 12), (1, 20_000, 3)], ids=["300-queries", "20000-queries"])
def table(request):
    return _table(*request.param)


def _expected(res, fmt, to_stdout):
    if fmt == "json":
        doc = {"results": [dict([("runId", RUN_ID)] + list(r.items())) for r in res], "config": None}
        return po.to_json_compact(doc) if to_stdout else po.to_json_pretty(doc)
    if fmt == "jsonl":
        return "null\n" + po.results_to_jsonl(res, RUN_ID)  # (the config line, write_blutils_output.rs:165-175)
    if fmt == "yaml":
        return po.results_to_yaml(res, RUN_ID)
    return po.results_to_tabular(res, RUN_ID, to_stdout=to_stdout)


def _write(t, path, fmt, **layout):
    rc = sim_ffi.run_write(t["ids"], t["lin"], "bacteria", "relaxed", t["text"], path, fmt, RUN_ID, headers=t["headers"], **layout)
    assert rc == 0, (fmt, path, rc)


def _stdout_through_pipe(fn):
    """Runs fn with fd 1 on a pipe (drained by a thread); returns what it wrote."""
    r, w = os.pipe()
    chunks = []
    reader = threading.Thread(target=lambda: chunks.extend(iter(lambda: os.read(r, 1 << 16), b"")))
    reader.start()
    saved = os.dup(1)
    try:
        os.dup2(w, 1)
        os.close(w)
        fn()
    finally:
        os.dup2(saved, 1)
        os.close(saved)
        reader.join()
        os.close(r)
    return b"".join(chunks)


@pytest.mark.parametrize("layout", list(LAYOUTS))
@pytest.mark.parametrize("fmt", FORMATS)
def test_every_writer_like_the_oracle(table, fmt, layout, tmp_path, capfd):
    """To a file (pretty JSON), to stdout on a regular file (capfd) and to stdout on a pipe (compact JSON, TSV with a line
    break after every piece)."""
    _write(table, str(tmp_path / "out.txt"), fmt, **LAYOUTS[layout])  # the extension is forced to the format's
    assert (tmp_path / f"out.{fmt}").read_bytes().decode("utf-8") == _expected(table["res"], fmt, False)
    want = _expected(table["res"], fmt, True)
    capfd.readouterr()
    _write(table, None, fmt, **LAYOUTS[layout])
    assert capfd.readouterr().out == want
    assert _stdout_through_pipe(lambda: _write(table, None, fmt, **LAYOUTS[layout])).decode("utf-8") == want


def test_build_tabular_of_the_written_result(table, tmp_path, capfd):
    """Writing a result as JSON or YAML and running build-tabular on the file gives the TSV written straight from the records,
    to a file and to stdout."""
    from blutils_b200 import OutputFormat, parse_consensus_as_tabular

    _write(table, str(tmp_path / "direct"), "tsv", two_parts=True)
    _write(table, str(tmp_path / "res"), "json", two_parts=True)
    _write(table, str(tmp_path / "res"), "yaml", two_parts=True)
    direct = (tmp_path / "direct.tsv").read_bytes()
    for src, fmt in (("res.json", OutputFormat.Json), ("res.yaml", OutputFormat.Yaml)):
        parse_consensus_as_tabular(str(tmp_path / src), str(tmp_path / "via.tsv"), fmt)
        assert (tmp_path / "via.tsv").read_bytes() == direct, src
    capfd.readouterr()
    _write(table, None, "json", two_parts=True)
    (tmp_path / "compact.json").write_bytes(capfd.readouterr().out.encode("utf-8"))
    _write(table, None, "tsv", two_parts=True)
    direct = capfd.readouterr().out
    parse_consensus_as_tabular(str(tmp_path / "compact.json"), None, OutputFormat.Json)
    assert capfd.readouterr().out == direct
