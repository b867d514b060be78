"""Parity tests proper: the CUDA path (through the C ABI) against the CPU oracle, bit for bit on the canonical
JSONL (every field of every result, sorted by query, runId masked)."""
import ctypes as C
import os
import random

import pytest

from helpers import (CUTOFFS_16S, current_stream, engine, hit_row, random_blast, random_taxonomy, synth_case, to_device,
                     write_taxonomy)
from oracle_ffi import Oracle

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("seed", range(24))
def test_random_small(seed):
    from blutils_b200 import ConsensusPanic
    from oracle_ffi import OracleDataError

    rng = random.Random(1000 + seed)
    units = random_taxonomy(rng, n_leaves=rng.choice([5, 20, 60]), shared_root=rng.random() < 0.9)
    text = random_blast(rng, units, n_queries=rng.choice([1, 10, 60]), contiguous=True, low_pident=rng.choice([60.0, 45.0]))
    for taxon in ("bacteria", "fungi", "custom"):
        for strategy in ("cautious", "relaxed"):
            use_taxid = bool((seed + len(strategy)) & 1)
            custom = None
            if taxon == "custom":
                custom = CUTOFFS_16S if seed % 3 else {"domain": 50, "species": 99, "genus": 95}
            lin = [(u["numericLineage"] if use_taxid else u["textLineage"]) for u in units]
            ids = [u["taxid"] for u in units]
            try:
                want = Oracle(ids, lin, taxon, strategy, custom).run_raw(text)[0]
            except OracleDataError:
                want = None
            eng = engine(taxon, strategy, use_taxid, custom, lineages=(ids, lin))
            if want is None:
                with pytest.raises(ConsensusPanic):
                    eng.run_host(text)
            else:
                assert eng.run_host(text).jsonl() == want
            eng.close()


@pytest.mark.parametrize("n_queries,hits,zipf", [(300, 50, False), (4000, 50, False), (2000, 100, False), (600, 5000, True),
                                                 (40000, 1, False), (30000, 2, False), (3000, 200, False)])
def test_synth_vs_oracle(n_queries, hits, zipf):
    """Multi-tile inputs (0.1 - 30 MB): windows, ownership, look-ahead, long-run path (Zipf up to 5000 hits)."""
    ids, lin, text = synth_case(5000, n_queries, hits, zipf)
    for strategy in ("cautious", "relaxed"):
        want, nq, nr = Oracle(ids, lin, "bacteria", strategy).run_raw(text)
        eng = engine("bacteria", strategy, lineages=(ids, lin))
        out = eng.run_host(text)
        assert len(out) == nq and out.n_rows == nr
        assert out.jsonl() == want
        eng.close()


def test_device_resident_equals_host_and_streamed():
    """Same text through: host single chunk, host streamed in 1 MiB chunks (carry-over of the unfinished query),
    and device-resident (torch tensor)."""
    ids, lin, text = synth_case(5000, 6000, 50, seed=5)
    want = Oracle(ids, lin, "bacteria", "relaxed").run_raw(text)[0]
    eng = engine("bacteria", "relaxed", lineages=(ids, lin))
    assert eng.run_host(text).jsonl() == want
    t = to_device(text)
    out = eng.run_device(t.data_ptr(), len(text), current_stream())
    assert out.jsonl() == want
    assert out.checksum() == __import__("oracle_ffi").checksum_jsonl(want)
    eng.close()
    for chunk in (1 << 20, 3 << 20):
        eng2 = engine("bacteria", "relaxed", chunk_bytes=chunk, lineages=(ids, lin))
        assert eng2.run_host(text).jsonl() == want
        eng2.close()


def test_streamed_zipf_long_runs():
    ids, lin, text = synth_case(5000, 400, 5000, zipf=True, seed=9)
    want = Oracle(ids, lin, "bacteria", "cautious").run_raw(text)[0]
    eng = engine("bacteria", "cautious", chunk_bytes=2 << 20, lineages=(ids, lin))
    assert eng.run_host(text).jsonl() == want
    eng.close()


def test_big_top_group_and_edge_rows():
    """Top group of 40 and 700 rows (block path), no trailing newline, empty lines, fractional bit scores in one group."""
    lin = ["d__bac;p__p1;c__c1;o__o1;f__f1;g__g1;s__s1", "d__bac;p__p1;c__c1;o__o1;f__f1;g__g1;s__s2", "d__bac;p__p1;c__c1;o__o1;f__f1;g__g2",
           "d__bac;clade__x;p__p2;c__c2;o__o2;f__f2;g__g3;species group__sg;s__s3;strain__st1"]
    ids = [11, 12, 13, 14]
    rows = []
    for i in range(40):
        rows.append(hit_row("qA", f"ACC{i % 7}.1", ids[i % 2], "99.5", 400, "700"))
    rows.append(hit_row("qA", "LOW.1", 13, "80.0", 400, "100"))
    for i in range(700):
        rows.append(hit_row("qB", f"B{i % 50:03d}.1", ids[i % 3], f"{97 + (i % 3)}.{i % 10}", 300 + i % 2, "512.0" if i % 2 else "512.9"))
    rows.append("\n\n")
    rows.append(hit_row("qC", "C1.1", 14, "99.9", 1500, "84.2"))
    rows.append(hit_row("qC", "C2.1", 14, "98.1", 1500, "84.9"))
    rows.append(hit_row("qC", "C0.1", 13, "99.0", 1500, "83.99"))
    rows.append(hit_row("qD", "D1.1", 14, "100.000", 1500, "1.000e+03").rstrip("\n"))
    text = "".join(rows).encode()
    for strategy in ("cautious", "relaxed"):
        want = Oracle(ids, lin, "bacteria", strategy).run_raw(text)[0]
        eng = engine("bacteria", strategy, lineages=(ids, lin))
        assert eng.run_host(text).jsonl() == want
        eng.close()


@pytest.mark.parametrize("bad", [b"", b"q\tacc\t1\t99.0\t10\t0\t0\t1\t10\t1\t10\t0.0\n", b"q\tacc\tN/A\t99.0\t10\t0\t0\t1\t10\t1\t10\t0.0\t50\n",
                                 b"q\tacc\t1\t99.0\t10\t0\t0\t1\t10\t1\t10\t0.0\t50\textra\n", b"q\t\"acc\t1\t99.0\t10\t0\t0\t1\t10\t1\t10\t0.0\t50\n",
                                 b"q\tacc\t1\t99.0\t10\t0\t0\t1\t10\t1\t10\t0.0\t50\r\n", b"q\tacc\t1\t9x\t10\t0\t0\t1\t10\t1\t10\t0.0\t50\n",
                                 b"q\tacc\t2\t99.0\t10\t0\t0\t1\t10\t1\t10\t0.0\t50\n", b"\n\n",
                                 b"q\tacc\t1\t10.0\t10\t0\t0\t1\t10\t1\t10\t0.0\t50\n"])
def test_reference_abort_cases(bad):
    """Inputs on which the reference panics must yield an error, never a result."""
    from blutils_b200 import ConsensusPanic

    eng = engine("bacteria", "cautious")
    eng.load_taxonomy_arrays([1], ["d__a;p__b"])
    with pytest.raises(ConsensusPanic):
        eng.run_host(bad)
    eng.close()


@pytest.mark.parametrize("seed", range(6))
def test_noncontiguous_tables(seed):
    """Rows of one query scattered over the file (legal for the reference's HashMap grouping, mod.rs:145,192):
    detected on the GPU (dup_kernel), regrouped by query, then the normal path."""
    rng = random.Random(300 + seed)
    units = random_taxonomy(rng, n_leaves=30)
    text = random_blast(rng, units, n_queries=40, contiguous=False)
    lin = [u["textLineage"] for u in units]
    ids = [u["taxid"] for u in units]
    from oracle_ffi import OracleDataError

    try:
        want = Oracle(ids, lin, "fungi", "relaxed").run_raw(text)[0]
    except OracleDataError:
        pytest.skip("generated case hits a reference abort")
    eng = engine("fungi", "relaxed", lineages=(ids, lin))
    out = eng.run_host(text)
    assert out.jsonl() == want
    assert int(eng.timings()["n_regrouped"]) in (0, 2)
    eng.close()


def test_sharded_equals_whole():
    """SURVEY 8e: query-range shards (blu_shard_cuts) processed independently and concatenated == the whole table."""
    from blutils_b200 import shard_cuts

    ids, lin, text = synth_case(3000, 3000, 50, seed=21)
    eng = engine("bacteria", "cautious", lineages=(ids, lin))
    whole = eng.run_host(text).jsonl()
    for n in (2, 3, 8):
        cuts = shard_cuts(text, n)
        assert cuts[0] == 0 and cuts[-1] == len(text) and cuts == sorted(cuts)
        parts = []
        for a, b in zip(cuts[:-1], cuts[1:]):
            if b > a:
                parts += eng.run_host(text[a:b]).jsonl().decode().splitlines()
        assert "\n".join(sorted(parts, key=lambda l: l.encode())) + "\n" == whole.decode()
    eng.close()


def test_file_api_headers_and_writer(tmp_path):
    """build_consensus_identities(ParallelBlastOutput{output_file, headers}, tax_file, ...) + write_blutils_output."""
    import json

    import pyoracle as po
    from blutils_b200 import ConsensusStrategy, OutputFormat, ParallelBlastOutput, Taxon, build_consensus_identities, write_blutils_output

    rng = random.Random(77)
    units = random_taxonomy(rng, n_leaves=30)
    text = random_blast(rng, units, n_queries=25)
    tax_path = write_taxonomy(str(tmp_path / "db.blutils.json"), units)
    blast_path = tmp_path / "blast.out"
    blast_path.write_bytes(text)
    headers = ["zz_no_hit", "aa_no_hit"] + sorted({l.split(b"\t")[0].decode() for l in text.splitlines() if l})
    res = build_consensus_identities(ParallelBlastOutput(str(blast_path), headers), tax_path, Taxon.Bacteria, ConsensusStrategy.Relaxed, True)
    tax = po.load_taxonomy(tax_path, True)
    want = po.build_consensus_identities(text, tax, "bacteria", "relaxed", headers=headers)
    assert res.jsonl().decode() == po.results_to_jsonl(want)
    # writer: pretty JSON to a file (extension forced), JSONL with the leading `null` config line
    write_blutils_output(res, None, str(tmp_path / "out.txt"), OutputFormat.Json)
    got = (tmp_path / "out.json").read_text()
    doc = json.loads(got)
    run_id = doc["results"][0]["runId"]
    exp = {"results": [dict([("runId", run_id)] + list(r.items())) for r in want], "config": None}
    assert got == po.to_json_pretty(exp)
    # build-tabular straight from the records (parse_consensus_as_tabular), file mode keeps the reference's missing line breaks
    res.write_tabular(str(tmp_path / "tab.txt"), run_id)
    assert (tmp_path / "tab.tsv").read_text() == po.results_to_tabular(want, run_id, to_stdout=False)
    write_blutils_output(res, None, str(tmp_path / "out2"), OutputFormat.Jsonl)
    lines = (tmp_path / "out2.jsonl").read_text().splitlines()
    assert lines[0] == "null" and len(lines) == 1 + len(want)
    assert [json.loads(l)["query"] for l in lines[1:]] == [r["query"] for r in want]


def test_tile_and_window_edges():
    """Texts cut at every kind of position relative to the 48 KiB tile grid, with and without a trailing newline,
    with empty lines, through both the host path and tiny streaming chunks."""
    ids, lin, text = synth_case(2000, 2600, 50, seed=31)
    rows = text.split(b"\n")
    rows = [r for r in rows if r]
    orc = Oracle(ids, lin, "bacteria", "relaxed")
    eng = engine("bacteria", "relaxed", lineages=(ids, lin))
    eng_small = engine("bacteria", "relaxed", chunk_bytes=96 << 10, lineages=(ids, lin))
    # prefix lengths (in rows) that put the end of the text just before / at / after tile and window borders
    sizes = []
    acc = 0
    marks = [49152, 49152 + 10240, 2 * 49152, 3 * 49152 + 1024]
    for i, r in enumerate(rows):
        acc += len(r) + 1
        for m in marks:
            if abs(acc - m) <= 80:
                sizes.append(i + 1)
    sizes = sorted(set(sizes))[:12] + [1, 2, 51]
    for n in sizes:
        for tail in (b"\n", b"", b"\n\n\n"):
            t = b"\n".join(rows[:n]) + tail
            want = orc.run_raw(t)[0]
            assert eng.run_host(t).jsonl() == want, (n, tail)
            assert eng_small.run_host(t).jsonl() == want, (n, tail, "streamed")
    # empty lines sprinkled between rows
    t = b"\n\n".join(rows[:700]) + b"\n"
    want = orc.run_raw(t)[0]
    assert eng.run_host(t).jsonl() == want
    assert eng_small.run_host(t).jsonl() == want
    eng.close()
    eng_small.close()


def test_long_rows():
    """Rows whose first field is longer than the 1 KiB look-behind (predecessor not in the window -> block path),
    and a row longer than the whole window (documented limit: loud BLU_ERR_UNSUPPORTED)."""
    from blutils_b200 import Unsupported

    lin = ["d__bac;p__p1;c__c1;o__o1;f__f1;g__g1;s__s1", "d__bac;p__p1;c__c1;o__o1;f__f1;g__g1;s__s2"]
    ids = [11, 12]
    rows = []
    for q in range(120):
        name = f"q{q:04d}_" + "x" * (1500 if q % 3 == 0 else 20)
        for h in range(30):
            rows.append(hit_row(name, f"ACC{h % 5}.1", ids[(q + h) % 2], "99.5" if h < 3 else "90.1", 400, "700" if h < 3 else "300"))
    text = "".join(rows).encode()
    want = Oracle(ids, lin, "bacteria", "cautious").run_raw(text)[0]
    eng = engine("bacteria", "cautious", lineages=(ids, lin))
    assert eng.run_host(text).jsonl() == want
    big = (hit_row("q_small", "A.1", 11, "99.0", 10, "50") + hit_row("q" + "y" * 70000, "A.1", 11, "99.0", 10, "50")).encode()
    with pytest.raises(Unsupported):
        eng.run_host(big)
    eng.close()


def test_streamed_chunk_sizes_zipf():
    """Carry-over logic under stress: chunk sizes from 64 KiB up, long-tail (Zipf) queries of up to ~380 KB."""
    ids, lin, text = synth_case(3000, 250, 5000, zipf=True, seed=17)
    want = Oracle(ids, lin, "bacteria", "relaxed").run_raw(text)[0]
    for chunk in (512 << 10, 1 << 20, (1 << 20) + 4096 + 128):
        eng = engine("bacteria", "relaxed", chunk_bytes=chunk, lineages=(ids, lin))
        assert eng.run_host(text).jsonl() == want, chunk
        eng.close()
