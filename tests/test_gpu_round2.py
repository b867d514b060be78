"""Round-2 GPU parity tests: device-resident results, text references, the block-parallel long-tail consensus,
top groups of every size class, consensus-class errors on reused contexts and on scattered tables."""
import json
import random

import pytest

from helpers import current_stream, engine, hit_row, random_blast, random_taxonomy, scattered_table, synth_case, to_device
from oracle_ffi import Oracle

pytestmark = pytest.mark.gpu

@pytest.mark.parametrize("n_queries,hits,zipf", [(300, 50, False), (6000, 50, False), (400, 5000, True)])
def test_device_resident_result(n_queries, hits, zipf):
    """Text in HBM -> records in HBM (no download, strings stay references into the device text); downloaded afterwards
    the result is the one of the host path.  Twice on the same context: the result arrays are recycled."""
    ids, lin, text = synth_case(5000, n_queries, hits, zipf, seed=13)
    want, nq, nr = Oracle(ids, lin, "bacteria", "relaxed").run_raw(text)
    eng = engine("bacteria", "relaxed", lineages=(ids, lin))
    t = to_device(text)
    stream = current_stream()
    for _ in range(2):
        out = eng.run_device_resident(t.data_ptr(), len(text), stream)
        assert len(out) == nq and out.n_rows == nr
        rec_ptr, beans_ptr, nb, accs_ptr, na = out.device_arrays()
        assert rec_ptr and beans_ptr and accs_ptr and nb >= nq and na >= nb
        assert int(eng.timings()["d2h_bytes"]) < 1024  # nothing but the counters crossed PCIe
        assert out.download().jsonl() == want
        assert out.jsonl(head=37) == b"".join(want.splitlines(keepends=True)[:37])  # (what bench.py's in-run check reads)
        assert out.jsonl(head=10 ** 9) == want
        out.close()
    # the download variant of the same call
    assert eng.run_device(t.data_ptr(), len(text), stream).jsonl() == want
    eng.close()


@pytest.mark.parametrize("chunk", [0, 1 << 20])
def test_text_refs_equal_pool(chunk):
    """BLU_OPT_TEXT_REFS: the result's strings are references into the caller's text (nothing is gathered or downloaded
    but records / beans / 8-byte accession references); same result, fewer bytes."""
    ids, lin, text = synth_case(5000, 5000, 50, seed=19)
    want = Oracle(ids, lin, "bacteria", "cautious").run_raw(text)[0]
    d2h = {}
    for refs in (False, True):
        eng = engine("bacteria", "cautious", chunk_bytes=chunk, text_refs=refs, lineages=(ids, lin))
        out = eng.run_host(text)
        assert out.jsonl() == want
        d2h[refs] = int(eng.timings()["d2h_bytes"])
        out.close()
        eng.close()
    assert d2h[True] < d2h[False]


def _group_rows(q, n, ids, rng, n_acc=50, bits="700"):
    rows = []
    for i in range(n):
        pid = rng.choice(["99.5", "99.50", "98.123", "100.000", "97", "99.999"])
        rows.append(hit_row(q, f"AC{rng.randrange(n_acc):04d}.{rng.randint(1, 2)}", rng.choice(ids), pid, rng.choice([400, 401, 1500]), bits))
    return rows


@pytest.mark.parametrize("sizes", [(2, 3, 8, 9, 16, 31, 32), (33, 64, 100), (1024, 1025), (3000,), (5000, 8192)])
def test_top_groups_of_every_size(sizes):
    """Top bit-score groups of 2..8 rows (four queries per warp), 9..32 (one warp), 33..8192 (block-parallel sort / fold in the
    long-run kernel; BASELINE C4 allows 5000 hits per query): lineages of unequal length, ties on every sort key, repeated
    accessions (Vec::dedup), many distinct beans."""
    rng = random.Random(sum(sizes))
    lin = ["d__bac;p__p1;c__c1;o__o1;f__f1;g__g1;s__s1", "d__bac;p__p1;c__c1;o__o1;f__f1;g__g1;s__s2", "d__bac;p__p1;c__c1;o__o1;f__f1;g__g2",
           "d__bac;clade__x;p__p2;c__c2;o__o2;f__f2;g__g3;species group__sg;s__s3;strain__st1", "d__bac;p__p1;c__c1;o__o1;f__f9",
           "d__bac;p__p1;c__c1;o__o1;f__f1;g__g1;s__s1;strain__a", "d__bac;p__p1;c__c1;o__o1;f__f1;g__g1;s__s1;strain__b"]
    lin += [f"d__bac;p__p1;c__c1;o__o1;f__f1;g__g1;s__sx{i}" for i in range(40)]
    ids = list(range(11, 11 + len(lin)))
    rows = []
    for k, n in enumerate(sizes):
        pool = ids if k % 3 == 0 else (ids[:2] + ids[5:7] if k % 3 == 1 else ids[:1])
        rows += _group_rows(f"big{k}_{n}", n, pool, rng, n_acc=max(3, n // 7))
        rows += [hit_row(f"big{k}_{n}", "LOW.1", ids[2], "80.0", 400, "100")] * 3
        rows += _group_rows(f"small{k}", rng.randint(1, 8), ids[:3], rng)
    text = "".join(rows).encode()
    for strategy in ("cautious", "relaxed"):
        want = Oracle(ids, lin, "bacteria", strategy).run_raw(text)[0]
        eng = engine("bacteria", strategy, lineages=(ids, lin))
        assert eng.run_host(text).jsonl() == want, strategy
        eng.close()


def test_top_group_beyond_the_cap_is_loud():
    from blutils_b200 import Unsupported

    lin = ["d__bac;p__p1"]
    rows = [hit_row("q", f"A{i}.1", 1, "99.0", 100, "500") for i in range(8193)]
    eng = engine("bacteria", "cautious", lineages=([1], lin))
    with pytest.raises(Unsupported):
        eng.run_host("".join(rows).encode())
    eng.close()


def test_mixed_group_sizes_random():
    """Random tables whose top groups fall into all three size classes inside the same warps / CTAs."""
    rng = random.Random(4242)
    units = random_taxonomy(rng, n_leaves=60)
    ids = [u["taxid"] for u in units]
    lin = [u["textLineage"] for u in units]
    from oracle_ffi import OracleDataError

    done = 0
    for rep in range(6):
        text = random_blast(rng, units, n_queries=300, max_hits=45, tie_rate=0.9)
        for strategy in ("cautious", "relaxed"):
            try:
                want = Oracle(ids, lin, "bacteria", strategy).run_raw(text)[0]
            except OracleDataError:
                continue
            eng = engine("bacteria", strategy, lineages=(ids, lin))
            assert eng.run_host(text).jsonl() == want
            eng.close()
            done += 1
    assert done >= 4


def test_consensus_errors_on_a_reused_context():
    """Root-level disagreement and an empty adjusted taxonomy (reference panics) after a successful run on the same
    context, and after a run that had to grow its output arrays: a data error every time, never a capacity loop."""
    from blutils_b200 import ConsensusPanic

    lin = ["d__bac;p__p1;c__c1", "d__arc;p__p9;c__c9", "d__bac;p__p1;c__c2"]
    ids = [1, 2, 3]
    good = "".join(hit_row(f"q{i}", "A.1", 1 + 2 * (i % 2), "99.0", 100, "500") for i in range(200)).encode()
    root = (good.decode() + hit_row("qr", "A.1", 1, "99.0", 100, "500") + hit_row("qr", "B.1", 2, "99.0", 100, "500")).encode()
    empty = (good.decode() + hit_row("qe", "A.1", 1, "10.0", 100, "500")).encode()
    many = "".join(hit_row(f"m{i}", f"A{i}.1", 1, "99.0", 100, "500") for i in range(60000)).encode()  # tiny rows: the arrays must grow
    eng = engine("bacteria", "cautious", lineages=(ids, lin))
    want = Oracle(ids, lin, "bacteria", "cautious").run_raw(good)[0]
    for bad in (root, empty):
        assert eng.run_host(good).jsonl() == want
        with pytest.raises(ConsensusPanic):
            eng.run_host(bad)
    assert len(eng.run_host(many)) == 60000
    for bad in (root, empty):
        with pytest.raises(ConsensusPanic):
            eng.run_host(bad)
        assert eng.run_host(good).jsonl() == want
    eng.close()


def test_scattered_query_with_a_failing_fragment():
    """The reference groups rows by a HashMap (mod.rs:145,192) and only parses the taxonomy of the TOP group's rows: a
    low-score fragment of a scattered query may carry an unmapped taxid / disagree at the root without the merged query
    failing.  The fragment's error must not abort the run before the table is known to be scattered."""
    lin = ["d__bac;p__p1;c__c1", "d__arc;p__p9;c__c9"]
    ids = [1, 2]
    rows = [hit_row("qA", "A.1", 1, "99.0", 100, "100"), hit_row("qB", "B.1", 1, "98.0", 100, "90"), hit_row("qA", "A2.1", 999, "97.0", 100, "50"),
            hit_row("qC", "C.1", 1, "98.0", 100, "90"), hit_row("qA", "A3.1", 2, "97.0", 100, "50"), hit_row("qA", "A4.1", 1, "97.0", 100, "50")]
    text = "".join(rows).encode()
    want = Oracle(ids, lin, "bacteria", "cautious").run_raw(text)[0]
    eng = engine("bacteria", "cautious", lineages=(ids, lin))
    out = eng.run_host(text)
    assert out.jsonl() == want
    assert int(eng.timings()["n_regrouped"]) == 2  # regrouped on the GPU
    eng.close()


@pytest.mark.parametrize("group", [3, 20, 32])
def test_windows_full_of_top_rows(group):
    """Every row of every query ties on the top bit score: each 32 KB window holds several hundred top rows, far more than
    the tile kernel's shared-memory queue of top rows to parse -- runs that do not fit parse their rows in place, the
    others are parsed one window later (or at the end of the CTA's segment), and queries span window boundaries."""
    rng = random.Random(77 + group)
    n_taxa = 40
    ids = list(range(1, n_taxa + 1))
    lin = [f"d__bac;p__p{t % 3};c__c{t % 7};o__o{t % 11};f__f{t % 13};g__g{t % 17};s__s{t}" for t in ids]
    rows = []
    for q in range(4000):
        t0 = rng.randrange(n_taxa)
        for h in range(group):
            t = ids[(t0 + (h % 3 if rng.random() < 0.5 else 0)) % n_taxa]
            rows.append(hit_row(f"q{q:05d}", f"ACC{q}_{h}.1", t, f"{90 + (h * 7 + q) % 10}.{(q + h) % 100:02d}", 200 + h, "640"))
    text = "".join(rows).encode()
    want = Oracle(ids, lin, "bacteria", "relaxed").run_raw(text)[0]
    eng = engine("bacteria", "relaxed", lineages=(ids, lin))
    assert eng.run_host(text).jsonl() == want
    eng.close()


@pytest.mark.parametrize("where", ["gpu", "host"])
@pytest.mark.parametrize("shape", ["plain", "blank_lines", "no_final_newline", "big"])
def test_scattered_tables_regrouped(where, shape, monkeypatch):
    """Non-contiguous tables (the reference's HashMap grouping, mod.rs:145,192) through both regrouping paths: on the GPU
    (blu_regroup.cu: row index, id hash table with byte-exact check, stable radix sort, copy) and on the host; host text,
    device text and a file; against the oracle, which groups the way the reference does."""
    if where == "host":
        monkeypatch.setenv("BLU_REGROUP_HOST", "1")
    else:
        monkeypatch.delenv("BLU_REGROUP_HOST", raising=False)
    rng = random.Random(len(shape) * 31 + 5)
    ids, lin, text = scattered_table(rng, 60_000 if shape == "big" else 700, 9, 60, blank_lines=shape == "blank_lines",
                                      final_newline=shape != "no_final_newline")
    want = Oracle(ids, lin, "bacteria", "relaxed").run_raw(text)[0]
    eng = engine("bacteria", "relaxed", lineages=(ids, lin))
    code = 2 if where == "gpu" else 1
    out = eng.run_host(text)
    assert out.jsonl() == want
    assert int(eng.timings()["n_regrouped"]) == code
    out.close()
    t = to_device(text)
    out = eng.run_device(t.data_ptr(), len(text), current_stream())
    assert out.jsonl() == want
    assert int(eng.timings()["n_regrouped"]) == code
    out.close()
    # a contiguous table afterwards on the same context: nothing is regrouped
    ids2, lin2, text2 = synth_case(5000, 300, 20, seed=3)
    eng2 = engine("bacteria", "relaxed", lineages=(ids2, lin2))
    eng2.run_host(text2).close()
    assert int(eng2.timings()["n_regrouped"]) == 0
    eng2.close()
    eng.close()


def test_scattered_table_from_a_file(tmp_path):
    rng = random.Random(99)
    ids, lin, text = scattered_table(rng, 3000, 6, 40)
    want = Oracle(ids, lin, "bacteria", "cautious").run_raw(text)[0]
    path = tmp_path / "scattered.blast.out"
    path.write_bytes(text)
    eng = engine("bacteria", "cautious", lineages=(ids, lin))
    out = eng.run_file(str(path))
    assert out.jsonl() == want
    assert int(eng.timings()["n_regrouped"]) == 2
    out.close()
    eng.close()


def test_scattered_table_device_resident():
    """A non-contiguous table through the device-resident entry point: regrouped in HBM, the records stay on the device and
    reference the regrouped copy (blu_result_device_text), which the result owns; downloaded afterwards it is the oracle's
    result.  The caller's text may be released as soon as the call has returned."""
    import torch

    rng = random.Random(4711)
    ids, lin, text = scattered_table(rng, 5000, 8, 50)
    want = Oracle(ids, lin, "bacteria", "relaxed").run_raw(text)[0]
    eng = engine("bacteria", "relaxed", lineages=(ids, lin))
    t = to_device(text)
    out = eng.run_device_resident(t.data_ptr(), len(text), current_stream())
    assert int(eng.timings()["n_regrouped"]) == 2
    ptr, n = out.device_text()
    assert ptr and ptr != t.data_ptr() and n >= len(text)  # (every row newline-terminated; nothing else changes)
    t.zero_()  # the result must not depend on the caller's text any more
    torch.cuda.synchronize()
    assert out.download().jsonl() == want
    out.close()
    # contiguous table: the references point into the caller's text
    ids2, lin2, text2 = synth_case(5000, 300, 20, seed=3)
    eng2 = engine("bacteria", "relaxed", lineages=(ids2, lin2))
    t2 = to_device(text2)
    out2 = eng2.run_device_resident(t2.data_ptr(), len(text2), current_stream())
    assert out2.device_text() == (t2.data_ptr(), len(text2))
    out2.close()
    eng2.close()
    eng.close()


@pytest.mark.parametrize("group", [2, 7, 20, 40])
def test_fully_tied_beans(group):
    """Two beans with the same identifier and the same number of occurrences under different rank names tie completely in
    the reference's bean sort (build_blast_consensus_identity.rs:50-60), which leaves them in HashMap order.  Every
    implementation here breaks the tie by the order in which the beans' keys first appear in the taxonomy map -- in the
    8-lane, the 32-lane and the block-parallel consensus alike, and whichever way round the map lists them."""
    lineages = {1: "d__bac;clade__x0;k__k0;p__p1", 2: "d__bac;species group__x0;k__k0;p__p2", 3: "d__bac;no rank__x0;k__k1", 4: "d__bac;k__k0"}
    rows = []
    for q in range(50):
        for h in range(group):
            rows.append(hit_row(f"q{q:03d}", f"A{q}_{h}.1", 1 + (h + q) % 3, "91.5", 300, "700"))
        rows.append(hit_row(f"q{q:03d}", f"L{q}.1", 4, "80.0", 300, "100"))
    text = "".join(rows).encode()
    for order in ([1, 2, 3, 4], [3, 2, 1, 4], [2, 4, 3, 1]):
        ids = order
        lin = [lineages[i] for i in order]
        for strategy in ("cautious", "relaxed"):
            want = Oracle(ids, lin, "bacteria", strategy).run_raw(text)[0]
            eng = engine("bacteria", strategy, lineages=(ids, lin))
            assert eng.run_host(text).jsonl() == want, (order, strategy)
            eng.close()
    first = [json.loads(l)["taxon"]["consensusBeans"][0]["rank"] for l in want.decode().splitlines()[:1]]
    assert first  # (the beans really are listed)
