"""Several configurations in one pass (blu_consensus_run_*_configs): the table is parsed once and every context gets the
result its own single run gives -- compared with that run and with the CPU oracle -- and the timings of every context
report the one shared pass.

Launch counts per range / chunk of a pass with K > 1 configurations: the tile kernel and the fan-out kernel once, the
long-run, consensus (and gather) kernels and the advance per configuration, the duplicate-id check once -- or, with text
references, per configuration (the others relocate their references into the caller's text)."""
import ctypes as C
import random

import pytest

from helpers import random_blast, random_taxonomy
from test_gpu_file_stream import IDS, LIN, _row, _table

pytestmark = pytest.mark.gpu

YAML16S = {"domain": 50, "kingdom": 60, "phylum": 75, "class": 80, "order": 85, "family": 92, "genus": 97, "species": 99}
STRICT = {k: 96 for k in YAML16S}  # an identity below 96 % misses every cutoff
COUNTERS_BYTES = 120
CHUNK = 1 << 20


def _ct(d):
    from blutils_b200 import CustomTaxon

    return CustomTaxon(domain=d["domain"], kingdom=d["kingdom"], phylum=d["phylum"], class_=d["class"], order=d["order"], family=d["family"],
                       genus=d["genus"], species=d["species"])


def _engine(ids, lin, taxon, strategy, custom=None, numeric=False, chunk_bytes=0, text_refs=False):
    from blutils_b200 import ConsensusEngine, ConsensusStrategy, Taxon

    eng = ConsensusEngine({"bacteria": Taxon.Bacteria, "custom": Taxon.Custom}[taxon],
                          {"cautious": ConsensusStrategy.Cautious, "relaxed": ConsensusStrategy.Relaxed}[strategy], numeric,
                          _ct(custom) if custom else None, chunk_bytes=chunk_bytes, text_refs=text_refs)
    eng.load_taxonomy_arrays(ids, lin)
    return eng


class Group:
    """Contexts (engines) of one group with the oracle of each."""

    def __init__(self, specs, chunk_bytes=0, text_refs=False):
        from oracle_ffi import Oracle

        self.engines, self.oracles = [], []
        for ids, lin, taxon, strategy, custom, numeric in specs:
            self.engines.append(_engine(ids, lin, taxon, strategy, custom, numeric, chunk_bytes, text_refs))
            self.oracles.append(Oracle(ids, lin, taxon, strategy, custom))

    def close(self):
        for e in self.engines:
            e.close()


def _knobs(chunk_bytes=0, seed=20261020):
    """cautious / relaxed x bacteria / custom 16S cutoffs x text / numeric lineages: the eight configurations of one table."""
    from blutils_b200.synth import SynthWorkload

    w = SynthWorkload(3000, seed=seed)
    lins = {}
    for numeric in (False, True):
        ids, off, blob = w.lineages(numeric=numeric)
        lins[numeric] = (ids.tolist(), [bytes(blob[int(off[i]):int(off[i + 1])]).decode() for i in range(len(ids))])
    specs = [(*lins[numeric], taxon, strategy, YAML16S if taxon == "custom" else None, numeric)
             for numeric in (False, True) for taxon in ("bacteria", "custom") for strategy in ("cautious", "relaxed")]
    return w, Group(specs, chunk_bytes)


def _small_specs(custom=YAML16S):
    return [(IDS, LIN, "bacteria", "cautious", None, False), (IDS, LIN, "bacteria", "relaxed", None, False),
            (IDS, LIN, "custom", "cautious", custom, False), (IDS, LIN, "custom", "relaxed", custom, False)]


def _to_device(text):
    import torch

    n = len(text)
    t = torch.zeros((n + 255) // 128 * 128, dtype=torch.uint8, device="cuda")
    t[:n] = torch.frombuffer(bytearray(text), dtype=torch.uint8).cuda()
    torch.cuda.synchronize()
    return t


def _stream():
    import torch

    return torch.cuda.current_stream().cuda_stream


def _run(kind, engines, text, tmp_path, dev=None):
    """The group's results through `kind`, downloaded."""
    from blutils_b200 import run_device_resident_configs, run_file_configs, run_host_configs

    if kind == "host":
        return run_host_configs(engines, text)
    if kind == "file":
        path = tmp_path / "blast.out"
        path.write_bytes(text)
        return run_file_configs(engines, str(path))
    t = _to_device(text) if dev is None else dev
    outs = run_device_resident_configs(engines, t.data_ptr(), len(text), _stream())
    for o in outs:
        o.download()
    return outs


def _single(kind, eng, text, tmp_path):
    if kind == "host":
        return eng.run_host(text)
    if kind == "file":
        path = tmp_path / "single.out"
        path.write_bytes(text)
        return eng.run_file(str(path))
    t = _to_device(text)
    return eng.run_device_resident(t.data_ptr(), len(text), _stream()).download()


def _check_group(g, outs, text, tmp_path, kind):
    assert len(outs) == len(g.engines)
    for k, (eng, orc, out) in enumerate(zip(g.engines, g.oracles, outs)):
        want, nq, nr = orc.run_raw(text)
        got = out.jsonl()
        assert got == want, f"configuration {k}"
        assert len(out) == nq and out.n_rows == nr
        single = _single(kind, eng, text, tmp_path)
        assert single.jsonl() == got and single.checksum() == out.checksum() and len(single) == len(out), f"configuration {k}"
        single.close()


@pytest.mark.parametrize("kind", ["host", "file", "resident"])
def test_all_four_knobs_in_one_group(tmp_path, kind):
    w, g = _knobs()
    text = w.hits(0, 4000, 50)
    outs = _run(kind, g.engines, text, tmp_path)
    _check_group(g, outs, text, tmp_path, kind)
    g.close()


def _size_classes():
    """Top groups of 1..8, 9..32, 33..8192 rows and bit scores beyond int32 in one table: the long-run kernel has work
    in every configuration."""
    rows = []
    sizes = [1, 2, 5, 8, 9, 17, 32, 33, 120, 1500, 8192]
    for q, g in enumerate(sizes * 3):
        bits = "950" if q % 2 else "3000000000"
        for h in range(g + 3):
            top = h < g
            rows.append(_row(f"sz_{q:03d}", f"NR_{(q * 7 + h) % 500:06d}.1", IDS[(q + h) % 4] if q % 3 else IDS[h % 2],
                             f"{90 + h % 10}.{(q + h) % 1000:03d}", 300 + h % 50, bits if top else str(100 + h % 300)))
    return "".join(rows).encode()


@pytest.mark.parametrize("kind", ["host", "resident"])
def test_every_top_group_size_class(tmp_path, kind):
    g = Group(_small_specs())
    text = _size_classes()
    outs = _run(kind, g.engines, text, tmp_path)
    _check_group(g, outs, text, tmp_path, kind)
    assert int(g.engines[0].timings()["n_deferred_runs"]) > 0
    g.close()


def _tiny_rows():
    rows = []
    for q in range(120000):
        for h in range(1 + (q % 5 == 0)):
            rows.append(f"q{q}\tA\t{IDS[q % 2]}\t9{h}\t{1 + q % 9}\t0\t0\t1\t1\t1\t1\t0\t{5 + (q + h) % 3}\n")
    return "".join(rows).encode()


@pytest.mark.parametrize("kind", ["host", "file", "resident"])
def test_capacity_retry_on_fresh_contexts(tmp_path, kind):
    """More queries than a fresh context's first estimate: the whole pass runs again with grown capacities."""
    text = _tiny_rows()
    g = Group(_small_specs(), chunk_bytes=CHUNK)
    outs = _run(kind, g.engines, text, tmp_path)
    for k, (orc, out) in enumerate(zip(g.oracles, outs)):
        assert len(out) == 120000 and out.jsonl() == orc.run_raw(text)[0], f"configuration {k}"
    g.close()


def _scattered():
    rng = random.Random(77)
    units = random_taxonomy(rng, n_leaves=40)
    text = random_blast(rng, units, n_queries=400, max_hits=12, contiguous=False)
    ids = [u["taxid"] for u in units]
    specs = [(ids, [u["numericLineage" if numeric else "textLineage"] for u in units], taxon, strategy, YAML16S if taxon == "custom" else None,
              numeric) for numeric in (False, True) for taxon, strategy in (("bacteria", "cautious"), ("custom", "relaxed"))]
    return text, specs


@pytest.mark.parametrize("kind", ["host", "file", "resident"])
def test_scattered_table_is_regrouped_once(tmp_path, kind):
    text, specs = _scattered()
    g = Group(specs)
    outs = _run(kind, g.engines, text, tmp_path)
    for eng in g.engines:
        assert int(eng.timings()["n_regrouped"]) == 2
    _check_group(g, outs, text, tmp_path, kind)
    g.close()


def test_scattered_resident_results_share_the_regrouped_text(tmp_path):
    from blutils_b200 import run_device_resident_configs

    text, specs = _scattered()
    g = Group(specs)
    t = _to_device(text)
    outs = run_device_resident_configs(g.engines, t.data_ptr(), len(text), _stream())
    texts = {o.device_text() for o in outs}
    assert len(texts) == 1
    ptr, n = texts.pop()
    assert ptr != t.data_ptr() and n == len(text)
    for o in outs[:-1]:  # the last result keeps the regrouped copy alive
        o.close()
    last = outs[-1]
    assert last.device_text() == (ptr, n)
    assert last.download().jsonl() == g.oracles[-1].run_raw(text)[0]
    g.close()


def test_text_references_point_into_the_callers_text():
    from blutils_b200 import _ffi, run_host_configs

    text = _table(900, 0, seed=3)
    buf = C.create_string_buffer(text, len(text))
    g = Group(_small_specs(), chunk_bytes=CHUNK, text_refs=True)
    outs = run_host_configs(g.engines, C.addressof(buf), len(text))
    chunks = (len(text) + CHUNK - 1) // CHUNK
    K = len(outs)
    for orc, out in zip(g.oracles, outs):
        n = C.c_uint64()
        assert _ffi.lib().blu_result_pool(out._h, C.byref(n)) == C.addressof(buf) and n.value == len(text)
        assert out.jsonl() == orc.run_raw(text)[0]
        ids = out.query_ids()
        assert len(ids) == 900 and all(i.startswith(b"query_") for i in ids)
    t = g.engines[0].timings()
    assert int(t["n_kernel_launches"]) == chunks * (1 + 1 + 2 * K + K + K)
    g.close()


def test_grammar_error_fails_the_call(tmp_path):
    from blutils_b200 import ConsensusPanic, run_file_configs, run_host_configs

    text = _table(50, 0, seed=5) + b"broken\trow\n" + _table(5, 0, seed=6)
    g = Group(_small_specs())
    with pytest.raises(ConsensusPanic) as single:
        g.engines[2].run_host(text)
    with pytest.raises(ConsensusPanic) as grouped:
        run_host_configs(g.engines, text)
    assert str(grouped.value) == str(single.value)
    path = tmp_path / "bad.out"
    path.write_bytes(text)
    with pytest.raises(ConsensusPanic):
        run_file_configs(g.engines, str(path))
    g.close()


@pytest.mark.parametrize("kind", ["host", "file", "resident"])
def test_consensus_error_of_one_configuration_names_it(tmp_path, kind):
    """Under the STRICT cutoffs a single match of 95.5 % identity misses every cutoff (an empty adjusted taxonomy), under the
    bacteria ones it does not; every other query is above 96 %.  The call fails with the error of the lowest failing context."""
    from blutils_b200 import ConsensusPanic
    from oracle_ffi import OracleDataError

    text = (_row("qa", "NR_1.1", IDS[0], "95.5", 300, "900") +
            "".join(_row(f"q{q}", f"NR_{q}.{h}", IDS[(q + h) % 4], f"9{7 + h % 3}.5", 300, str(900 - h)) for q in range(30) for h in range(4))).encode()
    g = Group([(IDS, LIN, "bacteria", "relaxed", None, False), (IDS, LIN, "custom", "cautious", STRICT, False),
               (IDS, LIN, "custom", "relaxed", STRICT, False)])
    assert g.oracles[0].run_raw(text)[1] == 31
    for orc in g.oracles[1:]:
        with pytest.raises(OracleDataError):
            orc.run_raw(text)
    with pytest.raises(ConsensusPanic) as single:
        _single(kind, g.engines[1], text, tmp_path)
    with pytest.raises(ConsensusPanic) as grouped:
        _run(kind, g.engines, text, tmp_path)
    assert str(grouped.value) == "ctxs[1]: " + str(single.value)
    for eng in g.engines:
        assert eng_error(eng) == str(grouped.value)
    g.close()


def eng_error(eng):
    from blutils_b200 import _ffi

    return (_ffi.lib().blu_last_error(eng._h) or b"").decode()


def test_bad_groups_are_refused():
    from blutils_b200 import ConsensusEngine, ConsensusStrategy, Taxon, _ffi, run_host_configs

    text = _table(20, 0, seed=4)
    a = _engine(IDS, LIN, "bacteria", "relaxed")
    b = _engine(IDS, LIN, "bacteria", "cautious")
    other_chunk = _engine(IDS, LIN, "bacteria", "cautious", chunk_bytes=CHUNK)
    other_flags = _engine(IDS, LIN, "bacteria", "cautious", text_refs=True)
    no_tax = ConsensusEngine(Taxon.Bacteria, ConsensusStrategy.Relaxed, False, None)
    multi = ConsensusEngine(Taxon.Bacteria, ConsensusStrategy.Relaxed, False, None, devices=[0])
    multi.load_taxonomy_arrays(IDS, LIN)
    cases = [([a, a], "ctxs[1]: the same context as ctxs[0]"), ([a, multi], "ctxs[1]: a multi-device context"),
             ([a, no_tax], "ctxs[1]: no taxonomy loaded"), ([a, other_chunk], "ctxs[1]: chunk_bytes differs"),
             ([a, other_flags], "ctxs[1]: flags differ"), ([a, b] * 4 + [a], "a group holds 1 to 8 contexts")]
    for engines, msg in cases:
        with pytest.raises(RuntimeError, match=r"blu error 4: " + msg.replace("[", r"\[").replace("]", r"\]")):
            run_host_configs(engines, text)
    lib = _ffi.lib()
    outs = (C.c_void_p * 2)()
    buf = C.create_string_buffer(text, len(text))
    assert lib.blu_consensus_run_host_configs((C.c_void_p * 2)(a._h, None), 2, C.addressof(buf), len(text), outs) == _ffi.BLU_ERR_ARG
    assert lib.blu_consensus_run_host_configs((C.c_void_p * 2)(a._h, b._h), 0, C.addressof(buf), len(text), outs) == _ffi.BLU_ERR_ARG
    assert lib.blu_consensus_run_host_configs((C.c_void_p * 2)(a._h, b._h), 2, None, len(text), outs) == _ffi.BLU_ERR_ARG
    assert eng_error(a) == eng_error(b) == "null argument"
    # one context is the single entry point itself, multi-device context included
    (one,) = run_host_configs([multi], text)
    assert one.jsonl() == multi.run_host(text).jsonl()
    for e in (a, b, other_chunk, other_flags, no_tax, multi):
        e.close()


@pytest.mark.parametrize("kind", ["host", "file"])
def test_the_pass_is_shared(tmp_path, kind):
    """Host text and files cross PCIe once: the group copies and tiles what one single run does."""
    text = _table(900, 0, seed=3)
    chunks = (len(text) + CHUNK - 1) // CHUNK
    assert chunks > 2
    g = Group(_small_specs(), chunk_bytes=CHUNK)
    single = _single(kind, g.engines[1], text, tmp_path)
    st = g.engines[1].timings()
    outs = _run(kind, g.engines, text, tmp_path)
    K = len(outs)
    d2h = sum(int(e.timings()["result_bytes"]) for e in g.engines)
    for eng, out in zip(g.engines, outs):
        t = eng.timings()
        assert int(t["h2d_bytes"]) == int(st["h2d_bytes"]) == len(text)
        assert int(t["n_tile_launches"]) == int(st["n_tile_launches"]) == chunks
        assert int(t["text_bytes"]) == len(text)
        assert int(t["n_kernel_launches"]) == chunks * (1 + 1 + 3 * K + 1 + K)
        assert int(t["n_queries"]) == 900
        assert int(t["d2h_bytes"]) >= d2h + K * COUNTERS_BYTES
    assert outs[1].checksum() == single.checksum()
    g.close()


def test_resident_timings():
    text = _table(900, 0, seed=3)
    g = Group(_small_specs())
    t = _to_device(text)
    from blutils_b200 import run_device_resident_configs

    outs = run_device_resident_configs(g.engines, t.data_ptr(), len(text), _stream())
    K = len(outs)
    for eng in g.engines:
        tm = eng.timings()
        assert int(tm["n_tile_launches"]) == 1 and int(tm["h2d_bytes"]) == 0
        assert int(tm["n_kernel_launches"]) == 1 + 1 + 2 * K + 1 + K
        assert int(tm["d2h_bytes"]) == K * COUNTERS_BYTES
    g.close()


def test_sort_and_headers_as_for_single_runs(tmp_path):
    from blutils_b200 import run_device_resident_configs

    w, g = _knobs(seed=11)
    text = w.hits(0, 3000, 20)
    t = _to_device(text)
    outs = run_device_resident_configs(g.engines, t.data_ptr(), len(text), _stream())
    headers = [f"absent_{i}" for i in range(5)]
    for k, (eng, orc, out) in enumerate(zip(g.engines, g.oracles, outs)):
        out.sort_by_query().download()
        single = eng.run_device_resident(t.data_ptr(), len(text), _stream()).sort_by_query().download()
        assert out.query_ids() == single.query_ids() == sorted(single.query_ids()), f"configuration {k}"
        out.add_headers(headers)
        single.add_headers(headers)
        assert out.jsonl() == single.jsonl() == orc.run_raw(text, headers=headers)[0]
        a, b = tmp_path / f"g{k}.json", tmp_path / f"s{k}.json"
        out.write(str(a), run_id="r")
        single.write(str(b), run_id="r")
        assert a.read_bytes() == b.read_bytes()
        single.close()
    # a result is sorted with its own context only
    from blutils_b200 import _ffi

    other = run_device_resident_configs(g.engines[:2], t.data_ptr(), len(text), _stream())
    assert _ffi.lib().blu_result_sort_by_query(g.engines[0]._h, other[1]._h) == _ffi.BLU_ERR_ARG
    assert _ffi.lib().blu_result_sort_by_query(g.engines[1]._h, other[1]._h) == 0
    for o in other:
        o.close()
    g.close()
