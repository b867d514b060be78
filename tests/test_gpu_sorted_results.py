"""Results whose records are in query-id order (blu_result_sort_by_query): every producing path, adversarial ids, hit-less
headers, multi-device contexts and a large table.  A sorted result must list its record ids strictly increasing (bytewise),
keep every record's own beans and accessions, and give the unsorted result's checksum and writer bytes."""
import ctypes as C
import random

import numpy as np
import pytest

from test_gpu_multi import _device_sets, _multi
from test_gpu_parity import _engine, _oracle, _row
from test_gpu_round2 import _scattered_table, _to_device

pytestmark = pytest.mark.gpu

RUN_ID = "00000000-0000-4000-8000-000000000000"


def _writer_bytes(out, tmp_path, tag):
    from blutils_b200 import OutputFormat

    got = {"jsonl()": out.jsonl(), "checksum": out.checksum(), "len": len(out)}
    for fmt, ext in ((OutputFormat.Json, "json"), (OutputFormat.Jsonl, "jsonl"), (OutputFormat.Yaml, "yaml")):
        p = tmp_path / f"{tag}.{ext}"
        out.write(str(p), fmt, run_id=RUN_ID)
        got[ext] = p.read_bytes()
    p = tmp_path / f"{tag}.tsv"
    out.write_tabular(str(p), run_id=RUN_ID)
    got["tsv"] = p.read_bytes()
    return got


def _assert_strictly_increasing(ids):
    for a, b in zip(ids, ids[1:]):
        assert a < b, (a, b)


def _check(unsorted, sorted_, tmp_path):
    """`sorted_` went through sort_by_query, `unsorted` is the same table through the same path without it."""
    ids = sorted_.query_ids()
    assert len(ids) == len(sorted_.records())
    _assert_strictly_increasing(ids)
    assert sorted(unsorted.query_ids()) == ids
    want = _writer_bytes(unsorted, tmp_path, "unsorted")
    got = _writer_bytes(sorted_, tmp_path, "sorted")
    for k in want:
        assert got[k] == want[k], k
    # the records themselves are in the writer's order: the ids of the jsonl lines that carry a consensus, in line order
    import json

    lines = [json.loads(l) for l in got["jsonl()"].splitlines()]
    assert [d["query"].encode() for d in lines if d["taxon"] is not None] == [i for i in ids]


def _device_ids(out):
    """The query ids of a device-resident result, read from its device record array (before any download)."""
    import torch

    from blutils_b200 import _ffi

    n = _ffi.lib().blu_result_num_records(out._h)
    rec_ptr = out.device_arrays()[0]
    tptr, tn = out.device_text()

    class _Dev:
        def __init__(self, ptr, nbytes):
            self.__cuda_array_interface__ = {"shape": (nbytes,), "typestr": "|u1", "data": (ptr, False), "version": 3}

    recs = torch.as_tensor(_Dev(rec_ptr, n * 64), device="cuda").cpu().numpy()
    text = torch.as_tensor(_Dev(tptr, tn), device="cuda").cpu().numpy().tobytes()
    r = recs.view(np.uint64).reshape(n, 8)
    off = r[:, 0]
    ln = r[:, 1] & 0xFFFFFFFF
    return [text[int(o):int(o) + int(l)] for o, l in zip(off, ln)]


def _table(query_ids, seed=5):
    """A small table: every query gets 1-4 hits over a handful of lineages; file order = the order of `query_ids`."""
    rng = random.Random(seed)
    lin = ["d__bac;p__p1;c__c1;o__o1;f__f1;g__g1;s__s1", "d__bac;p__p1;c__c1;o__o1;f__f1;g__g1;s__s2", "d__bac;p__p1;c__c1;o__o1;f__f1;g__g2",
           "d__bac;p__p2;c__c2;o__o2;f__f2;g__g3;s__s3"]
    ids = [11, 12, 13, 14]
    rows = []
    for k, q in enumerate(query_ids):
        for h in range(rng.randint(1, 4)):
            rows.append(_row("\x00", f"ACC{k % 97}_{h}.1", ids[(k + h) % 4], f"{90 + (k + h) % 10}.5", 150, str(800 - 7 * h)).encode().replace(b"\x00", q))
    return ids, lin, b"".join(rows)


def _run_both(eng, run):
    return run(eng), run(eng).sort_by_query()


# --- 1. every producing path ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("text_refs", [False, True])
def test_run_host_sorted(text_refs, tmp_path):
    from blutils_b200 import ConsensusEngine, ConsensusStrategy, Taxon

    from test_gpu_parity import _synth_case

    ids, lin, text = _synth_case(5000, 4000, 30, seed=23)
    eng = ConsensusEngine(Taxon.Bacteria, ConsensusStrategy.Relaxed, False, None, text_refs=text_refs)
    eng.load_taxonomy_arrays(ids, lin)
    a, b = _run_both(eng, lambda e: e.run_host(text))
    _check(a, b, tmp_path)
    assert a.jsonl() == _oracle(ids, lin, "bacteria", "relaxed").run_raw(text)[0]


def test_run_file_and_device_sorted(tmp_path):
    import torch

    from test_gpu_parity import _synth_case

    ids, lin, text = _synth_case(5000, 6000, 20, seed=29)
    path = tmp_path / "t.blast.out"
    path.write_bytes(text)
    eng = _engine("bacteria", "cautious")
    eng.load_taxonomy_arrays(ids, lin)
    a, b = _run_both(eng, lambda e: e.run_file(str(path)))
    _check(a, b, tmp_path)
    t = _to_device(text)
    s = torch.cuda.current_stream().cuda_stream
    a, b = _run_both(eng, lambda e: e.run_device(t.data_ptr(), len(text), s))
    _check(a, b, tmp_path)


def test_device_resident_sorted_before_download(tmp_path):
    import torch

    from test_gpu_parity import _synth_case

    ids, lin, text = _synth_case(5000, 20000, 10, seed=31)
    eng = _engine("bacteria", "relaxed")
    eng.load_taxonomy_arrays(ids, lin)
    t = _to_device(text)
    s = torch.cuda.current_stream().cuda_stream
    a = eng.run_device_resident(t.data_ptr(), len(text), s).download()
    b = eng.run_device_resident(t.data_ptr(), len(text), s)
    b.sort_by_query()
    dev_ids = _device_ids(b)
    _assert_strictly_increasing(dev_ids)
    b.download()
    assert b.query_ids() == dev_ids
    _check(a, b, tmp_path)


def test_device_resident_needs_its_own_context():
    import torch

    from blutils_b200 import _ffi

    from test_gpu_parity import _synth_case

    ids, lin, text = _synth_case(500, 300, 5, seed=3)
    e1, e2 = _engine("bacteria", "relaxed"), _engine("bacteria", "relaxed")
    for e in (e1, e2):
        e.load_taxonomy_arrays(ids, lin)
    t = _to_device(text)
    out = e1.run_device_resident(t.data_ptr(), len(text), torch.cuda.current_stream().cuda_stream)
    assert _ffi.lib().blu_result_sort_by_query(e2._h, out._h) == _ffi.BLU_ERR_ARG
    out.sort_by_query()
    _assert_strictly_increasing(_device_ids(out))


# --- 2. adversarial ids ----------------------------------------------------------------------------------------------
def _accepted_control_bytes():
    """The control bytes the input grammar accepts inside a query id, as the oracle decides."""
    from oracle_ffi import OracleDataError

    ok = []
    for c in list(range(0, 32)) + [127]:
        if c in (9, 10):
            continue
        ids, lin, text = _table([b"ctl" + bytes([c]) + b"x"])
        try:
            _oracle(ids, lin, "bacteria", "relaxed").run_raw(text)
        except OracleDataError:
            continue
        ok.append(c)
    return ok


def _adversarial_ids(rng):
    out = set()
    for plen in (7, 8, 9, 15, 16, 17, 40):
        p = bytes(rng.choice(b"ACGTNacgt:_-0123456789") for _ in range(plen))
        out.add(p)
        for suf in (b"a", b"b", b"ab", b"\x7f", b"\xc3\xa9", b"zzzzzzzzz", b"0", b"00000000", b"0000000000000000"):
            out.add(p + suf)
            out.add(p[:-1] + suf)
    # ids that are prefixes of one another, across chunk boundaries
    base = b"prefixchain-0123456789abcdefghijklmnopqrstuvwxyz"
    for i in range(1, len(base) + 1):
        out.add(base[:i])
    # multi-byte UTF-8 and bytes >= 0x80
    for s in ("é", "éa", "é", "日本", "日本語のリード", "\U0001f9ec", "Ωmega", "z", "ÿ", "ÿÿ"):
        out.add(s.encode())
    # lengths up to ~4 KB sharing long prefixes
    for n in (1, 2, 63, 64, 65, 1000, 4000, 4095):
        out.add(b"L" * n)
        out.add(b"L" * (n - 1) + b"M")
    return out


def test_adversarial_ids(tmp_path):
    rng = random.Random(77)
    ids_set = _adversarial_ids(rng)
    for c in _accepted_control_bytes():
        ids_set.add(b"ctl" + bytes([c]))
        ids_set.add(b"ctl" + bytes([c]) + b"tail")
        ids_set.add(b"ctlprefix" + bytes([c]) * 9)
    qids = sorted(ids_set)
    rng.shuffle(qids)
    ids, lin, text = _table(qids)
    want = _oracle(ids, lin, "bacteria", "relaxed").run_raw(text)[0]
    for refs in (False, True):
        from blutils_b200 import ConsensusEngine, ConsensusStrategy, Taxon

        eng = ConsensusEngine(Taxon.Bacteria, ConsensusStrategy.Relaxed, False, None, text_refs=refs)
        eng.load_taxonomy_arrays(ids, lin)
        a, b = _run_both(eng, lambda e: e.run_host(text))
        assert a.jsonl() == want
        assert b.query_ids() == sorted(qids)
        _check(a, b, tmp_path)


def test_single_query(tmp_path):
    ids, lin, text = _table([b"only-one"])
    eng = _engine("bacteria", "relaxed")
    eng.load_taxonomy_arrays(ids, lin)
    a, b = _run_both(eng, lambda e: e.run_host(text))
    assert b.query_ids() == [b"only-one"]
    _check(a, b, tmp_path)


def test_reverse_file_order(tmp_path):
    """10^5 queries whose file order is the reverse of their sorted order (shared prefixes of 8, 9 and 17 bytes)."""
    qids = sorted({b"%s%06d" % (p, i) for i in range(34000) for p in (b"SRR0000", b"SRR00001", b"M0001:12:000000000")})[:100_000]
    qids.reverse()
    ids, lin, text = _table(qids)
    eng = _engine("bacteria", "relaxed")
    eng.load_taxonomy_arrays(ids, lin)
    a, b = _run_both(eng, lambda e: e.run_host(text))
    assert b.query_ids() == qids[::-1]
    _check(a, b, tmp_path)


# --- 3. a scattered table, device-resident --------------------------------------------------------------------------
def test_scattered_table_device_resident_sorted(tmp_path):
    import torch

    rng = random.Random(4711)
    ids, lin, text = _scattered_table(rng, 5000, 8, 50)
    eng = _engine("bacteria", "relaxed")
    eng.load_taxonomy_arrays(ids, lin)
    t = _to_device(text)
    s = torch.cuda.current_stream().cuda_stream
    a = eng.run_host(text)
    b = eng.run_device_resident(t.data_ptr(), len(text), s)
    assert int(eng.timings()["n_regrouped"]) == 2
    assert b.device_text()[0] != t.data_ptr()
    b.sort_by_query()
    dev_ids = _device_ids(b)
    _assert_strictly_increasing(dev_ids)
    b.download()
    assert b.query_ids() == dev_ids
    _check(a, b, tmp_path)


# --- 4. hit-less headers ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("when", ["before", "after"])
def test_hitless_headers(when, tmp_path):
    qids = [b"read_%04d" % i for i in range(0, 2000, 2)]
    random.Random(8).shuffle(qids)
    ids, lin, text = _table(qids)
    headers = ["read_0001", "read_1999", "read_0000", "read_0001", "aaa", "zzz", "read_0500x", "read_0500"]  # between records, dups, a record's id
    eng = _engine("bacteria", "relaxed")
    eng.load_taxonomy_arrays(ids, lin)
    a = eng.run_host(text)
    a.add_headers(headers)
    b = eng.run_host(text)
    if when == "before":
        b.add_headers(headers)
        b.sort_by_query()
    else:
        b.sort_by_query()
        b.add_headers(headers)
    assert len(b) == len(a) == len(qids) + len(headers) - 2
    assert len(b.records()) == len(qids) and len(a.records()) == len(qids)  # (records only: the headers are not records)
    assert len(a.query_ids()) == len(qids)
    _check(a, b, tmp_path)


# --- 5. multi-device contexts ----------------------------------------------------------------------------------------
def test_multi_device_sorted_equals_single(tmp_path):
    from test_gpu_parity import _synth_case

    ids, lin, text = _synth_case(5000, 30000, 8, seed=37)
    ref = None
    for devs in _device_sets():
        for refs in (False, True):
            eng = _multi(devs, text_refs=refs)
            eng.load_taxonomy_arrays(ids, lin)
            a, b = _run_both(eng, lambda e: e.run_host(text))
            if ref is None:
                ref = b.query_ids()
            assert b.query_ids() == ref
            _check(a, b, tmp_path)
            eng.close()


# --- 6. determinism --------------------------------------------------------------------------------------------------
def test_two_runs_same_order():
    import torch

    from test_gpu_parity import _synth_case

    ids, lin, text = _synth_case(5000, 20000, 10, seed=41)
    eng = _engine("bacteria", "relaxed")
    eng.load_taxonomy_arrays(ids, lin)
    t = _to_device(text)
    s = torch.cuda.current_stream().cuda_stream
    seqs = []
    for _ in range(2):
        out = eng.run_device_resident(t.data_ptr(), len(text), s).sort_by_query()
        seqs.append(_device_ids(out))
        out.close()
    assert seqs[0] == seqs[1]


# --- 7. scale --------------------------------------------------------------------------------------------------------
def test_million_queries():
    from blutils_b200 import ConsensusEngine, ConsensusStrategy, Taxon, _ffi
    from blutils_b200.synth import SynthWorkload

    nq, hits = 1_000_000, 50
    w = SynthWorkload(30000, seed=20261018 + 9)
    tids, off, blob = w.lineages(False)
    eng = ConsensusEngine(Taxon.Bacteria, ConsensusStrategy.Relaxed, False, None)
    eng.load_taxonomy_raw(tids.ctypes.data, off.ctypes.data, blob.ctypes.data, len(tids))
    cap = nq * hits * 96 + (1 << 20)
    pinned = _ffi.lib().blu_host_alloc(cap)
    assert pinned
    try:
        n, _ = w.hits_into(pinned, cap, 0, nq, hits)
        a = eng.run_host(pinned, n)
        b = eng.run_host(pinned, n)
        b.sort_by_query()
        assert len(b) == nq and b.checksum() == a.checksum()
        recs = b.records()
        assert len(recs) == nq
        base = _ffi.lib().blu_result_pool(b._h, None)
        prev = None
        for r in recs:  # linear pass
            q = C.string_at(base + r.query_off, r.query_len)
            assert prev is None or prev < q
            prev = q
        assert b.jsonl(head=1000) == a.jsonl(head=1000)
        a.close()
        b.close()
    finally:
        _ffi.lib().blu_host_free(pinned)
