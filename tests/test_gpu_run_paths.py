"""What each consensus entry point reports in its timings, and the capacity retry of the device-text paths.

Expected launch counts come from the run loop: every range (device text) or chunk (host text, file) queues five kernels
(tile, long-run, consensus, duplicate-id check, advance) plus the gather kernel when the strings go to a pool that is
downloaded with the records.  A downloaded result moves its records, beans, accession references and string pool plus
one counter snapshot; a device-resident result moves the snapshot only."""
import ctypes as C

import pytest

from test_gpu_file_stream import IDS, LIN, _engine, _table

pytestmark = pytest.mark.gpu

COUNTERS_BYTES = 120  # sizeof(Counters), blu_kernels.h: eleven 8-byte and eight 4-byte fields
CHUNK = 1 << 20


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


def _pool_len(out):
    from blutils_b200 import _ffi

    n = C.c_uint64()
    _ffi.lib().blu_result_pool(out._h, C.byref(n))
    return n.value


def _tiny_rows():
    """One or two tiny rows per query (the shape of the streamed-file retry test): a fresh context's first capacity
    estimate holds about a third of the records."""
    rows = []
    for q in range(120000):
        for h in range(1 + (q % 5 == 0)):
            rows.append(f"q{q}\tA\t{IDS[q % 2]}\t9{h}\t{1 + q % 9}\t0\t0\t1\t1\t1\t1\t0\t{5 + (q + h) % 3}\n")
    return "".join(rows).encode()


def _check(t, tiles, launches, h2d, d2h, regrouped=0):
    assert int(t["n_tile_launches"]) == tiles
    assert int(t["n_kernel_launches"]) == launches
    assert int(t["h2d_bytes"]) == h2d
    assert int(t["d2h_bytes"]) == d2h
    assert int(t["n_regrouped"]) == regrouped


def test_device_download_retries_over_four_ranges(monkeypatch):
    """The first attempt overflows; every range of it is dropped (the downloads already queued included) and the run
    starts over with grown capacities.  The timings are those of the final attempt."""
    from oracle_ffi import Oracle

    monkeypatch.setenv("BLU_RANGE_FRACS", "1,1,1,1")
    text = _tiny_rows()
    want = Oracle(IDS, LIN, "bacteria", "relaxed").run_raw(text)[0]
    eng = _engine()
    t = _to_device(text)
    out = eng.run_device(t.data_ptr(), len(text), _stream())
    assert len(out) == 120000 and out.jsonl() == want
    tm = eng.timings()
    _check(tm, 4, 4 * 6, 0, int(tm["result_bytes"]) + _pool_len(out) + COUNTERS_BYTES)
    out.close()
    eng.close()


def test_device_resident_retries():
    from oracle_ffi import Oracle

    text = _tiny_rows()
    want = Oracle(IDS, LIN, "bacteria", "relaxed").run_raw(text)[0]
    eng = _engine()
    t = _to_device(text)
    out = eng.run_device_resident(t.data_ptr(), len(text), _stream())
    _check(eng.timings(), 1, 5, 0, COUNTERS_BYTES)
    assert out.download().jsonl() == want and len(out) == 120000
    out.close()
    eng.close()


def test_timings_of_every_entry_point(tmp_path, monkeypatch):
    """A contiguous ~9 MB table that fits the first capacity estimate, through every entry point."""
    text = _table(900, 0, seed=3)
    n = len(text)
    chunks = (n + CHUNK - 1) // CHUNK
    assert chunks > 2
    t = _to_device(text)

    eng = _engine()
    out = eng.run_device_resident(t.data_ptr(), n, _stream())
    _check(eng.timings(), 1, 5, 0, COUNTERS_BYTES)
    want = out.download().checksum()
    out.close()

    monkeypatch.setenv("BLU_RANGE_FRACS", "1,1,1,1")
    out = eng.run_device(t.data_ptr(), n, _stream())
    tm = eng.timings()
    _check(tm, 4, 4 * 6, 0, int(tm["result_bytes"]) + _pool_len(out) + COUNTERS_BYTES)
    assert out.checksum() == want
    out.close()
    monkeypatch.delenv("BLU_RANGE_FRACS")
    eng.close()

    eng = _engine(CHUNK)
    out = eng.run_host(text)
    tm = eng.timings()
    _check(tm, chunks, chunks * 6, n, int(tm["result_bytes"]) + _pool_len(out) + COUNTERS_BYTES)
    assert out.checksum() == want
    out.close()

    path = tmp_path / "blast.out"
    path.write_bytes(text)
    out = eng.run_file(str(path))
    tm = eng.timings()
    _check(tm, chunks, chunks * 6, n, int(tm["result_bytes"]) + _pool_len(out) + COUNTERS_BYTES)
    assert out.checksum() == want
    out.close()
    eng.close()

    # text references: no string pool is gathered or downloaded
    from blutils_b200 import ConsensusEngine, ConsensusStrategy, Taxon

    eng = ConsensusEngine(Taxon.Bacteria, ConsensusStrategy.Relaxed, False, None, chunk_bytes=CHUNK, text_refs=True)
    eng.load_taxonomy_arrays(IDS, LIN)
    out = eng.run_host(text)
    tm = eng.timings()
    _check(tm, chunks, chunks * 5, n, int(tm["result_bytes"]) + COUNTERS_BYTES)
    assert out.checksum() == want
    out.close()
    eng.close()
