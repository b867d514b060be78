"""What each consensus entry point reports in its timings, and the capacity retry of the device-text paths.

Expected launch counts come from the run loop: every range (device text) or chunk (host text, file) queues five kernels
(tile, long-run, consensus, duplicate-id check, advance) plus the gather kernel when the strings go to a pool that is
downloaded with the records.  A downloaded result moves its records, beans, accession references and string pool plus
one counter snapshot; a device-resident result moves the snapshot only."""
import ctypes as C

import pytest

from helpers import CHUNK, COUNTERS_BYTES, IDS, LIN, current_stream, engine, hit_table, tiny_rows, to_device
from oracle_ffi import Oracle

pytestmark = pytest.mark.gpu


def _pool_len(out):
    from blutils_b200 import _ffi

    n = C.c_uint64()
    _ffi.lib().blu_result_pool(out._h, C.byref(n))
    return n.value


def _check(t, tiles, launches, h2d, d2h, regrouped=0):
    assert int(t["n_tile_launches"]) == tiles
    assert int(t["n_kernel_launches"]) == launches
    assert int(t["h2d_bytes"]) == h2d
    assert int(t["d2h_bytes"]) == d2h
    assert int(t["n_regrouped"]) == regrouped


def test_device_download_retries_over_four_ranges(monkeypatch):
    """The first attempt overflows; every range of it is dropped (the downloads already queued included) and the run
    starts over with grown capacities.  The timings are those of the final attempt."""
    monkeypatch.setenv("BLU_RANGE_FRACS", "1,1,1,1")
    text = tiny_rows()
    want = Oracle(IDS, LIN, "bacteria", "relaxed").run_raw(text)[0]
    eng = engine("bacteria", "relaxed", lineages=(IDS, LIN))
    t = to_device(text)
    out = eng.run_device(t.data_ptr(), len(text), current_stream())
    assert len(out) == 120000 and out.jsonl() == want
    tm = eng.timings()
    _check(tm, 4, 4 * 6, 0, int(tm["result_bytes"]) + _pool_len(out) + COUNTERS_BYTES)
    out.close()
    eng.close()


def test_device_resident_retries():
    text = tiny_rows()
    want = Oracle(IDS, LIN, "bacteria", "relaxed").run_raw(text)[0]
    eng = engine("bacteria", "relaxed", lineages=(IDS, LIN))
    t = to_device(text)
    out = eng.run_device_resident(t.data_ptr(), len(text), current_stream())
    _check(eng.timings(), 1, 5, 0, COUNTERS_BYTES)
    assert out.download().jsonl() == want and len(out) == 120000
    out.close()
    eng.close()


def test_timings_of_every_entry_point(tmp_path, monkeypatch):
    """A contiguous ~9 MB table that fits the first capacity estimate, through every entry point."""
    text = hit_table(900, 0, seed=3)
    n = len(text)
    chunks = (n + CHUNK - 1) // CHUNK
    assert chunks > 2
    t = to_device(text)

    eng = engine("bacteria", "relaxed", lineages=(IDS, LIN))
    out = eng.run_device_resident(t.data_ptr(), n, current_stream())
    _check(eng.timings(), 1, 5, 0, COUNTERS_BYTES)
    want = out.download().checksum()
    out.close()

    monkeypatch.setenv("BLU_RANGE_FRACS", "1,1,1,1")
    out = eng.run_device(t.data_ptr(), n, current_stream())
    tm = eng.timings()
    _check(tm, 4, 4 * 6, 0, int(tm["result_bytes"]) + _pool_len(out) + COUNTERS_BYTES)
    assert out.checksum() == want
    out.close()
    monkeypatch.delenv("BLU_RANGE_FRACS")
    eng.close()

    eng = engine("bacteria", "relaxed", chunk_bytes=CHUNK, lineages=(IDS, LIN))
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
    eng = engine("bacteria", "relaxed", chunk_bytes=CHUNK, text_refs=True, lineages=(IDS, LIN))
    out = eng.run_host(text)
    tm = eng.timings()
    _check(tm, chunks, chunks * 5, n, int(tm["result_bytes"]) + COUNTERS_BYTES)
    assert out.checksum() == want
    out.close()
    eng.close()
