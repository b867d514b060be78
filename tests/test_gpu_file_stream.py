"""`blu_consensus_run_file`: the blast output is streamed from the file through a ring of pinned staging buffers
(parallel pread()s) instead of being read whole.  Same results as the in-memory path and as the CPU oracle; the
reference's error classes for unreadable / empty files (mod.rs:357-364 and the CsvReader panic)."""
import os
import random

import pytest

from helpers import IDS, LIN, engine, hit_table, random_blast, random_taxonomy, tiny_rows
from oracle_ffi import Oracle, OracleDataError

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("chunk,threads", [(1 << 20, None), (1 << 20, "1"), (3 << 20, "5"), (0, None)])
def test_streamed_file_equals_memory_and_oracle(tmp_path, chunk, threads, monkeypatch):
    """~9 MB table: nine 1 MiB chunks (the staging ring wraps three times), three 3 MiB chunks, and one chunk."""
    if threads:
        monkeypatch.setenv("BLU_READ_THREADS", threads)
    text = hit_table(900, 0, seed=3)
    path = tmp_path / "blast.out"
    path.write_bytes(text)
    want = Oracle(IDS, LIN, "bacteria", "relaxed").run_raw(text)[0]
    eng = engine("bacteria", "relaxed", chunk_bytes=chunk, lineages=(IDS, LIN))
    from_file = eng.run_file(str(path))
    assert from_file.jsonl() == want
    t = eng.timings()
    assert int(t["h2d_bytes"]) == len(text)
    from_mem = eng.run_host(text)
    assert from_mem.checksum() == from_file.checksum() and len(from_mem) == len(from_file) == 900
    eng.close()


def test_streamed_file_restarts_after_a_capacity_retry(tmp_path):
    """Tiny rows, one or two per query: more queries than the first capacity estimate allows, so the run starts over from
    chunk 0 while the reader is already ahead."""
    text = tiny_rows()
    path = tmp_path / "tiny.out"
    path.write_bytes(text)
    want = Oracle(IDS, LIN, "bacteria", "relaxed").run_raw(text)[0]
    eng = engine("bacteria", "relaxed", chunk_bytes=1 << 20, lineages=(IDS, LIN))
    out = eng.run_file(str(path))
    assert len(out) == 120000 and out.jsonl() == want
    eng.close()


def test_noncontiguous_file_is_regrouped(tmp_path):
    rng = random.Random(301)
    units = random_taxonomy(rng, n_leaves=30)
    text = random_blast(rng, units, n_queries=40, contiguous=False)
    lin = [u["textLineage"] for u in units]
    ids = [u["taxid"] for u in units]
    try:
        want = Oracle(ids, lin, "fungi", "relaxed").run_raw(text)[0]
    except OracleDataError:
        pytest.skip("generated case hits a reference abort")
    path = tmp_path / "scattered.out"
    path.write_bytes(text)
    eng = engine("fungi", "relaxed", lineages=(ids, lin))
    out = eng.run_file(str(path))
    assert out.jsonl() == want
    eng.close()


def test_file_errors(tmp_path):
    from blutils_b200 import ConsensusPanic, MappedErrors

    eng = engine("bacteria", "relaxed", lineages=(IDS, LIN))
    with pytest.raises(MappedErrors):
        eng.run_file(str(tmp_path / "absent.out"))
    with pytest.raises(MappedErrors):
        eng.run_file(str(tmp_path))  # a directory
    empty = tmp_path / "empty.out"
    empty.write_bytes(b"")
    with pytest.raises(ConsensusPanic):
        eng.run_file(str(empty))
    bad = tmp_path / "bad.out"
    bad.write_bytes(hit_table(50, 30, seed=1) + b"q\tacc\t7\t99.0\t10\t0\t0\t1\t10\t1\t10\t0.0\n")  # 12 fields in the last row
    with pytest.raises(ConsensusPanic):
        eng.run_file(str(bad))
    # the context stays usable after a failed run
    good = tmp_path / "good.out"
    good.write_bytes(hit_table(50, 30, seed=1))
    assert len(eng.run_file(str(good))) == 50
    eng.close()
