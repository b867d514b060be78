"""BASELINE configs C2..C5 at sizes a test run affords, checked against the CPU oracle through the order-independent
checksum of the canonical JSONL (sum of FNV-1a per line) and through sharding / streaming invariance."""
import ctypes as C

import pytest

from helpers import CUTOFFS_16S, engine
from oracle_ffi import Oracle

pytestmark = pytest.mark.gpu


def _baseline_case(n_taxa, seed, taxon="bacteria", strategy="relaxed", custom=None, chunk_bytes=0, numeric=False):
    """A synthetic workload, an engine that holds its lineage map (loaded through the raw-array entry point), the oracle."""
    from blutils_b200.synth import SynthWorkload

    w = SynthWorkload(n_taxa, seed=seed)
    ids, off, blob = w.lineages(numeric=numeric)
    eng = engine(taxon, strategy, numeric, custom, chunk_bytes=chunk_bytes)
    eng.load_taxonomy_raw(ids.ctypes.data, off.ctypes.data, blob.ctypes.data, len(ids))
    lin = [bytes(blob[int(off[i]):int(off[i + 1])]).decode() for i in range(len(ids))]
    return w, eng, Oracle(ids.tolist(), lin, taxon, strategy, custom)


def _check(eng, orc, text, n_queries):
    from oracle_ffi import checksum_jsonl

    want, nq, nr = orc.run_raw(text)
    out = eng.run_host(text)
    assert len(out) == nq == n_queries and out.n_rows == nr
    assert out.checksum() == checksum_jsonl(want)
    return out


def test_c2_custom_16s_cutoffs():
    """C2 shape: 50 hits/query, 30 k taxa, --taxon custom with the 16S YAML values (120 k queries, 458 MB)."""
    w, eng, orc = _baseline_case(30_000, 20261020, taxon="custom", custom=CUTOFFS_16S)
    text = w.hits(0, 120_000, 50)
    _check(eng, orc, text, 120_000)
    eng.close()


def test_c3_two_million_taxa():
    """C3 shape: 100 hits/query against a 2 M-taxon lineage map (hash table + tables beyond L1, 60 k queries)."""
    w, eng, orc = _baseline_case(2_000_000, 20261021, strategy="cautious", numeric=True)
    text = w.hits(0, 60_000, 100)
    out = _check(eng, orc, text, 60_000)
    # device-resident path on the same table
    import torch

    n = len(text)
    t = torch.empty((n + 255) // 128 * 128, dtype=torch.uint8, device="cuda")
    t[:n] = torch.frombuffer(bytearray(text), dtype=torch.uint8).cuda()
    torch.cuda.synchronize()
    assert eng.run_device(t.data_ptr(), n, torch.cuda.current_stream().cuda_stream).checksum() == out.checksum()
    eng.close()


def test_c4_zipf_skew():
    """C4 shape: Zipf(1.1) hits/query on [1, 5000] (long-tail queries take the block path), ~400 MB."""
    w, eng, orc = _baseline_case(200_000, 20261022)
    text = w.hits(0, 12_000, 5000, zipf=True)
    out = _check(eng, orc, text, 12_000)
    assert eng.timings()["n_deferred_runs"] >= 0  # (the streaming kernels carry queries of any length; only top groups > 32 rows take the block path)
    eng.close()


def test_c5_streamed_shards():
    """C5 shape: 50 hits/query streamed from host memory in 64 MiB chunks; query-sharded 8 ways, every shard processed
    on its own, the shard checksums must add up to the checksum of the whole (and to the oracle's)."""
    from blutils_b200 import shard_cuts

    w, eng, orc = _baseline_case(200_000, 20261023, chunk_bytes=64 << 20)
    text = w.hits(0, 300_000, 50)
    whole = _check(eng, orc, text, 300_000).checksum()
    cuts = shard_cuts(text, 8)
    total = 0
    nq = 0
    for a, b in zip(cuts[:-1], cuts[1:]):
        part = eng.run_host(text[a:b])
        total = (total + part.checksum()) % (1 << 64)
        nq += len(part)
    assert nq == 300_000 and total == whole
    eng.close()
