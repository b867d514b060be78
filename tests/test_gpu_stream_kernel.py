"""Parity cases aimed at the mechanisms of the streaming tile kernel (blu_kernels.cu): queries carried from window to
window (best bit score found late, top group collected across windows, carried top group overflowing to the block path),
windows with more finished queries than the record buffer holds, slot slabs, the lean row parser / top-row splitter next
to their full-grammar fallbacks, non-ASCII bytes, and run-to-run determinism of a large device-resident table.
All against the CPU oracle, bit for bit on the canonical JSONL."""
import random

import pytest

from helpers import IDS5, LIN5, current_stream, engine, hit_row, synth_case, to_device
from oracle_ffi import Oracle, checksum_jsonl

pytestmark = pytest.mark.gpu


def _want(text, strategy="relaxed"):
    return Oracle(IDS5, LIN5, "bacteria", strategy).run_raw(text)[0]


def _check(text, strategies=("relaxed", "cautious"), chunks=(0,)):
    if isinstance(text, str):
        text = text.encode()
    for st in strategies:
        want = _want(text, st)
        for ch in chunks:
            eng = engine("bacteria", st, chunk_bytes=ch, lineages=(IDS5, LIN5))
            assert eng.run_host(text).jsonl() == want, (st, ch)
            eng.close()


def test_best_score_found_in_a_later_window():
    """Queries of 1500 rows (~4 windows each): the best bit score sits at a random depth, so the carried top group is
    dropped and restarted; ties are spread over several windows (carried top rows + this window's)."""
    rng = random.Random(5)
    rows = []
    for q in range(60):
        n = 1500
        best = sorted(rng.sample(range(n), rng.choice([1, 2, 5, 9])))
        for h in range(n):
            bits = "900" if h in best else str(100 + (h * 7 + q) % 700)
            rows.append(hit_row(f"query_{q:05d}", f"NR_{(q * 31 + h) % 1000:06d}.1", IDS5[(q + h) % 4], f"{90 + (h % 10)}.{h % 1000:03d}", 400 + h % 50, bits,
                                mismatch=3, sstart=17))
    _check("".join(rows), chunks=(0, 1 << 20))


def test_carried_top_group_overflows_to_the_block_path():
    """A top group of 40 rows spread over three windows (more than the 32 the carry holds): the query is handed to the
    long-run kernel when it ends; its neighbours are not disturbed."""
    rows = []
    for q in range(12):
        n = 1300
        tops = set(range(0, n, 33)) if q % 3 == 0 else {5, 700}
        for h in range(n):
            rows.append(hit_row(f"q{q:03d}", f"ACC{h % 9}.1", IDS5[h % 3], "98.500", 300, "500" if h in tops else str(50 + h % 400), mismatch=3, sstart=17))
    text = "".join(rows)
    want = _want(text.encode())
    eng = engine("bacteria", "relaxed", lineages=(IDS5, LIN5))
    assert eng.run_host(text.encode()).jsonl() == want
    assert eng.timings()["n_deferred_runs"] >= 4  # the four 40-row top groups really took the block path
    eng.close()


def test_windows_full_of_tiny_queries():
    """Rows of 27-40 bytes, one or two hits per query: > 1000 rows and > 256 finished queries per 32 KB window (several
    row-loop rounds, record buffer overflow, a slot slab every few windows)."""
    rng = random.Random(11)
    rows = []
    for q in range(60000):
        for h in range(1 + (q % 7 == 0)):
            rows.append(f"q{q}\tA\t{IDS5[q % 2]}\t9{h}\t{1 + q % 9}\t0\t0\t1\t1\t1\t1\t0\t{5 + (q + h) % 3}\n")
    rng.random()
    _check("".join(rows), strategies=("relaxed",), chunks=(0, 1 << 20))


def test_number_shapes_lean_and_fallback():
    """Every numeric shape the lean parser / splitter accept next to the ones they hand to the full grammar."""
    pidents = ["100", "99.", ".5", "99.123456", "87.5", "1e2", "9.95e1", "100.000"]
    bitss = ["7", "1234", "12345678", "123456789", "57.9", "0.5", "1e3", "2.5e2", "99999999.5"]
    evalues = ["0.0", "0", "1e-180", "2.51e-117", "3.4E-08", "0.001", "5", "1.e-5", ".5e-3"]
    rows = []
    q = 0
    for pid in pidents:
        for bits in bitss:
            ev = evalues[q % len(evalues)]
            for h in range(3):
                rows.append(hit_row(f"q{q:04d}", f"WP_{q}.{h}", IDS5[(q + h) % 5], pid, 250 + h, bits, mismatch=3, sstart=17, evalue=ev))
            q += 1
    _check("".join(rows))


def test_non_ascii_and_long_identifiers():
    """UTF-8 bytes in qseqid / saccver (exact byte-wise classification path), identifiers longer than 32 and 64 bytes."""
    rows = []
    for q in range(300):
        name = ["müller_%d" % q, "q%d_" % q + "x" * 40, "漢字_%d" % q, "r%d_" % q + "y" * 90][q % 4]
        for h in range(20):
            acc = "ACC_é%d.1" % (h % 3) if q % 5 == 0 else "NR_%06d.1" % h
            rows.append(hit_row(name, acc, IDS5[h % 4], "97.125", 300, "450" if h < 2 else str(100 + h), mismatch=3, sstart=17))
    _check("".join(rows).encode("utf-8"))


def test_large_table_is_deterministic():
    """A 200 MB device-resident table run five times: identical checksums (a race between phases / windows would show up
    as a varying result), equal to the oracle's."""
    ids, lin, text = synth_case(20000, 52000, 50, seed=77)
    want = checksum_jsonl(Oracle(ids, lin, "bacteria", "relaxed").run_raw(text)[0])
    eng = engine("bacteria", "relaxed", lineages=(ids, lin))
    t = to_device(text)
    for _ in range(5):
        out = eng.run_device(t.data_ptr(), len(text), current_stream())
        assert len(out) == 52000 and out.checksum() == want
        out.close()
    eng.close()


def test_query_spanning_many_segments():
    """One query of 150 k rows (~10 MB: dozens of 128 KB+ segments lie entirely inside it) between ordinary queries: the CTA
    that owns its first row walks through all of them, the CTAs of the segments in between find no query of their own."""
    rows = []
    for q in range(40):
        for h in range(30):
            rows.append(hit_row(f"small_a{q:03d}", f"NR_{h:06d}.1", IDS5[h % 3], "97.500", 300, "400" if h < 2 else str(100 + h), mismatch=3, sstart=17))
    for h in range(150_000):
        bits = "999" if h in (7, 70_000, 149_999) else str(100 + h % 800)
        rows.append(hit_row("the_big_one", f"NR_{h % 5000:06d}.1", IDS5[h % 4], f"9{h % 10}.{h % 1000:03d}", 250 + h % 100, bits, mismatch=3, sstart=17))
    for q in range(40):
        for h in range(30):
            rows.append(hit_row(f"small_b{q:03d}", f"NR_{h:06d}.1", IDS5[(h + 1) % 3], "96.250", 300, "380" if h < 3 else str(90 + h), mismatch=3, sstart=17))
    _check("".join(rows), strategies=("relaxed",), chunks=(0, 4 << 20))
