"""Hypothesis strategies of the property tests -- lineage maps, hit tables, rows of the input grammar -- and the three-way
comparison of the CPU implementations: oracle/pyoracle.py, oracle/blu_oracle.cpp and the product's device core compiled for
the host.  The CPU property tests (tests/test_properties_hypothesis.py), the variant generator (tests/consensus_variants.py)
and the GPU property tests draw from here."""
from hypothesis import HealthCheck, event
from hypothesis import strategies as st

import pyoracle as po
import sim_ffi
from oracle_ffi import Oracle, OracleDataError

# Settings of the GPU property tests: derandomised, so every run draws the same cases.
GPU = dict(max_examples=150, derandomize=True, deadline=None, database=None, suppress_health_check=list(HealthCheck))

RANKS = ["d", "k", "p", "c", "o", "f", "g", "s"]
EXTRA = ["clade", "species group", "strain", "no rank", "subspecies"]


@st.composite
def lineage_maps(draw):
    """A small tree: every lineage shares the domain (the reference aborts on root disagreement), ranks in Linnaean order with
    optional non-Linnaean levels spliced in, identifiers from a tiny alphabet so that lineages share prefixes."""
    n = draw(st.integers(2, 9))
    lineages = []
    for _ in range(n):
        depth = draw(st.integers(2, len(RANKS)))
        parts = ["d__bac"]
        for r in RANKS[1:depth]:
            if draw(st.integers(0, 9)) == 0:
                # (the same identifier under two rank names at one level: two beans that tie completely -- the reference's order is
                # its HashMap's there; the implementations of this repository agree on the taxonomy map's order)
                parts.append(draw(st.sampled_from(EXTRA)) + "__x" + str(draw(st.integers(0, 2))))
            parts.append(r + "__" + r + str(draw(st.integers(0, 2))))
        if draw(st.integers(0, 5)) == 0:
            parts.append("strain__st" + str(draw(st.integers(0, 3))))
        lineages.append(";".join(parts))
    taxids = draw(st.lists(st.integers(1, 10_000), min_size=n, max_size=n, unique=True))
    return dict(zip(taxids, lineages))


def _pident(draw):
    whole = draw(st.integers(40, 100))
    if whole == 100 or draw(st.booleans()):
        return f"{whole}.000" if draw(st.booleans()) else str(whole)
    return f"{whole}.{draw(st.integers(0, 999)):03d}"


@st.composite
def tables(draw, tax):
    """queries: list of (id, rows); a row = (acc, taxid, pident, length, bitscore text).  Bit scores come from a few levels so
    that top groups of several rows are common; one in ten is written with a decimal fraction (truncated by the reference)."""
    ids = sorted(tax)
    n_q = draw(st.integers(1, 6))
    queries = []
    for q in range(n_q):
        rows = []
        for h in range(draw(st.integers(1, 9))):
            level = draw(st.integers(0, 3))
            bits = 900 - 50 * level
            bits_txt = f"{bits}.{draw(st.integers(0, 9))}" if draw(st.integers(0, 9)) == 0 else str(bits)
            rows.append((f"AC{q}_{h}.{draw(st.integers(1, 3))}", draw(st.sampled_from(ids)), _pident(draw), draw(st.integers(50, 1500)), bits_txt))
        queries.append((f"q{q:02d}_{draw(st.integers(0, 99))}", rows))
    # distinct query ids (a repeated id would merge two groups: legal, but not what these properties talk about)
    seen = set()
    out = []
    for qid, rows in queries:
        while qid in seen:
            qid += "x"
        seen.add(qid)
        out.append((qid, rows))
    return out


def _text(queries) -> bytes:
    return "".join(f"{qid}\t{acc}\t{taxid}\t{pid}\t{ln}\t0\t0\t1\t{ln}\t1\t{ln}\t1e-50\t{bits}\n" for qid, rows in queries for acc, taxid, pid, ln, bits in rows).encode()


def _three_ways(tax, text, taxon, strategy, loud_limits=False, custom=None, headers=None):
    """canonical JSONL (bytes) or None when the reference would abort; asserts that the three implementations agree.
    loud_limits: the product may answer BLU_ERR_UNSUPPORTED (5) where the oracles have a result -- its documented limits
    (DESIGN.md section 5: numbers outside the exactly-parsed range; the host-compiled core has no regrouping of scattered
    tables) -- but never a different result and never a silent one."""
    ids = list(tax)
    lin = [tax[i] for i in ids]
    try:
        a = po.results_to_jsonl(po.build_consensus_identities(text, tax, taxon, strategy, custom, headers=headers)).encode()
    except po.DataError:
        a = None
    try:
        b = Oracle(ids, lin, taxon, strategy, custom, threads=2).run_raw(text, headers=headers)[0]
    except OracleDataError:
        b = None
    rc, c, msg = sim_ffi.run(ids, lin, taxon, strategy, text, custom=custom, headers=headers)
    assert (a is None) == (b is None), (a is None, b is None)
    if loud_limits and rc == 5 and a is not None:
        event("product: loud limit (" + msg.split(" at ")[0] + ")")
        return a
    assert (a is None) == (rc != 0), (a is None, rc, msg)
    if a is not None:
        assert a == b
        assert a == c
    return a


# ---- the input grammar: rows with clean and with odd fields -------------------------------------------------------------------
INTS = ["0", "7", "12", "1500", "-3", "+4", "007", "1_0", "", " 5", "5 ", "1e3", "9223372036854775807", "9223372036854775808", "123456789012345678",
        "1234567890123456789", "1.0", "0x10", "٣", "--1"]
FLOATS = ["99.5", "100", "100.000", "0", "0.0", "1e-5", "1E+3", "2.5e-10", ".5", "5.", "-0.0", "+1.5", "inf", "nan", "NaN", "-inf", "1e400", "1e-400", "0x10",
          "1.2.3", "", "1,5", "1e", "e5", "1e+", " 1.0", "1.0 ", "4.9e-324", "1.7976931348623157e308", "123456789012345678901234567890", "0.1234567890123456789",
          "1d5", "1_0.0", "١.٥"]
BITS = ["900", "900.0", "900.9", "52.8", "1e3", "0", "-5", "2147483647", "2147483648", "99999999999", "1234567890123456", "9.99e2", "", "x", "900.", ".9"]
IDS = ["q1", "read/1", "a b", "q\"x", "'q'", "é漢", "\U0001d518", "", " ", "q1 ", "#q", "x" * 70, "q\\t"]


@st.composite
def grammar_rows(draw, taxids):
    n = draw(st.integers(1, 5))
    rows = []
    for _ in range(n):
        weird = draw(st.integers(0, 3)) == 0  # most rows are clean so that a table is often accepted as a whole
        pick = (lambda clean, pool: draw(st.sampled_from(pool)) if weird and draw(st.booleans()) else clean)
        f = [pick("q1", IDS), pick("ACC.1", IDS), pick(str(draw(st.sampled_from(taxids))), INTS), pick("97.5", FLOATS), pick("300", INTS), pick("0", INTS),
             pick("0", INTS), pick("1", INTS), pick("300", INTS), pick("1", INTS), pick("300", INTS), pick("1e-50", FLOATS), pick("640", BITS)]
        shape = draw(st.integers(0, 19)) if weird else 9
        if shape == 0:
            f = f[:12]
        elif shape == 1:
            f = f + ["extra"]
        elif shape == 2:
            f[-1] += "\t"
        line = "\t".join(f) + ("\r\n" if shape == 3 else "\n")
        if shape == 4:
            line = "\n" + line
        rows.append(line)
    text = "".join(rows)
    if draw(st.integers(0, 5)) == 0 and text.endswith("\n"):
        text = text[:-1]  # no newline at the end of the file
    return text.encode("utf-8")
