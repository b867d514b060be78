"""Variants of the generated cases of tests/generators.py that reach every consensus implementation of the GPU.

The size of a query's top bit-score group picks the implementation on the GPU:

* ``narrow``: 1..8 rows -- ``cons_compute<8>`` of the consensus kernel (four queries per warp);
* ``warp32``: 9..32 rows -- ``cons_compute<32>`` (one query per warp);
* ``block``: more than 32 rows, or any bit score beyond int32 -- the long-run kernel (``long_consensus``, and
  ``consensus_single`` for a single row).

``tables()`` gives top groups of 1..4 rows nearly always, so the generated cases alone only reach the first.  Every query of a
case is rewritten here into five variants, each under its own query id:

* ``orig``: the query as drawn;
* ``lift``: 3 000 000 000 added to the integer part of every bit score ("850.3" -> "3000000850.3"): ties and the order under
  truncation stay, the value stays inside the exactly parsed range, and the query -- a single-row one too -- takes the block path;
* ``w32``: the top group grown to 9..32 rows by repeating its rows cyclically;
* ``block``: the top group grown to 33..1000 rows the same way;
* ``lw32``: the lift applied to a ``w32`` query: a 9..32 group through ``long_consensus``.

A grown query's copies keep their source's accession (the Vec::dedup after the sort drops them) or get a fresh one each (long
accession lists, accessions longer than 16 bytes that share their first 16); its lower rows stay, spread among the top rows.

Fully tied beans -- one identifier under two rank names at one level, with equal occurrences -- need two top lineages that
differ in a rank name only; the drawn lineage maps hardly ever put such a pair into one top group.  So every lineage of a case
gets a twin: the same lineage under a new taxid, with the rank name of one level replaced.  In a grown query drawn to use them,
every other cycle of copies maps to the twins, which makes the two beans of a source row tie whenever the cycles are even.  A
twin that differs at the root makes its query a root-level disagreement: an error in every configuration.

No GPU imports: the CPU tests use the generator as the GPU tests do."""
from hypothesis import strategies as st

from generators import lineage_maps, tables  # noqa: F401  (the strategies the variants start from)

LIFT = 3_000_000_000
INT32_MAX = 2 ** 31 - 1
TWIN = 100_000  # taxid of a twin = taxid + TWIN (lineage_maps() draws taxids up to 10 000)
W32_SIZES = [9, 10, 17, 31, 32]
BLOCK_SIZES = [33, 34, 64, 257, 1000]
CLASSES = ["narrow", "warp32", "block"]
CONFIGS = [(taxon, strategy) for taxon in ("bacteria", "fungi", "eukaryotes", "custom") for strategy in ("cautious", "relaxed")]


def truncated(bits: str) -> int:
    """The bit score as the reference compares it (mod.rs:162,184: the f64 truncated)."""
    return int(float(bits))


def expected_class(rows) -> str:
    """The implementation the dispatch rule picks for a query's rows: the count of rows at the maximal truncated bit score,
    and whether any bit score lies beyond int32."""
    bits = [truncated(r[4]) for r in rows]
    top = max(bits)
    if top > INT32_MAX:
        return "block"
    g = bits.count(top)
    return "narrow" if g <= 8 else "warp32" if g <= 32 else "block"


def lift(rows):
    out = []
    for acc, taxid, pid, ln, bits in rows:
        whole, dot, frac = bits.partition(".")
        out.append((acc, taxid, pid, ln, str(int(whole) + LIFT) + dot + frac))
    return out


def twin_lineage(lineage: str, level: int) -> str:
    """`lineage` with the rank name of `level` replaced (the identifier stays)."""
    levels = lineage.split(";")
    rank, ident = levels[level].split("__", 1)
    levels[level] = ("clade" if rank == "no rank" else "no rank") + "__" + ident
    return ";".join(levels)


def grow(rows, size, fresh, twins=False):
    """The top group grown to `size` rows: its rows repeated cyclically, the copies spread evenly over the query's rows.
    fresh: every copy gets an accession of its own; twins: the copies of odd cycles map to the twin of their source's taxid."""
    top = max(truncated(r[4]) for r in rows)
    tops = [r for r in rows if truncated(r[4]) == top]
    copies = []
    for i in range(len(tops), size):
        acc, taxid, pid, ln, bits = tops[i % len(tops)]
        copies.append((f"{acc}_copy_{i:05d}" if fresh else acc, taxid + TWIN if twins and (i // len(tops)) % 2 else taxid, pid, ln, bits))
    out, k = [], 0
    for j, r in enumerate(rows):
        out.append(r)
        upto = (j + 1) * len(copies) // len(rows)
        out.extend(copies[k:upto])
        k = upto
    return out


@st.composite
def variants(draw, tax, queries):
    """(the lineage map with the twins added, [(query id, rows, kind, expected class)]): every query of `queries` (as drawn by
    tables() over `tax`) in the five variants."""
    full = dict(tax)
    for taxid, lineage in tax.items():
        depth = lineage.count(";") + 1
        level = 0 if draw(st.integers(0, 5)) == 0 else draw(st.integers(1, depth - 1))
        full[taxid + TWIN] = twin_lineage(lineage, level)
    out = []
    for qid, rows in queries:
        fresh, twins = draw(st.booleans()), draw(st.booleans())
        w32 = grow(rows, draw(st.sampled_from(W32_SIZES)), fresh, twins)
        for kind, vrows in (("orig", rows), ("lift", lift(rows)), ("w32", w32),
                            ("block", grow(rows, draw(st.sampled_from(BLOCK_SIZES)), fresh, twins)), ("lw32", lift(w32))):
            out.append((f"{qid}~{kind}", vrows, kind, expected_class(vrows)))
    return full, out


def custom_cutoffs(draw):
    """A custom cutoff table as the property tests draw it (taxon.rs:14-65: domain and species required, the others optional)."""
    custom = {"domain": draw(st.integers(0, 100)), "species": draw(st.integers(0, 100))}
    for k in ["kingdom", "phylum", "class", "order", "family", "genus"]:
        custom[k] = draw(st.one_of(st.none(), st.integers(0, 100)))
    return custom
