"""Shared test helpers: seeded random taxonomies / hit tables for small parity cases, the cutoff tables and lineage maps
several modules use, and the constructors of engines and device-resident texts.

Generators avoid, by construction, inputs on which the reference is non-deterministic (bean full
ties: same identifier under different ranks) unless a test asks for error cases explicitly.

Nothing here imports blutils_b200 or torch at module level: the CPU-only suite collects every module."""
from __future__ import annotations

import json
import math
import os
import random
import sys
from typing import Dict, List, Optional, Tuple

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle"))

# The 16S cutoffs of the reference's custom-taxon YAML example.
CUTOFFS_16S = {"domain": 50, "kingdom": 60, "phylum": 75, "class": 80, "order": 85, "family": 92, "genus": 97, "species": 99}

# A small lineage map; IDS5 adds a 16-digit taxid, so that the taxids have 1 .. 16 digits (lean splitter: <= 8, <= 16, beyond).
LIN = ["d__bac;p__p1;c__c1;o__o1;f__f1;g__g1;s__s1", "d__bac;p__p1;c__c1;o__o1;f__f1;g__g1;s__s2", "d__bac;p__p1;c__c1;o__o1;f__f1;g__g2;s__s3",
       "d__bac;p__p1;c__c1;o__o1;f__f2;g__g3;s__s4"]
IDS = [7, 4242, 1660760528, 99999999]
LIN5 = LIN + ["d__bac;p__p2;c__c2;o__o2;f__f3;g__g4;s__s5"]
IDS5 = IDS + [1234567890123456]

COUNTERS_BYTES = 120  # sizeof(Counters), blu_kernels.h: eleven 8-byte and eight 4-byte fields
CHUNK = 1 << 20

# Known answers of InterpolatedIdentity::interpolate_identities (linnaean_ranks.rs:220-383), SURVEY.md section 3.3: rank names,
# the bacteria cutoffs, the CUTOFFS_16S cutoffs.
NAN = float("nan")
KAT = [
    ("d p c o f g s", [60, 75, 80, 85, 92, 97, 99], [50, 75, 80, 85, 92, 97, 99]),
    ("d clade p c o f g species-group species-subgroup s", [60, 67.5, 75, 80, 85, 92, 97, 97.667, 98.333, 99],
     [50, 62.5, 75, 80, 85, 92, 97, 97.667, 98.333, 99]),
    ("d p c o f g s strain", [60, 75, 80, 85, 92, 97, 99, 100], [50, 75, 80, 85, 92, 97, 99, 100]),
    ("d clade clade p c o f g s strain", [60, 65, 70, 75, 80, 85, 92, 97, 99, 100], [50, 58.333, 66.667, 75, 80, 85, 92, 97, 99, 100]),
    ("no-rank d p c o f g s", [99, 60, 75, 80, 85, 92, 97, 99], [50, 50, 75, 80, 85, 92, 97, 99]),
    ("d p c o suborder f g s", [60, 75, 80, 85, 88.5, 92, 97, 99], [50, 75, 80, 85, 88.5, 92, 97, 99]),
    ("d p c o f no-rank g s", [60, 75, 80, 85, 92, 94.333, 97, 99], [50, 75, 80, 85, 92, 94.333, 97, 99]),
    ("d p c o f g s subspecies no-rank", [60, 75, 80, 85, 92, 97, 99, 99.5, 100], [50, 75, 80, 85, 92, 97, 99, 99.5, 100]),
    ("d k p c o f g s", [60, 67.5, 75, 80, 85, 92, 97, 99], [50, 60, 75, 80, 85, 92, 97, 99]),
    ("superkingdom p c o f g s", [99, 75, 80, 85, 92, 97, 99], [50, 75, 80, 85, 92, 97, 99]),
    ("no-rank d k p c o f g s no-rank", [99, 60, 66.667, 75, 80, 85, 92, 97, 99, NAN], [50, 50, 60, 75, 80, 85, 92, 97, 99, NAN]),
    ("clade", [NAN], [NAN]),
]


def same(a, b):
    """Equal cutoff vectors, NaN equal to NaN."""
    return len(a) == len(b) and all((math.isnan(x) and math.isnan(y)) or x == y for x, y in zip(a, b))


def engine(taxon, strategy, use_taxid=False, custom=None, lineages=None, **kwargs):
    """A ConsensusEngine from taxon ("bacteria", "fungi", "eukaryotes", "custom") and strategy ("cautious", "relaxed")
    names and a cutoff dict; keyword arguments (chunk_bytes, text_refs, devices) go to the constructor, and
    `lineages` = (ids, lineage strings) is loaded when given."""
    from blutils_b200 import ConsensusEngine, ConsensusStrategy, CustomTaxon, Taxon

    ct = None
    if custom is not None:
        ct = CustomTaxon(domain=custom["domain"], species=custom["species"], kingdom=custom.get("kingdom"), phylum=custom.get("phylum"),
                         class_=custom.get("class"), order=custom.get("order"), family=custom.get("family"), genus=custom.get("genus"))
    eng = ConsensusEngine(Taxon[taxon.capitalize()], ConsensusStrategy[strategy.capitalize()], use_taxid, ct, **kwargs)
    if lineages is not None:
        eng.load_taxonomy_arrays(*lineages)
    return eng


def to_device(text):
    """`text` in a zero-padded device buffer (a multiple of 128 bytes, at least 128 bytes of padding)."""
    import torch

    n = len(text)
    t = torch.zeros((n + 255) // 128 * 128, dtype=torch.uint8, device="cuda")
    t[:n] = torch.frombuffer(bytearray(text), dtype=torch.uint8).cuda()
    torch.cuda.synchronize()
    return t


def current_stream():
    import torch

    return torch.cuda.current_stream().cuda_stream


def device_sets():
    """Device lists of multi-device contexts: [0] always, more where the box has the GPUs."""
    import torch

    n = torch.cuda.device_count()
    sets = [[0]]
    if n >= 2:
        sets += [[0, 1], [1, 0]]
    if n >= 4:
        sets.append([0, 1, 2, 3])
    if n >= 8:
        sets.append(list(range(8)))
    return sets


def hit_row(q, acc, taxid, pident, ln, bits, *, mismatch=0, sstart=1, evalue="0.0"):
    """One 13-column hit row (outfmt 6 std + bitscore): an alignment of `ln` columns, the subject's from `sstart`."""
    return f"{q}\t{acc}\t{taxid}\t{pident}\t{ln}\t{mismatch}\t0\t1\t{ln}\t{sstart}\t{ln + sstart - 1}\t{evalue}\t{bits}\n"


def hit_table(n_queries, rows_per_query, seed):
    """Queries over IDS / LIN, `rows_per_query` rows each (0: 1, 2, 3, 40 or 700 at random), 1, 2 or 4 of them top rows."""
    rng = random.Random(seed)
    rows = []
    for q in range(n_queries):
        n = rows_per_query if rows_per_query > 0 else rng.choice([1, 2, 3, 40, 700])
        best = set(rng.sample(range(n), min(n, rng.choice([1, 2, 4]))))
        for h in range(n):
            rows.append(hit_row(f"query_{q:06d}", f"NR_{(q * 17 + h) % 3000:06d}.1", IDS[(q + h) % 4], f"{88 + h % 12}.{(q + h) % 1000:03d}",
                                300 + h % 200, "950" if h in best else str(100 + (h * 13 + q) % 800), mismatch=3, sstart=17, evalue="1e-50"))
    return "".join(rows).encode()


def tiny_rows():
    """120 000 queries of one or two tiny rows over IDS: a fresh context's first capacity estimate holds about a third of
    the records."""
    rows = []
    for q in range(120000):
        for h in range(1 + (q % 5 == 0)):
            rows.append(f"q{q}\tA\t{IDS[q % 2]}\t9{h}\t{1 + q % 9}\t0\t0\t1\t1\t1\t1\t0\t{5 + (q + h) % 3}\n")
    return "".join(rows).encode()


def synth_case(n_taxa, n_queries, hits, zipf=False, seed=11):
    """(taxids, lineage strings, hit table) of a synthetic workload."""
    from blutils_b200.synth import SynthWorkload

    w = SynthWorkload(n_taxa, seed=seed)
    ids, off, blob = w.lineages()
    lin = [bytes(blob[int(off[i]):int(off[i + 1])]).decode() for i in range(len(ids))]
    text = w.hits(0, n_queries, hits, zipf=zipf)
    return ids.tolist(), lin, text


def scattered_table(rng, n_queries, max_hits, n_taxa, blank_lines=False, final_newline=True):
    """Rows of every query dealt out over the file in up to three far-apart fragments (file order inside a query kept)."""
    ids = list(range(1, n_taxa + 1))
    lin = [f"d__bac;p__p{t % 3};c__c{t % 7};o__o{t % 11};f__f{t % 13};g__g{t % 17};s__s{t}" for t in ids]
    parts = [[], [], []]
    for q in range(n_queries):
        t0 = rng.randrange(n_taxa)
        hits = rng.randint(1, max_hits)
        for h in range(hits):
            t = ids[(t0 + rng.choice([0, 0, 1, 2, 17])) % n_taxa]
            bits = 900 - 10 * (h // 3) + (1 if rng.random() < 0.05 else 0)  # now and then the best row sits in a later fragment
            row = hit_row(f"read_{q:06d}/1" if q % 7 else f"M0{q}:long:read:name:{q:09d}:abcdefgh", f"ACC{q}_{h}.{h % 3}", t,
                          f"{88 + (h * 5 + q) % 12}.{(q + h) % 100:02d}", 150 + h, str(bits))
            parts[min(2, rng.randrange(4))].append(row)
    rows = parts[0] + parts[1] + parts[2]
    if blank_lines:
        for i in range(5, len(rows), 211):
            rows[i] = "\n" + rows[i]
    text = "".join(rows)
    if not final_newline:
        text = text[:-1]
    return ids, lin, text.encode()


BACKBONE_RANKS = ["d", "p", "c", "o", "f", "g", "s"]
ODD_RANKS = ["clade", "no rank", "species group", "species subgroup", "strain", "subspecies", "k", "superkingdom",
             "Sub-Order", "u", "forma specialis", "serotype", "Domain", " Phylum "]


def random_taxonomy(rng: random.Random, n_leaves: int = 40, odd: float = 0.35, shared_root: bool = True,
                    truncate: float = 0.15) -> List[dict]:
    """A random tree; every leaf lineage becomes one taxonomy unit.  Identifiers are globally unique
    per node so that no two different (rank, identifier) pairs share an identifier."""
    counter = [0]

    def ident(prefix):
        counter[0] += 1
        return f"{prefix}{counter[0]}"

    # nodes at each backbone depth
    roots = [("d", ident("dom"))] if shared_root else [("d", ident("dom")) for _ in range(2)]
    units = []
    numid: Dict[str, int] = {}
    used_taxids = set()
    paths: List[List[Tuple[str, str]]] = [[r] for r in roots]
    for depth, rk in enumerate(BACKBONE_RANKS[1:], start=1):
        new_paths = []
        for p in paths:
            for _ in range(rng.choice([1, 1, 2, 3]) if len(paths) < n_leaves else 1):
                q = list(p)
                if rng.random() < odd / 2:
                    q.append((rng.choice(ODD_RANKS), ident("x")))
                q.append((rk, ident(rk)))
                new_paths.append(q)
        rng.shuffle(new_paths)
        paths = new_paths[: max(n_leaves, 1)]
    prefix_mode = rng.choice(["none"] * 6 + ["all"] * 3 + ["mixed"])
    prefix_rank = rng.choice(["no rank", "clade", "cellular root"])
    for p in paths:
        q = list(p)
        r = rng.random()
        if r < truncate:
            q = q[: rng.randint(1, len(q))]
        elif r < truncate + odd / 2:
            q.append((rng.choice(["strain", "subspecies", "no rank", "serotype"]), ident("t")))
        if prefix_mode == "all" or (prefix_mode == "mixed" and rng.random() < 0.5):
            q.insert(0, (prefix_rank, "cellular-organisms"))
        while True:
            t = rng.randint(1, 2_000_000_000)
            if t not in used_taxids:
                used_taxids.add(t)
                break
        text = ";".join(f"{a}__{b}" for a, b in q)
        num = ";".join(f"{a}__{numid.setdefault(b, 1000 + len(numid))}" for a, b in q)
        units.append({"taxid": t, "rank": q[-1][0], "numericLineage": num, "textLineage": text,
                      "accessions": [{"accession": f"NR_{t}.1", "oid": str(t)}]})
    return units


def taxonomy_json(units: List[dict]) -> dict:
    return {"blutilsVersion": "8.3.1", "ignoreTaxids": None, "replaceRank": None, "dropNonLinnaeanTaxonomies": False,
            "sourceDatabase": "/synthetic/db", "taxonomies": units}


def write_taxonomy(path: str, units: List[dict]) -> str:
    with open(path, "w") as f:
        json.dump(taxonomy_json(units), f)
    return path


def _fmt_pident(rng: random.Random, low: float = 60.0) -> str:
    v = rng.choice([100.0, 99.356, 98.927, 97.0, 96.999, 99.0, 92.0, 85.5, 80.001, 75.0, 60.0, 97.667, 98.333, 67.5])
    if rng.random() < 0.5:
        v = round(rng.uniform(low, 100.0), 3)
    s = f"{v:.3f}"
    if rng.random() < 0.3:
        s = s.rstrip("0").rstrip(".")
    return s


def random_blast(rng: random.Random, units: List[dict], n_queries: int = 30, max_hits: int = 12,
                 contiguous: bool = True, tie_rate: float = 0.6, low_pident: float = 60.0) -> bytes:
    taxids = [u["taxid"] for u in units]
    rows_by_q: List[List[str]] = []
    for qi in range(n_queries):
        q = rng.choice(["q%05d", "SRR1.%d_size_3", "draft-%d", "NR_%d.x"]) % qi
        nh = rng.randint(1, max_hits)
        base_bits = rng.choice([845, 833, 100, 84, 1200, 57])
        rows = []
        for h in range(nh):
            t = rng.choice(taxids[: max(3, len(taxids) // rng.choice([1, 2, 8]))]) if rng.random() < 0.7 else rng.choice(taxids)
            acc = f"NR_{rng.randint(100000, 100040)}.{rng.randint(1, 2)}"
            if rng.random() < tie_rate:
                bits = f"{base_bits}" if rng.random() < 0.7 else f"{base_bits}.{rng.randint(0, 9)}"
            else:
                bits = str(rng.randint(50, base_bits))
            if rng.random() < 0.05:
                bits = "%.3e" % float(bits)
            ln = rng.choice([455, 456, 1500, 200])
            rows.append("\t".join([q, acc, str(t), _fmt_pident(rng, low_pident), str(ln), str(rng.randint(0, 30)), str(rng.randint(0, 5)),
                                   "1", str(ln), str(rng.randint(1, 900)), str(rng.randint(901, 1800)),
                                   rng.choice(["0.0", "1e-50", "2.51e-117", "3.4", "1E-5", "5e+00"]), bits]))
        if rng.random() < 0.1 and rows:
            rows.append(rows[-1])  # exact duplicate row (exercises accessions dedup)
        rows_by_q.append(rows)
    if contiguous:
        lines = [r for rows in rows_by_q for r in rows]
    else:
        lines = [r for rows in rows_by_q for r in rows]
        # interleave: split some queries into several runs
        chunks = []
        for rows in rows_by_q:
            k = rng.randint(1, 3)
            cut = sorted(rng.sample(range(1, len(rows)), min(k - 1, max(0, len(rows) - 1)))) if len(rows) > 1 else []
            prev = 0
            for c in cut + [len(rows)]:
                chunks.append(rows[prev:c])
                prev = c
        rng.shuffle(chunks)
        # shuffling runs changes the relative order of a query's rows vs the file; that is fine (file order is what counts)
        lines = [r for ch in chunks for r in ch]
    text = "\n".join(lines)
    if rng.random() < 0.8:
        text += "\n"
    return text.encode()


def canon(results: List[dict]) -> List[dict]:
    """Sort by query bytes, drop runId."""
    out = []
    for r in results:
        r = dict(r)
        r.pop("runId", None)
        out.append(r)
    out.sort(key=lambda r: r["query"].encode())
    return out
