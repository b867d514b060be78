"""CPU-side checks of the product: the C-ABI library loads and exports every symbol include/blu_consensus.h
declares (no compute without a GPU: it must fail loudly), the host logic (taxonomy encoder, cutoff
interpolation, custom-cutoff file, JSON reader, decoder/writer) and the device-side per-row / per-query logic
compiled for the host (tests/csrc/sim_harness.cpp) agree with the oracle."""
import json
import os
import random
import re

import pytest

import pyoracle as po
import sim_ffi
from helpers import CUTOFFS_16S, KAT, ROOT, random_blast, random_taxonomy, same, write_taxonomy
from oracle_ffi import Oracle, OracleDataError


def test_header_symbols_exported():
    from blutils_b200 import _ffi

    hdr = open(os.path.join(ROOT, "include", "blu_consensus.h")).read()
    declared = set(re.findall(r"\b(blu_[a-z0-9_]+)\s*\(", hdr))
    assert declared, "no declarations found"
    lib = _ffi.lib()
    bound = {name for name, _, _ in _ffi.SYMBOLS}
    assert declared == bound, (declared ^ bound)
    for name in declared:
        assert hasattr(lib, name)
    assert lib.blu_abi_version() == 2


def test_no_gpu_is_loud():
    import torch

    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    from blutils_b200 import ConsensusEngine, ConsensusStrategy, CudaUnavailable, Taxon

    with pytest.raises(CudaUnavailable):
        ConsensusEngine(Taxon.Bacteria, ConsensusStrategy.Cautious)


def test_product_has_no_oracle_dependency():
    """The product tree must not reference the oracle or any CPU fallback."""
    pkg = os.path.join(ROOT, "blutils_b200")
    for dp, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cpp", ".cu", ".cuh", ".h")):
                txt = open(os.path.join(dp, f), errors="ignore").read()
                assert "oracle_ffi" not in txt and "pyoracle" not in txt and "blu_oracle" not in txt, f


@pytest.mark.parametrize("ranks,bact,cust", KAT)
def test_product_interpolation_kat(ranks, bact, cust):
    names = ranks.split()
    assert same(sim_ffi.interpolate(names, "bacteria"), [float(x) for x in bact])
    assert same(sim_ffi.interpolate(names, "custom", CUTOFFS_16S), [float(x) for x in cust])


def test_custom_cutoff_files(tmp_path):
    y = tmp_path / "c.yaml"
    y.write_text("domain: 50\nkingdom: 60\nphylum: 75\nclass: 80\norder: 85\nfamily: 92\ngenus: 97\nspecies: 99\n")
    assert sim_ffi.custom_cutoffs(str(y)) == CUTOFFS_16S == po.load_custom_cutoffs(str(y))
    y2 = tmp_path / "d.yaml"
    y2.write_text("# partial\n---\ndomain: 40\nspecies: 98   # trailing comment\ngenus: ~\n")
    assert sim_ffi.custom_cutoffs(str(y2)) == {"domain": 40, "kingdom": None, "phylum": None, "class": None, "order": None, "family": None,
                                               "genus": None, "species": 98}
    j = tmp_path / "c.json"
    j.write_text(json.dumps({"domain": 55, "species": 97, "family": None, "extra": 1}))
    assert sim_ffi.custom_cutoffs(str(j))["domain"] == 55 and sim_ffi.custom_cutoffs(str(j))["family"] is None
    for bad, body in (("m.yaml", "kingdom: 60\nspecies: 99\n"), ("r.yaml", "domain: 70000\nspecies: 99\n"), ("x.txt", "domain: 1\nspecies: 2\n"),
                      ("s.yaml", "domain: abc\nspecies: 2\n")):
        p = tmp_path / bad
        p.write_text(body)
        with pytest.raises(ValueError):
            sim_ffi.custom_cutoffs(str(p))
    with pytest.raises(ValueError):
        sim_ffi.custom_cutoffs(str(tmp_path / "missing.yaml"))


def test_taxonomy_json_reader(tmp_path):
    units = random_taxonomy(random.Random(3), n_leaves=20)
    p = write_taxonomy(str(tmp_path / "t.json"), units)
    assert sim_ffi.read_taxonomy_json(p) == len(units)
    doc = json.load(open(p))
    for drop in ("blutilsVersion", "sourceDatabase", "taxonomies"):
        d = dict(doc)
        del d[drop]
        q = tmp_path / f"no_{drop}.json"
        q.write_text(json.dumps(d))
        with pytest.raises(IOError):
            sim_ffi.read_taxonomy_json(str(q))
    d = json.loads(json.dumps(doc))
    del d["taxonomies"][0]["accessions"]
    (tmp_path / "noacc.json").write_text(json.dumps(d))
    with pytest.raises(IOError):
        sim_ffi.read_taxonomy_json(str(tmp_path / "noacc.json"))
    (tmp_path / "garbage.json").write_text("{not json")
    with pytest.raises(IOError):
        sim_ffi.read_taxonomy_json(str(tmp_path / "garbage.json"))
    with pytest.raises(IOError):
        sim_ffi.read_taxonomy_json(str(tmp_path / "nope.json"))
    # escapes + unknown keys + null options
    d = json.loads(json.dumps(doc))
    d["futureField"] = {"a": [1, 2, {"b": None}]}
    d["taxonomies"][0]["textLineage"] = "d__café;p__x\"y"
    (tmp_path / "esc.json").write_text(json.dumps(d))
    assert sim_ffi.read_taxonomy_json(str(tmp_path / "esc.json")) == len(units)


@pytest.mark.parametrize("seed", range(40))
def test_device_core_on_host_vs_oracle(seed):
    """blu_core.cuh (the code the kernels run per row / per query) + taxonomy encoder + decoder, compiled for the
    host, against the C++ oracle: identical JSONL, identical error class."""
    rng = random.Random(5000 + seed)
    units = random_taxonomy(rng, n_leaves=rng.choice([5, 20, 60]), shared_root=rng.random() < 0.9)
    text = random_blast(rng, units, n_queries=rng.choice([1, 10, 40]), contiguous=True, low_pident=rng.choice([60.0, 45.0]))
    for taxon in ("bacteria", "fungi", "custom"):
        for strategy in ("cautious", "relaxed"):
            for use_taxid in (False, True):
                custom = None
                if taxon == "custom":
                    custom = CUTOFFS_16S if seed % 3 else {"domain": 50, "species": 99, "genus": 95}
                lin = [(u["numericLineage"] if use_taxid else u["textLineage"]) for u in units]
                ids = [u["taxid"] for u in units]
                try:
                    want = Oracle(ids, lin, taxon, strategy, custom, threads=2).run_raw(text)[0]
                except OracleDataError:
                    want = None
                rc, got, err = sim_ffi.run(ids, lin, taxon, strategy, text, custom)
                if want is None:
                    assert rc == 2, err
                else:
                    assert rc == 0, err
                    assert got == want


def test_device_core_number_grammar():
    """Field grammar decisions of light_parse_row == the oracle's, plus the documented UNSUPPORTED range."""
    lin, ids = ["d__a;p__b"], [1]

    def row(pident="99.0", bits="50", ln="10", ev="0.0", mm="0"):
        return f"q\tacc\t1\t{pident}\t{ln}\t{mm}\t0\t1\t10\t1\t10\t{ev}\t{bits}\n".encode()

    ok = [row(), row(pident="99."), row(pident=".5e2"), row(bits="84.2"), row(bits="1.000e+02"), row(ev="1e-180"), row(ev="2.5E-7"),
          row(bits="0070"), row(pident="100"), row(mm="-3")]
    bad = [row(pident="99.0.1"), row(pident="."), row(pident="e5"), row(bits="5e"), row(bits="+5"), row(ln="1.5"), row(ln=""), row(ev="--1"),
           row(mm="1234567890123456789"), row(pident="nan"), row(bits="inf")]
    for t in ok:
        want = Oracle(ids, lin, "custom", "cautious", {"domain": 0, "species": 0}).run_raw(t)[0]
        rc, got, err = sim_ffi.run(ids, lin, "custom", "cautious", t, {"domain": 0, "species": 0})
        assert rc == 0 and got == want, (t, err)
    for t in bad:
        with pytest.raises(OracleDataError):
            Oracle(ids, lin, "bacteria", "cautious").run_raw(t)
        rc, _, _ = sim_ffi.run(ids, lin, "bacteria", "cautious", t)
        assert rc == 2, t
    # valid for the reference, outside the exactly-parsed range of the CUDA path: loud BLU_ERR_UNSUPPORTED (5)
    # ("1e30" as a bit score is an i64-range panic in the reference; here it is reported as UNSUPPORTED: loud either way)
    for t in (row(pident="99.12345678901234567890"), row(bits="123456789012345678e5"), row(bits="1e30")):
        rc, _, _ = sim_ffi.run(ids, lin, "bacteria", "cautious", t)
        assert rc == 5, t


def test_headers_hitless():
    lin, ids = ["d__a;p__b"], [1]
    text = b"q2\tacc\t1\t99.0\t10\t0\t0\t1\t10\t1\t10\t0.0\t50\n"
    want = Oracle(ids, lin, "bacteria", "cautious").run_raw(text, headers=["q1", "q2", "q3"])[0]
    rc, got, _ = sim_ffi.run(ids, lin, "bacteria", "cautious", text, headers=["q1", "q2", "q3"])
    assert rc == 0 and got == want
