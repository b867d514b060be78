"""The drop-in contract itself: `blu blastn build-consensus` (reference ports/cli/src/cmds/blast/commands.rs:105-143,
cmds/blast/mod.rs:104-146) through the CLI shim, every output format, against the Python restatement of
write_blutils_output (core/src/use_cases/write_blutils_output.rs:126-248): pretty JSON to a file, compact JSON / JSONL /
YAML to stdout, byte for byte modulo the random runId."""
import json
import os
import random
import re
import subprocess

import pytest

from helpers import CUTOFFS_16S, random_blast, random_taxonomy, write_taxonomy

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EXE = os.path.join(ROOT, "blutils_b200", "blu")
UUID = re.compile(r"[0-9a-f]{8}-[0-9a-f]{4}-4[0-9a-f]{3}-[89ab][0-9a-f]{3}-[0-9a-f]{12}")


def _case(tmp_path, seed, numeric=False):
    import pyoracle as po

    for seed in range(seed, seed + 50):  # (a generated table may hit one of the reference's aborts: take the first that does not)
        rng = random.Random(seed)
        units = random_taxonomy(rng, n_leaves=40)
        text = random_blast(rng, units, n_queries=120)
        try:
            for lin in ("textLineage", "numericLineage"):
                for strategy in ("cautious", "relaxed"):
                    po.build_consensus_identities(text, {u["taxid"]: u[lin] for u in units}, "bacteria", strategy)
            break
        except po.DataError:
            continue
    tax_path = write_taxonomy(str(tmp_path / "db.blutils.json"), units)
    blast = tmp_path / "blast.out"
    blast.write_bytes(text)
    tax = po.load_taxonomy(tax_path, numeric)
    return str(blast), tax_path, text, tax


def _run(args, **kw):
    return subprocess.run([EXE] + args, check=True, capture_output=True, **kw)


@pytest.mark.parametrize("taxon,strategy,numeric", [("bacteria", "relaxed", False), ("fungi", "cautious", True), ("eukaryotes", "relaxed", False)])
def test_build_consensus_formats(tmp_path, taxon, strategy, numeric):
    import pyoracle as po

    blast, tax_path, text, tax = _case(tmp_path, 7 + len(taxon), numeric)
    want = po.build_consensus_identities(text, tax, taxon, strategy)
    base = ["--threads", "4", "blastn", "build-consensus", blast, "-t", tax_path, "--taxon", taxon, "--strategy", strategy] + (["-u"] if numeric else [])

    def with_run_id(run_id):
        return [dict([("runId", run_id)] + list(r.items())) for r in want]

    # pretty JSON to a file; the extension is forced to .json (write_blutils_output.rs:42-52)
    _run(base + ["--blutils-out-file", str(tmp_path / "res.out")])
    got = (tmp_path / "res.json").read_text()
    run_id = UUID.search(got).group(0)
    assert got == po.to_json_pretty({"results": with_run_id(run_id), "config": None})
    # compact JSON to stdout
    got = _run(base).stdout.decode()
    run_id = UUID.search(got).group(0)
    assert got == po.to_json_compact({"results": with_run_id(run_id), "config": None})
    # JSONL to stdout: the config line (`null`) first
    got = _run(base + ["--out-format", "jsonl"]).stdout.decode()
    run_id = UUID.search(got).group(0)
    assert got == "null\n" + po.results_to_jsonl(want, run_id)
    # JSONL to a file
    _run(base + ["--out-format=jsonl", "--blutils-out-file", str(tmp_path / "res2")])
    got = (tmp_path / "res2.jsonl").read_text()
    assert got == "null\n" + po.results_to_jsonl(want, UUID.search(got).group(0))
    # YAML to stdout and to a file (serde_yaml 0.9 block style)
    got = _run(base + ["--out-format", "yaml"]).stdout.decode()
    run_id = UUID.search(got).group(0)
    assert got == po.results_to_yaml(want, run_id)
    _run(base + ["--out-format", "yaml", "--blutils-out-file", str(tmp_path / "res3.txt")])
    got = (tmp_path / "res3.yaml").read_text()
    assert got == po.results_to_yaml(want, UUID.search(got).group(0))


def test_build_consensus_custom_cutoffs_and_errors(tmp_path):
    import pyoracle as po

    blast, tax_path, text, tax = _case(tmp_path, 31)
    y = tmp_path / "cut.yaml"
    y.write_text("domain: 50\nkingdom: 60\nphylum: 75\nclass: 80\norder: 85\nfamily: 92\ngenus: 97\nspecies: 99\n")
    want = po.build_consensus_identities(text, tax, "custom", "cautious", CUTOFFS_16S)
    got = _run(["blastn", "build-consensus", blast, "--tax-file", tax_path, "--taxon", "custom", "-c", str(y), "--strategy", "cautious",
                "--out-format", "jsonl"]).stdout.decode()
    assert got == "null\n" + po.results_to_jsonl(want, UUID.search(got).group(0))
    # --taxon custom without the file, a missing blast file, a missing taxonomy file: the reference panics (exit 101)
    for bad in (["blastn", "build-consensus", blast, "-t", tax_path, "--taxon", "custom", "--strategy", "cautious"],
                ["blastn", "build-consensus", str(tmp_path / "nope"), "-t", tax_path, "--taxon", "bacteria", "--strategy", "cautious"],
                ["blastn", "build-consensus", blast, "-t", str(tmp_path / "nope.json"), "--taxon", "bacteria", "--strategy", "cautious"]):
        p = subprocess.run([EXE] + bad, capture_output=True)
        assert p.returncode == 101 and b"panicked" in p.stderr
