"""One hit table over several GPUs of one box through the multi-device context (blu_ctx_create_multi; SURVEY 8e,
reference fan-out core/src/use_cases/build_consensus_identities/mod.rs:104-128): the table is cut by query range, every
GPU runs its shard on its own host thread, the parts come back as ONE result.  Needs >= 2 GPUs (gpurun --gpus 2);
the single-GPU box runs the one-shard variant only."""
import json
import os
import random
import subprocess

import pytest

from helpers import ROOT, device_sets, engine, hit_row, random_blast, random_taxonomy, synth_case, write_taxonomy
from oracle_ffi import Oracle

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("zipf", [False, True])
def test_sharded_table_equals_oracle(zipf, tmp_path):
    """host text and file, pooled strings and text references, whole-table checksum == oracle."""
    from oracle_ffi import checksum_jsonl

    ids, lin, text = synth_case(5000, 300 if zipf else 20000, 5000 if zipf else 50, zipf=zipf, seed=23)
    want, nq, nr = Oracle(ids, lin, "bacteria", "relaxed").run_raw(text)
    path = tmp_path / "blast.out"
    path.write_bytes(text)
    for devs in device_sets():
        for refs in (False, True):
            eng = engine("bacteria", "relaxed", chunk_bytes=1 << 20, devices=devs, text_refs=refs, lineages=(ids, lin))
            out = eng.run_host(text)
            assert len(out) == nq and out.n_rows == nr, (devs, refs)
            assert out.checksum() == checksum_jsonl(want), (devs, refs)
            assert out.jsonl() == want, (devs, refs)
            # the concatenated binary view: records of all parts, indices rebased
            recs = out.records()
            assert len(recs) == nq and all(r.status == 1 for r in recs)
            assert sorted(out.query_ids()) == sorted(json.loads(l)["query"].encode() for l in want.decode().splitlines()), (devs, refs)
            t = eng.timings()
            assert int(t["n_queries"]) == nq and int(t["text_bytes"]) == len(text)
            out.close()
            if not refs:
                out = eng.run_file(str(path))
                assert out.jsonl() == want, (devs, "file")
                out.close()
            eng.close()


def test_scattered_table_across_shards():
    """A query whose rows lie in two different shards: invisible to every single GPU's duplicate-id check, caught by the
    merged check on the first device; the table is regrouped and run again (the reference groups by HashMap, mod.rs:145,192)."""
    lin = ["d__bac;p__p1;c__c1", "d__bac;p__p1;c__c2", "d__bac;p__p2;c__c3"]
    ids = [1, 2, 3]
    rng = random.Random(5)
    rows = []
    for q in range(400):
        for h in range(rng.randint(1, 6)):
            rows.append(hit_row(f"q{q:04d}", f"A{h}.1", rng.choice(ids), "99.0", 100, "500" if h < 2 else "300"))
    rows.insert(3, hit_row("q0399", "Z.1", 3, "99.5", 100, "900"))  # a better hit of the LAST query, at the start of the file
    text = "".join(rows).encode()
    want = Oracle(ids, lin, "bacteria", "cautious").run_raw(text)[0]
    for devs in device_sets():
        eng = engine("bacteria", "cautious", devices=devs, lineages=(ids, lin))
        out = eng.run_host(text)
        assert out.jsonl() == want, devs
        assert int(eng.timings()["n_regrouped"]) == 2  # regrouped on the first GPU of the context
        out.close()
        eng.close()


def test_errors_and_tiny_tables_multi():
    """Fewer queries than GPUs (empty shards), and a data error in one shard fails the whole run."""
    from blutils_b200 import ConsensusPanic

    lin = ["d__bac;p__p1;c__c1"]
    one = hit_row("only", "A.1", 1, "99.0", 100, "500").encode()
    want = Oracle([1], lin, "bacteria", "cautious").run_raw(one)[0]
    for devs in device_sets():
        eng = engine("bacteria", "cautious", devices=devs, lineages=([1], lin))
        assert eng.run_host(one).jsonl() == want
        bad = "".join(hit_row(f"q{i}", "A.1", 1 if i != 777 else 42, "99.0", 100, "500") for i in range(1000)).encode()  # taxid 42 is unmapped
        with pytest.raises(ConsensusPanic):
            eng.run_host(bad)
        eng.close()


def test_cli_devices(tmp_path):
    """`blu blastn build-consensus --devices ...` (commands.rs:105-143 + the device list): same file as one GPU writes."""
    import pyoracle as po

    for seed in range(99, 140):  # (a generated table may hit one of the reference's aborts: take the first that does not)
        rng = random.Random(seed)
        units = random_taxonomy(rng, n_leaves=40)
        text = random_blast(rng, units, n_queries=300)
        try:
            po.build_consensus_identities(text, {u["taxid"]: u["textLineage"] for u in units}, "bacteria", "relaxed")
            break
        except po.DataError:
            continue
    tax_path = write_taxonomy(str(tmp_path / "db.blutils.json"), units)
    blast = tmp_path / "blast.out"
    blast.write_bytes(text)
    exe = os.path.join(ROOT, "blutils_b200", "blu")
    outs = []
    for devs in device_sets():
        o = tmp_path / ("out_" + "_".join(map(str, devs)))
        subprocess.run([exe, "blastn", "build-consensus", str(blast), "--tax-file", tax_path, "--taxon", "bacteria", "--strategy", "relaxed",
                        "--blutils-out-file", str(o), "--out-format", "jsonl", "--devices", ",".join(map(str, devs))], check=True)
        lines = open(str(o) + ".jsonl").read().splitlines()
        objs = [json.loads(l) for l in lines[1:]]
        for x in objs:
            x.pop("runId")
        outs.append(objs)
    assert all(o == outs[0] for o in outs)
