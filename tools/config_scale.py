#!/usr/bin/env python
"""One pass for K consensus configurations (blu_consensus_run_*_configs) against K separate runs of the same table.

The table is C2-shaped (blu_synth: 120 k queries x 50 hits, 30 k taxa, ~458 MB).  The configurations are the eight of the
reference's consensus knobs -- cautious / relaxed x bacteria / custom 16S cutoffs x text / numeric lineages -- and the first
K of them are used, for K = 1, 2, 4, 8.  Per K and path, the grouped call and the K separate calls alternate, `--reps`
times each, after one warm-up of both:

  * device-resident: ms per pass (host clock around the synchronous call; the results stay on the device and are freed)
  * run_file from tmpfs (/dev/shm): wall ms
  * run_host from pinned memory (blu_host_alloc): wall ms

Every configuration's checksum from the grouped call must equal its separate run's.  The GPU name, power limit and SM
clock are read in the same process.  Measurement tool, not part of pytest / bench.py; prints one JSON object per line.

  python tools/config_scale.py --reps 5 > profiles/r03_config_scale.txt
"""
import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

YAML16S = dict(domain=50, kingdom=60, phylum=75, class_=80, order=85, family=92, genus=97, species=99)


def device_line():
    import torch

    try:
        smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:  # (the numbers below still say which GPU took them)
        smi = f"nvidia-smi unavailable: {e}"
    return {"device": torch.cuda.get_device_name(0), "nvidia_smi": smi}


def engines(w):
    from blutils_b200 import ConsensusEngine, ConsensusStrategy, CustomTaxon, Taxon

    lins = {numeric: w.lineages(numeric=numeric) for numeric in (False, True)}
    out = []
    for numeric in (False, True):
        for taxon in (Taxon.Bacteria, Taxon.Custom):
            for strategy in (ConsensusStrategy.Cautious, ConsensusStrategy.Relaxed):
                e = ConsensusEngine(taxon, strategy, numeric, CustomTaxon(**YAML16S) if taxon == Taxon.Custom else None)
                ids, off, blob = lins[numeric]
                e.load_taxonomy_raw(ids.ctypes.data, off.ctypes.data, blob.ctypes.data, len(ids))
                out.append(e)
    return out


def timed(fn):
    import torch

    torch.cuda.synchronize()
    t0 = time.perf_counter()
    res = fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) * 1e3, res


def stats(v):
    return {"median_ms": round(statistics.median(v), 3), "min_ms": round(min(v), 3), "max_ms": round(max(v), 3)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--queries", type=int, default=120_000)
    ap.add_argument("--hits", type=int, default=50)
    ap.add_argument("--taxa", type=int, default=30_000)
    ap.add_argument("--ks", default="1,2,4,8")
    ap.add_argument("--reps", type=int, default=5)
    a = ap.parse_args()

    import torch

    from blutils_b200 import _ffi, run_device_resident_configs, run_file_configs, run_host_configs
    from blutils_b200.synth import SynthWorkload

    if not torch.cuda.is_available():
        raise SystemExit("config_scale.py measures on a CUDA device; none is available")
    print(json.dumps(device_line()), flush=True)
    w = SynthWorkload(a.taxa, seed=20261020)
    text = w.hits(0, a.queries, a.hits)
    n = len(text)
    engs = engines(w)

    dev = torch.zeros((n + 255) // 128 * 128, dtype=torch.uint8, device="cuda")
    dev[:n] = torch.frombuffer(bytearray(text), dtype=torch.uint8).cuda()
    stream = torch.cuda.current_stream().cuda_stream
    lib = _ffi.lib()
    pinned = lib.blu_host_alloc(n)
    C.memmove(pinned, text, n)
    shm = "/dev/shm" if os.path.isdir("/dev/shm") else None
    fd, path = tempfile.mkstemp(suffix=".blast.out", dir=shm)
    with os.fdopen(fd, "wb") as f:
        f.write(text)
    del text
    print(json.dumps({"table_bytes": n, "queries": a.queries, "hits_per_query": a.hits, "taxa": a.taxa, "file": path}), flush=True)

    paths = {
        "resident": (lambda es: run_device_resident_configs(es, dev.data_ptr(), n, stream),
                     lambda e: e.run_device_resident(dev.data_ptr(), n, stream)),
        "file": (lambda es: run_file_configs(es, path), lambda e: e.run_file(path)),
        "host_pinned": (lambda es: run_host_configs(es, pinned, n), lambda e: e.run_host(pinned, n)),
    }

    def close(outs):
        for o in outs:
            o.close()

    try:
        for k in [int(x) for x in a.ks.split(",")]:
            es = engs[:k]
            for name, (grouped, single) in paths.items():
                # correctness first (not timed): every configuration equals its separate run
                g = grouped(es)
                s = [single(e) for e in es]
                for o in g + s:
                    if name == "resident":
                        o.download()
                ok = all(x.checksum() == y.checksum() and len(x) == len(y) for x, y in zip(g, s))
                close(g), close(s)
                if not ok:
                    raise SystemExit(f"K={k} {name}: a grouped result differs from its separate run")
                tg, ts = [], []
                for _ in range(a.reps):  # alternated
                    ms, outs = timed(lambda: grouped(es))
                    t = engs[0].timings()
                    close(outs)
                    tg.append(ms)
                    ms, outs = timed(lambda: [single(e) for e in es])
                    close(outs)
                    ts.append(ms)
                print(json.dumps({"k": k, "path": name, "checksums_equal": ok, "grouped": stats(tg), "separate": stats(ts),
                                  "speedup_median": round(statistics.median(ts) / statistics.median(tg), 3),
                                  "grouped_kernel_ms": {"tile": round(t["ms_tile_kernel"], 3), "longrun": round(t["ms_longrun_kernel"], 3),
                                                        "post": round(t["ms_gather_kernel"], 3)},
                                  "grouped_launches": int(t["n_kernel_launches"]), "grouped_h2d_bytes": int(t["h2d_bytes"])}), flush=True)
    finally:
        os.unlink(path)
        lib.blu_host_free(pinned)
        for e in engs:
            e.close()


if __name__ == "__main__":
    main()
