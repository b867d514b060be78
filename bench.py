#!/usr/bin/env python
"""bench.py -- consensus queries/s of the blutils consensus-identity hot path on B200.

One hit table, sharded by query range over the ranks (one process per GPU, no data-path collective; SURVEY 8e).
A "step" is one pass of the hot path over the rank's shard.

  --config c2 (default)  BASELINE configs[1]: synthetic 16S amplicon run, 1 M queries x 50 hits PER GPU (weak scaling: the
                         table grows with the GPUs), 30 k-taxon lineage map, --taxon custom with the cutoffs of
                         assets/custom-taxon-cutoffs-bacteria-16S.yaml, strategy relaxed
  --config c3            configs[2]: ONE table of 10 M queries x 100 hits, 2 M-taxon map, default (bacteria) cutoffs; strong scaling
  --config c4            configs[3]: ONE table of 2.4 M queries, Zipf(1.1) on [1, 5000] hits (~10^9 rows); strong scaling
  --config c5            configs[4]: 100 M queries x 50 hits streamed from pinned host memory; strong scaling.  A rank keeps a
                         block of --host-gb of its shard in pinned memory and streams it as many times as its shard is long
  --scaling weak|strong  overrides the config's default; --queries overrides its size (total for strong, per GPU for weak)

  value : device-resident throughput -- text already in HBM -> consensus records in HBM (SURVEY 8d(i));
          blu_consensus_run_device_resident: 5 kernel launches and one host synchronisation per step, nothing but the
          counters crosses PCIe.  `value_with_result_download` is the same step with the records, beans, accession
          references and strings downloaded to pinned host memory (blu_consensus_run_device).
  e2e   : the same metric through the reference-facing C-ABI call with the text in pinned HOST memory
          (blu_consensus_run_host: chunked H2D + kernels + result D2H inside the timed region)
  roofline : the tile kernel; achieved = algorithmic bytes (text + result records + lineage tables) / its CUDA-event
          duration measured in this run, against MEASURED_PEAKS.json hbm_gbs
  cpu_baseline : the C++ port of the reference (oracle/) timed on the host cores on a bounded sample of the workload
  verified : every rank compares the first 20 000 queries of its shard's timed output with the oracle (outside the timed
          region); a mismatch fails the run
`--impl reference` times that CPU port alone (the reference is Rust + polars and cannot be built in this image).
`--dump-outputs DIR` writes the result of the last timed step (the headline arm: device-resident, or C5's streamed run) to
DIR/*.npy in a canonical, sampled form (dump_outputs); the inputs are seeded, so two builds can be compared file by file.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

BASE_SEED = 20261018
CUSTOM = {"domain": 50, "kingdom": 60, "phylum": 75, "class": 80, "order": 85, "family": 92, "genus": 97, "species": 99}
CPU_SAMPLE_Q = 100_000
VERIFY_Q = 20_000
# --dump-outputs: queries sampled from the result, and at most this many of their beans / accession references
# (float64 columns: 16 x 64 Ki + 4 x 512 Ki + 3 x 1 Mi values = 48 MiB at most)
DUMP_QUERIES = 1 << 16
DUMP_BEANS = 1 << 19
DUMP_ACCESSIONS = 1 << 20

CONFIGS = {
    "c2": dict(cid=2, queries=1_000_000, hits=50, zipf=False, taxa=30_000, taxon="custom", strategy="relaxed", scaling="weak",
               what="C2 synthetic 16S amplicon run: {q} queries x 50 hits {per}, 30000-taxon lineage map, --taxon custom "
                    "(custom-taxon-cutoffs-bacteria-16S.yaml values), strategy relaxed"),
    "c3": dict(cid=3, queries=10_000_000, hits=100, zipf=False, taxa=2_000_000, taxon="bacteria", strategy="cautious", scaling="strong",
               what="C3: one table of {q} queries x 100 hits {per}, 2000000-taxon lineage map, default (bacteria) cutoffs, strategy cautious"),
    "c4": dict(cid=4, queries=2_400_000, hits=5000, zipf=True, taxa=2_000_000, taxon="bacteria", strategy="cautious", scaling="strong",
               what="C4: one table of {q} queries with Zipf(1.1) hit counts on [1, 5000] {per}, 2000000-taxon lineage map, default "
                    "(bacteria) cutoffs, strategy cautious"),
    "c5": dict(cid=5, queries=100_000_000, hits=50, zipf=False, taxa=2_000_000, taxon="bacteria", strategy="cautious", scaling="strong",
               what="C5: {q} queries x 50 hits {per} streamed from pinned host memory, 2000000-taxon lineage map, default (bacteria) cutoffs, "
                    "strategy cautious"),
}


def env_int(k, d):
    try:
        return int(os.environ.get(k, d))
    except ValueError:
        return d


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""

    def __init__(self, gpu_index: int):
        self.rows = []
        self.proc = None
        self.gpu = gpu_index
        self._t = None

    def start(self):
        q = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
            "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except OSError:
            self.proc = None
            return
        self._t = threading.Thread(target=self._read, daemon=True)
        self._t.start()

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[1]))
                mx.append(float(r[2]))
            except (ValueError, IndexError):
                continue
            for i, n in enumerate(names):
                if len(r) > 4 + i and r[4 + i].lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons),
                "samples": len(sm)}


def lineage_strings(lineages):
    ids, off, blob = lineages
    return [bytes(blob[int(off[i]):int(off[i + 1])]).decode() for i in range(len(ids))]


def make_oracle(cfg, lineages, threads):
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    from oracle_ffi import Oracle

    ids = lineages[0]
    return Oracle(ids.tolist(), lineage_strings(lineages), cfg["taxon"], cfg["strategy"], CUSTOM if cfg["taxon"] == "custom" else None, threads=threads)


def cpu_reference(cfg, w, lineages, q_sample: int, steps: int, warmup: int, q_begin: int = 0):
    """Times the CPU port of the reference (oracle/blu_oracle.cpp, all host threads) on a bounded sample."""
    try:
        os.sched_setaffinity(0, range(os.cpu_count() or 1))  # the CPU arm may use every core of the box
    except OSError:
        pass
    cores = len(os.sched_getaffinity(0))
    orc = make_oracle(cfg, lineages, cores)
    text = w.hits(q_begin, q_sample, cfg["hits"], zipf=cfg["zipf"])
    times = []
    nq = nr = 0
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        _, nq, nr = orc.run_raw(text)
        dt = time.perf_counter() - t0
        if i >= warmup:
            times.append(dt)
    t = sum(times) / len(times)
    return {"value": nq / t, "unit": "queries/s", "cores": cores, "kind": "port",
            "sample": f"first {q_sample} queries of the table ({nr} rows, {len(text) / 1e6:.0f} MB text), {len(times)} pass(es), {cores} threads; "
                      f"C++ restatement of blutils 8.3.1 (Rust+polars reference not buildable here)",
            "rows_per_s": nr / t, "ms_per_pass": t * 1e3}, t


def generate_shard(w, cfg, q_begin, n_queries, pinned, cap, dbuf, host_keep_bytes, block_q):
    """Generates queries [q_begin, q_begin + n_queries) block by block into the pinned buffer and uploads them into the device
    tensor `dbuf`.  The pinned buffer keeps the first `host_keep_bytes` (rounded up to whole blocks) of the shard for the
    end-to-end arm; later blocks only pass through the scratch area behind that prefix.
    Returns (shard bytes, shard rows, host bytes kept, host queries kept, host rows kept)."""
    import torch

    total = rows = 0
    host_bytes = host_q = host_rows = 0
    keeping = True
    q = 0
    while q < n_queries:
        nq = min(block_q, n_queries - q)
        at = host_bytes
        nbytes, nrows = w.hits_into(pinned + at, cap - at, q_begin + q, nq, cfg["hits"], zipf=cfg["zipf"])
        if total + nbytes > dbuf.numel():
            raise MemoryError("device text buffer too small for the generated shard")
        view = (C.c_uint8 * nbytes).from_address(pinned + at)
        dbuf[total:total + nbytes].copy_(torch.frombuffer(view, dtype=torch.uint8))
        torch.cuda.synchronize()
        if keeping:
            host_bytes += nbytes
            host_q += nq
            host_rows += nrows
            keeping = host_bytes < host_keep_bytes
        total += nbytes
        rows += nrows
        q += nq
    return total, rows, host_bytes, host_q, host_rows


def _ranges(starts, counts):
    """Concatenation of arange(s, s + n) over (starts, counts)."""
    import numpy as np

    counts = counts.astype(np.int64)
    ends = np.cumsum(counts)
    return np.repeat(starts.astype(np.int64) - (ends - counts), counts) + np.arange(int(ends[-1]) if len(ends) else 0, dtype=np.int64)


def dump_outputs(out, directory):
    """Writes a result as float64 .npy files: its sizes and checksum, and a seeded sample of its queries with their records,
    beans and accession references.  The kernels place records, beans and strings in an order that differs from run to run,
    so the dump is canonical: queries sorted by id, beans and accessions in the order their query lists them, strings as
    (CRC-32, length).  Two builds given the same arguments write the same files."""
    import zlib

    import numpy as np

    from blutils_b200 import _ffi

    out.download()
    lib, h = _ffi.lib(), out._h
    nq, nb, na = len(out), lib.blu_result_num_beans(h), lib.blu_result_num_accessions(h)
    plen = C.c_uint64()
    pptr = lib.blu_result_pool(h, C.byref(plen))
    pool = np.ctypeslib.as_array(C.cast(pptr, C.POINTER(C.c_uint8)), shape=(plen.value,)) if plen.value else np.zeros(0, np.uint8)
    recs = np.ctypeslib.as_array(lib.blu_result_records(h), shape=(nq,)) if nq else np.zeros(0, np.dtype(_ffi.blu_record))
    beans = np.ctypeslib.as_array(C.cast(lib.blu_result_beans(h), C.POINTER(_ffi.blu_bean)), shape=(nb,)) if nb else np.zeros(0, np.dtype(_ffi.blu_bean))
    accs = np.ctypeslib.as_array(C.cast(lib.blu_result_accessions(h), C.POINTER(C.c_uint64)), shape=(na,)) if na else np.zeros(0, np.uint64)

    ids = [pool[o:o + n].tobytes() for o, n in zip(recs["query_off"].tolist(), recs["query_len"].tolist())]
    by_id = np.array(sorted(range(nq), key=ids.__getitem__), dtype=np.int64)
    rank = np.sort(np.random.default_rng(BASE_SEED).choice(nq, size=min(nq, DUMP_QUERIES), replace=False))
    r = recs[by_id[rank]]
    cols = {"query_rank": rank, "query_crc32": [zlib.crc32(ids[i]) for i in by_id[rank].tolist()], "keep_mask_lo": r["keep_mask"] & 0xFFFFFFFF,
            "keep_mask_hi": r["keep_mask"] >> 32}
    for f in ("query_len", "n_rows", "status", "single_match", "mutated", "perc_identity", "bit_score", "ref_lineage", "reached_pos",
              "allowed_pos", "bean_level", "n_beans"):
        cols[f] = r[f]
    # beans of the sampled queries, query by query (bean_query: index into the sample)
    bean_query = np.repeat(np.arange(len(r)), r["n_beans"].astype(np.int64))[:DUMP_BEANS]
    b = beans[_ranges(r["bean_base"], r["n_beans"])[:DUMP_BEANS]]
    cols.update(bean_query=bean_query, bean_first_lineage=b["first_lineage"], bean_occurrences=b["occurrences"], bean_n_acc=b["n_acc"])
    # their accession references (acc_begin is relative to the query's acc_base), bean by bean
    acc_bean = np.repeat(np.arange(len(b)), b["n_acc"].astype(np.int64))[:DUMP_ACCESSIONS]
    a = accs[_ranges(r["acc_base"][bean_query].astype(np.int64) + b["acc_begin"], b["n_acc"])[:DUMP_ACCESSIONS]]
    a_off, a_len = (a >> 16).tolist(), (a & 0xFFFF).tolist()
    cols.update(accession_bean=acc_bean, accession_crc32=[zlib.crc32(pool[o:o + n].tobytes()) for o, n in zip(a_off, a_len)], accession_len=a_len)
    ck = out.checksum()
    cols.update(result_counts=[nq, out.n_rows, nb, na], result_checksum=[ck & 0xFFFFFFFF, ck >> 32])
    os.makedirs(directory, exist_ok=True)
    for name, v in cols.items():
        np.save(os.path.join(directory, name + ".npy"), np.asarray(v, dtype=np.float64))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default="c2", choices=sorted(CONFIGS))
    ap.add_argument("--scaling", default=None, choices=["weak", "strong"])
    ap.add_argument("--queries", type=int, default=None, help="queries of the table (strong scaling) / per GPU (weak scaling)")
    ap.add_argument("--hits", type=int, default=None)
    ap.add_argument("--taxa", type=int, default=None)
    ap.add_argument("--host-gb", type=float, default=8.0, help="pinned host text kept per rank for the end-to-end arm")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-verify", action="store_true")
    ap.add_argument("--no-file-arm", action="store_true", help="skip the blu_consensus_run_file timing (the call the CLI makes)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the timed path computed in its last step to DIR/<name>.npy (see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the results of the CUDA path (--impl b200)")

    cfg = dict(CONFIGS[args.config])
    if args.hits:
        cfg["hits"] = args.hits
    if args.taxa:
        cfg["taxa"] = args.taxa
    if args.queries:
        cfg["queries"] = args.queries
    scaling = args.scaling or cfg["scaling"]
    seed = BASE_SEED + cfg["cid"]  # base seed + config id (SURVEY 8d)

    rank = env_int("RANK", 0)
    world = env_int("WORLD_SIZE", 1)
    local_rank = env_int("LOCAL_RANK", 0)
    dump_dir = args.dump_outputs
    if dump_dir and world > 1:
        dump_dir = os.path.join(dump_dir, f"rank{rank}")
    if scaling == "weak":
        q_rank, q_begin, q_table = cfg["queries"], rank * cfg["queries"], world * cfg["queries"]
    else:
        q_table = cfg["queries"]
        q_begin = q_table * rank // world
        q_rank = q_table * (rank + 1) // world - q_begin
    per = f"per GPU ({world} GPU(s): {q_table} queries)" if scaling == "weak" else f"sharded by query range over {world} GPU(s)"
    config = {"workload": cfg["what"].format(q=cfg["queries"], per=per), "config": args.config, "queries_table": q_table,
              "queries_per_gpu": q_rank, "hits_per_query": cfg["hits"], "hit_distribution": "zipf(1.1)" if cfg["zipf"] else "fixed", "taxa": cfg["taxa"],
              "sharding": f"query-range x{world}, no collective", "l2_policy": "input (GBs) larger than the 126 MB L2; no flush needed"}

    if args.impl == "reference":
        if rank != 0:
            return
        from blutils_b200.synth import SynthWorkload

        w = SynthWorkload(cfg["taxa"], seed=seed)
        sample = min(q_rank, CPU_SAMPLE_Q if not cfg["zipf"] else CPU_SAMPLE_Q // 8)
        base, t = cpu_reference(cfg, w, w.lineages(False), sample, args.steps, min(args.warmup, 1))
        line = {"impl": "reference", "run_info": {"reference_sample": base["sample"]}, "metric": "consensus_queries_per_s", "value": base["value"], "unit": "queries/s", "n_gpus": args.gpus,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": t * 1e3, "higher_is_better": True, "scaling": scaling,
                "vs_baseline": None, "dtype": "u8", "data": "synthetic", "config": config, "cpu_baseline": base,
                "hit_rows_per_s": base["rows_per_s"],
                "e2e": {"value": base["value"], "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        print(json.dumps(line))
        return

    import torch
    import torch.distributed as dist

    from blutils_b200 import _ffi, ConsensusEngine, ConsensusStrategy, CustomTaxon, Taxon
    from blutils_b200.synth import SynthWorkload

    torch.cuda.set_device(local_rank)
    run_info = {}  # (what differs from run to run stays out of `config`: both arms print the same config)
    # keep this rank's threads and its pinned staging memory on the NUMA node of its GPU (one PCIe link per GPU)
    try:
        import pynvml

        pynvml.nvmlInit()
        pynvml.nvmlDeviceSetCpuAffinity(pynvml.nvmlDeviceGetHandleByIndex(local_rank))
        run_info["cpu_affinity"] = f"{len(os.sched_getaffinity(0))} cpus (NVML ideal affinity of GPU {local_rank})"
    except Exception as ex:  # noqa: BLE001
        run_info["cpu_affinity"] = f"not set ({type(ex).__name__})"
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def reduce(x: float, op) -> float:
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=op)
        return float(t.item())

    def max_over_ranks(x):
        return reduce(x, dist.ReduceOp.MAX if world > 1 else None)

    def sum_over_ranks(x):
        return reduce(x, dist.ReduceOp.SUM if world > 1 else None)

    def every_rank(x: float):
        """x of every rank, in rank order (evidence for what bounds a multi-GPU number: the slowest rank sets the time)"""
        if world == 1:
            return [x]
        t = torch.zeros(world, dtype=torch.float64, device="cuda")
        t[rank] = x
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return [float(v) for v in t.tolist()]

    def min_over_ranks(x):
        return reduce(x, dist.ReduceOp.MIN if world > 1 else None)

    # ---------------- the table: this rank's shard, in HBM and (a prefix of it) in pinned host memory ---------------------
    w = SynthWorkload(cfg["taxa"], seed=seed)
    lineages = w.lineages(numeric=False)
    ids, off, blob = lineages
    est_rows = q_rank * cfg["hits"] if not cfg["zipf"] else q_rank * 520
    est_bytes = est_rows * 80 + (1 << 20)
    streamed_only = args.config == "c5"
    host_keep = int(args.host_gb * (1 << 30))
    block_q = max(1, min(q_rank, 100_000 if not cfg["zipf"] else 20_000))
    block_cap = block_q * (cfg["hits"] * 84 if not cfg["zipf"] else 1200 * 84) + (1 << 20)
    cap = min(est_bytes, host_keep + block_cap) + 2 * block_cap
    pinned = _ffi.lib().blu_host_alloc(cap)
    if not pinned:
        raise MemoryError("pinned allocation failed")
    dbuf = None
    t_gen = time.perf_counter()
    if not streamed_only:
        dbuf = torch.empty((est_bytes + 255) // 128 * 128, dtype=torch.uint8, device="cuda")
        nbytes, nrows, host_bytes, host_q, host_rows = generate_shard(w, cfg, q_begin, q_rank, pinned, cap, dbuf, host_keep, block_q)
    else:
        # C5: only the block that fits the host buffer is generated; the shard is that block streamed `passes` times
        nbytes = nrows = 0
        host_q = max(1, min(q_rank, int(host_keep // (cfg["hits"] * 78))))
        host_bytes, host_rows = w.hits_into(pinned, cap, q_begin, host_q, cfg["hits"], zipf=cfg["zipf"])
    run_info["generate_s"] = round(time.perf_counter() - t_gen, 1)

    # custom cutoffs go through the YAML path (CustomTaxon::from_file semantics)
    custom = None
    if cfg["taxon"] == "custom":
        with tempfile.NamedTemporaryFile("w", suffix=".yaml", delete=False) as f:
            for k, v in CUSTOM.items():
                f.write(f"{k}: {v}\n")
            ypath = f.name
        custom = CustomTaxon.from_file(ypath)
        os.unlink(ypath)
    taxon = {"custom": Taxon.Custom, "bacteria": Taxon.Bacteria}[cfg["taxon"]]
    strategy = {"relaxed": ConsensusStrategy.Relaxed, "cautious": ConsensusStrategy.Cautious}[cfg["strategy"]]
    eng = ConsensusEngine(taxon, strategy, False, custom, device=local_rank)
    eng.load_taxonomy_raw(ids.ctypes.data, off.ctypes.data, blob.ctypes.data, len(ids))
    stream = torch.cuda.current_stream().cuda_stream

    line_extra = {}
    clocks = None
    launches = 0
    roof = None
    verified = None
    if not streamed_only:
        # ---------------- device-resident arm: text in HBM -> records in HBM ------------------------------------------------
        sampler = ClockSampler(local_rank)
        if rank == 0:
            sampler.start()  # spans warm-up + timed region; the median is taken over samples under load
        for _ in range(args.warmup):
            eng.run_device_resident(dbuf.data_ptr(), nbytes, stream).close()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        tile_ms, long_ms, post_ms = [], [], []
        nq = 0
        res_bytes = tax_bytes = 0
        last = None
        e0.record()
        for i in range(args.steps):
            out = eng.run_device_resident(dbuf.data_ptr(), nbytes, stream)
            t = eng.timings()
            tile_ms.append(t["ms_tile_kernel"])
            long_ms.append(t["ms_longrun_kernel"])
            post_ms.append(t["ms_gather_kernel"])
            launches += int(t["n_kernel_launches"])
            nq = len(out)
            res_bytes, tax_bytes = int(t["result_bytes"]), int(t["taxonomy_bytes"])
            if i + 1 == args.steps:
                last = out  # the timed output: verified below
            else:
                out.close()
        e1.record()
        barrier()
        clocks = sampler.stop() if rank == 0 else None
        dev_ms = max_over_ranks(e0.elapsed_time(e1)) / args.steps
        total_q = sum_over_ranks(float(nq))
        total_rows = sum_over_ranks(float(nrows))
        total_bytes = sum_over_ranks(float(nbytes))

        # ---------------- verification of the timed output (outside the timed region) -------------------------------------
        if not args.no_verify:
            vq = min(VERIFY_Q if not cfg["zipf"] else VERIFY_Q // 4, q_rank)
            got = last.download().jsonl(head=vq)
            want = make_oracle(cfg, lineages, len(os.sched_getaffinity(0))).run_raw(w.hits(q_begin, vq, cfg["hits"], zipf=cfg["zipf"]))[0]
            ok = 1.0 if got == want else 0.0
            all_ok = min_over_ranks(ok)
            verified = {"queries_per_shard": vq, "shards": world, "what": "first queries of every shard's timed output == oracle, byte for byte (canonical JSONL)",
                        "ok": bool(all_ok == 1.0)}
            if all_ok != 1.0:
                if rank == 0:
                    print(json.dumps({"error": "timed output differs from the oracle", "verified": verified}))
                sys.exit(3)
        if dump_dir:
            dump_outputs(last, dump_dir)
        last.close()

        # ---------------- the same step with the result downloaded to pinned host memory ----------------------------------
        for _ in range(max(1, args.warmup // 2)):
            eng.run_device(dbuf.data_ptr(), nbytes, stream).close()
        barrier()
        dl_steps = max(2, min(args.steps, 5))
        d2h_dev = 0
        e0.record()
        for _ in range(dl_steps):
            out = eng.run_device(dbuf.data_ptr(), nbytes, stream)
            d2h_dev = int(eng.timings()["d2h_bytes"])
            out.close()
        e1.record()
        barrier()
        dl_ms = max_over_ranks(e0.elapsed_time(e1)) / dl_steps
        line_extra["value_with_result_download"] = {"value": total_q / (dl_ms * 1e-3), "unit": "queries/s", "ms_per_step": dl_ms,
                                                    "d2h_bytes_per_step": d2h_dev, "d2h_bytes_per_query": d2h_dev / max(nq, 1), "steps": dl_steps}

        # ---------------- roofline of the dominant kernel ---------------------------------------------------------------------
        peaks = {}
        pth = os.path.join(ROOT, "MEASURED_PEAKS.json")
        if os.path.exists(pth):
            peaks = json.load(open(pth))
        peak = float(peaks.get("hbm_gbs", 6650.0))
        peak_src = "MEASURED_PEAKS.json hbm_gbs (measured)" if peaks else "B200_PROFILING.md fallback 6650 GB/s"
        # SURVEY 8d: B_text + B_out (+ B_tax, which the consensus kernel reads, not this one: reported beside, not added)
        algo_bytes = nbytes + res_bytes
        traffic = None
        for name in ("r02_tile_kernel_traffic.json", "r01_tile_kernel_traffic.json"):
            tpath = os.path.join(ROOT, "profiles", name)
            if os.path.exists(tpath):
                tj = json.load(open(tpath))
                if int(tj.get("text_bytes", -1)) == int(nbytes):
                    traffic = int(tj["dram_read_bytes"] + tj["dram_write_bytes"])  # of ONE launch, like `achieved`
                    break
        tile_avg = sum(tile_ms) / len(tile_ms)
        achieved = algo_bytes / (tile_avg * 1e-3) / 1e9 if tile_avg > 0 else 0.0
        roof = {"bound": "hbm", "kernel": "tile_kernel", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": traffic, "peak_source": peak_src, "algorithmic_bytes_per_launch": int(algo_bytes), "ms_per_launch": tile_avg,
                "launches_per_step": 1, "kernel_share_of_step": tile_avg / dev_ms if dev_ms else None, "taxonomy_bytes_not_counted": tax_bytes,
                "ms_longrun_kernel": sum(long_ms) / len(long_ms), "ms_post_pass_kernels": sum(post_ms) / len(post_ms),
                "whole_step_frac": (total_bytes / world) / (dev_ms * 1e-3) / 1e9 / peak if dev_ms else None}
    else:
        dev_ms = None
        total_q = total_rows = total_bytes = 0.0

    # ---------------- end-to-end arm: pinned host text through the C ABI ------------------------------------------------
    passes = 1
    if streamed_only:
        passes = max(1, -(-q_rank // host_q))  # the shard = the pinned block streamed this many times
    for _ in range(max(1, args.warmup // 2)):
        eng.run_host(pinned, host_bytes).close()
    barrier()
    e2e_steps = args.steps
    t0 = time.perf_counter()
    d2h = 0
    e2e_launches = 0
    last = None
    for i in range(e2e_steps):
        for _p in range(passes):
            out = eng.run_host(pinned, host_bytes)
            tm = eng.timings()
            d2h = int(tm["d2h_bytes"])
            e2e_launches += int(tm["n_kernel_launches"])
            if streamed_only and dump_dir and i + 1 == e2e_steps and _p + 1 == passes:
                last = out  # C5's timed output
            else:
                out.close()
    torch.cuda.synchronize()
    e2e_own = time.perf_counter() - t0
    if last is not None:
        dump_outputs(last, dump_dir)
        last.close()
    e2e_s = max_over_ranks(e2e_own) / e2e_steps
    e2e_per_rank = every_rank(e2e_own / e2e_steps * 1e3)
    barrier()
    e2e_q = sum_over_ranks(float(host_q * passes))
    e2e_rows = sum_over_ranks(float(host_rows * passes))
    e2e_bytes = sum_over_ranks(float(host_bytes * passes))
    # ---------------- the same from a file (tmpfs), the call `blu blastn build-consensus` makes -------------------------------
    e2e_file = None
    if not args.no_file_arm and not streamed_only and os.path.isdir("/dev/shm"):
        fpath = f"/dev/shm/blu_bench_{os.getpid()}_{rank}.out"
        try:
            with open(fpath, "wb") as fh:
                fh.write((C.c_uint8 * host_bytes).from_address(pinned))
            eng.run_file(fpath).close()
            barrier()
            t0 = time.perf_counter()
            fsteps = max(1, min(args.steps, 3))
            for _ in range(fsteps):
                eng.run_file(fpath).close()
            file_s = max_over_ranks(time.perf_counter() - t0) / fsteps
            e2e_file = {"value": e2e_q / file_s, "unit": "queries/s", "ms_per_step": file_s * 1e3, "text_gb_per_s": e2e_bytes / file_s / 1e9,
                        "what": "blu_consensus_run_file on a tmpfs copy of the same text (parallel pread ring -> pinned staging -> H2D)"}
        finally:
            try:
                os.unlink(fpath)
            except OSError:
                pass
        barrier()
    # pinned copy peaks: every rank alone is not what a multi-GPU box gives; all ranks copy at once behind a barrier
    barrier()
    h2d_c = eng.measure_h2d(1 << 30)
    barrier()
    d2h_c = eng.measure_d2h(1 << 30)
    barrier()
    h2d_sum, d2h_sum = sum_over_ranks(h2d_c), sum_over_ranks(d2h_c)
    h2d_per_rank = every_rank(h2d_c)
    if streamed_only:
        total_q, total_rows, total_bytes = e2e_q, e2e_rows, e2e_bytes
        launches = e2e_launches

    cpu = None
    if rank == 0 and not args.no_cpu_baseline:
        cpu, _ = cpu_reference(cfg, w, lineages, min(q_rank, CPU_SAMPLE_Q if not cfg["zipf"] else CPU_SAMPLE_Q // 8), 1, 1)

    if rank == 0:
        e2e = {"value": e2e_q / e2e_s, "unit": "queries/s", "h2d_bytes_per_step": int(host_bytes * passes), "d2h_bytes_per_step": d2h * passes,
               "ms_per_step": e2e_s * 1e3, "text_gb_per_s": e2e_bytes / e2e_s / 1e9, "hit_rows_per_s": e2e_rows / e2e_s,
               "pinned_h2d_concurrent_gb_per_s": h2d_sum, "pinned_d2h_concurrent_gb_per_s": d2h_sum,
               "frac_of_concurrent_h2d_peak": (e2e_bytes / e2e_s / 1e9) / h2d_sum if h2d_sum else None,
               "per_rank_ms_per_step": [round(v, 2) for v in e2e_per_rank], "per_rank_pinned_h2d_concurrent_gb_per_s": [round(v, 1) for v in h2d_per_rank],
               "sample": (f"{host_q} queries ({host_bytes / 1e9:.2f} GB of text) per rank in pinned host memory" +
                          (f", streamed {passes} times per step = the rank's {q_rank}-query shard" if streamed_only else
                           ("" if host_q == q_rank else f" = the first part of the rank's {q_rank}-query shard (--host-gb)")))}
        if streamed_only:
            value, ms_step = e2e["value"], e2e_s * 1e3
        else:
            value, ms_step = total_q / (dev_ms * 1e-3), dev_ms
        line = {
            "metric": "consensus_queries_per_s", "value": value, "unit": "queries/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": scaling, "vs_baseline": None, "dtype": "u8",
            "data": "synthetic", "config": config, "run_info": run_info,
            "value_definition": ("end to end from pinned host text (C5 is a streamed configuration)" if streamed_only else
                                 "text resident in HBM -> consensus records resident in HBM (SURVEY 8d(i)); e2e and value_with_result_download include PCIe"),
            "hit_rows_per_s": total_rows / (ms_step * 1e-3),
            "text_gb_per_s": total_bytes / (ms_step * 1e-3) / 1e9,
            "e2e": e2e, "e2e_file": e2e_file, "gpu_launches": launches, "roofline": roof, "cpu_baseline": cpu, "clocks": clocks, "verified": verified,
        }
        line.update(line_extra)
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
