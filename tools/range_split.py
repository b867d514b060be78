#!/usr/bin/env python
"""Device-resident step time of the C2 workload for several splits of the table into query-aligned ranges
(BLU_RANGE_FRACS, see resident_ranges in blu_api.cpp).  One process, one generated table; CUDA-event timing around
each run, median of --steps after --warmup.  Measurement tool, not part of pytest / bench.py.

  python tools/range_split.py "1,1,1,1" "0.28,0.28,0.28,0.16" "0.39,0.28,0.19,0.14"
"""
import argparse, ctypes as C, json, os, statistics, sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("fracs", nargs="+")
    ap.add_argument("--queries", type=int, default=1_000_000)
    ap.add_argument("--steps", type=int, default=9)
    ap.add_argument("--warmup", type=int, default=3)
    a = ap.parse_args()
    import torch
    from blutils_b200 import ConsensusEngine, ConsensusStrategy, Taxon, _ffi
    from blutils_b200.synth import SynthWorkload

    w = SynthWorkload(30000, seed=20261018 + 2)
    ids, off, blob = w.lineages(False)
    eng = ConsensusEngine(Taxon.Bacteria, ConsensusStrategy.Relaxed, False, None)
    eng.load_taxonomy_raw(ids.ctypes.data, off.ctypes.data, blob.ctypes.data, len(ids))
    cap = a.queries * 50 * 80 + (1 << 20)
    pinned = _ffi.lib().blu_host_alloc(cap)
    assert pinned
    nbytes, nrows = w.hits_into(pinned, cap, 0, a.queries, 50)
    dbuf = torch.empty((nbytes + 255) // 128 * 128, dtype=torch.uint8, device="cuda")
    dbuf[:nbytes].copy_(torch.frombuffer((C.c_uint8 * nbytes).from_address(pinned), dtype=torch.uint8))
    torch.cuda.synchronize()
    ref = None
    for fr in a.fracs:
        os.environ["BLU_RANGE_FRACS"] = fr
        ms = []
        for i in range(a.warmup + a.steps):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            e0.record()
            out = eng.run_device(dbuf.data_ptr(), nbytes, torch.cuda.current_stream().cuda_stream)
            e1.record()
            torch.cuda.synchronize()
            if i >= a.warmup:
                ms.append(e0.elapsed_time(e1))
            ck, n = out.checksum(), len(out)
            out.close()
            ref = ck if ref is None else ref
            assert ck == ref and n == a.queries
        tm = eng.timings()
        print(json.dumps({"fracs": fr, "ms_median": round(statistics.median(ms), 3), "ms_min": round(min(ms), 3),
                          "queries_per_s_median": round(a.queries / statistics.median(ms) * 1e3),
                          "ms_kernels": round(tm["ms_total_device"], 3)}), flush=True)


if __name__ == "__main__":
    main()
