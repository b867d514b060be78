#!/usr/bin/env python
"""Cost of ordering a result's records by query id on the GPU (blu_result_sort_by_query), and what it saves the writer.

Tables are generated on the GPU with fixed-width rows (one hit per query: the sort works on records, not rows), for two id
styles: `q%09d` (the synthetic workload's ids: 10 bytes, the first 8 shared by runs of 100) and 40-byte Illumina-style read
names (`A00587:112:HHVKLDSXY:1:1101:XXXXX:YYYYYY`, 31 shared bytes, hashed so that file order is not id order).  Per size:

  * device-resident result: sort ms (the record gather in HBM included)
  * host result: sort ms split into id packing, H2D, sort, D2H and the permutation on the host threads (BLU_SORT_TRACE)
  * blu_result_write (JSONL, JSON) of an unsorted result vs. sort + write of a sorted one, alternated; the bytes must match

Measurement tool, not part of pytest / bench.py; prints one JSON object per line.

  python tools/sort_scale.py --sizes 1000,100000,1000000,10000000 --resident-sizes 100000000
"""
import argparse
import hashlib
import json
import os
import re
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

TAIL = b"\tACC1.1\t11\t99.0\t150\t0\t0\t1\t150\t1\t150\t0.0\t300\n"
ILLUMINA = b"A00587:112:HHVKLDSXY:1:1101:"


def gpu_table(n, style):
    """(padded uint8 device tensor, n_bytes): n fixed-width rows, query i's id derived from i."""
    import torch

    q = torch.arange(n, device="cuda", dtype=torch.int64)

    def digits(x, w):
        p = torch.tensor([10 ** (w - 1 - i) for i in range(w)], device="cuda", dtype=torch.int64)
        return ((x[:, None] // p[None, :]) % 10 + 48).to(torch.uint8)

    def const(b):
        return torch.frombuffer(bytearray(b), dtype=torch.uint8).cuda()[None, :].expand(n, len(b))

    if style == "q9":
        cols = [const(b"q"), digits(q, 9)]
    else:
        h = (q * 0x9E3779B1) & ((1 << 27) - 1)  # a bijection of [0, 2^27): distinct ids, scrambled order
        cols = [const(ILLUMINA), digits(h // 1_000_000, 5), const(b":"), digits(h % 1_000_000, 6)]
    rows = torch.cat(cols + [const(TAIL)], dim=1).reshape(-1)
    nb = rows.numel()
    t = torch.zeros((nb + 255) // 128 * 128, dtype=torch.uint8, device="cuda")
    t[:nb] = rows
    del rows
    torch.cuda.synchronize()
    return t, nb


class CaptureStderr:
    """The library's BLU_SORT_TRACE line (C stderr) of the calls inside the block."""

    def __enter__(self):
        sys.stderr.flush()
        self.f = tempfile.TemporaryFile()
        self.saved = os.dup(2)
        os.dup2(self.f.fileno(), 2)
        return self

    def __exit__(self, *a):
        os.dup2(self.saved, 2)
        os.close(self.saved)
        self.f.seek(0)
        self.text = self.f.read().decode(errors="replace")
        self.f.close()

    def stages(self):
        m = re.findall(r"\[blu sort\] ms: (.*)", self.text)
        return {k: float(v) for k, v in (x.split(" ") for x in m[-1].split(", "))} if m else {}


def timed(f):
    t0 = time.perf_counter()
    r = f()
    return (time.perf_counter() - t0) * 1e3, r


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", default="1000,10000,100000,1000000,10000000")
    ap.add_argument("--resident-sizes", default="100000000", help="sizes measured device-resident only")
    ap.add_argument("--styles", default="q9,illumina")
    ap.add_argument("--reps", type=int, default=3)
    a = ap.parse_args()
    import torch

    from blutils_b200 import ConsensusEngine, ConsensusStrategy, OutputFormat, Taxon, _ffi

    try:
        smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True,
                             timeout=30).stdout.strip()
    except Exception as e:  # (the numbers below still say which device they come from)
        smi = f"nvidia-smi unavailable: {e}"
    print(json.dumps({"device": torch.cuda.get_device_name(0), "nvidia_smi": smi}), flush=True)
    eng = ConsensusEngine(Taxon.Bacteria, ConsensusStrategy.Relaxed, False, None)
    eng.load_taxonomy_arrays([11], ["d__bac;p__p1;c__c1;o__o1;f__f1;g__g1;s__s1"])
    stream = torch.cuda.current_stream().cuda_stream
    sizes = [int(x) for x in a.sizes.split(",") if x]
    resident_only = [int(x) for x in a.resident_sizes.split(",") if x]
    tmp = tempfile.mkdtemp(prefix="blu_sort_scale_")
    for style in a.styles.split(","):
        for n in sizes + resident_only:
            t, nb = gpu_table(n, style)
            row = {"style": style, "queries": n, "text_bytes": nb}
            # device-resident
            ms = []
            for _ in range(a.reps):
                out = eng.run_device_resident(t.data_ptr(), nb, stream)
                assert _ffi.lib().blu_result_num_records(out._h) == n
                ms.append(timed(out.sort_by_query)[0])
                out.close()
            row["resident_sort_ms"] = round(min(ms), 3)
            row["resident_sort_all_ms"] = [round(x, 3) for x in ms]
            if n in resident_only:
                print(json.dumps(row), flush=True)
                del t
                torch.cuda.empty_cache()
                continue
            host = t[:nb].cpu().numpy()
            hptr = host.ctypes.data
            # host result: the split of the sort
            os.environ["BLU_SORT_TRACE"] = "1"
            splits = []
            for _ in range(a.reps):
                out = eng.run_host(hptr, nb)
                with CaptureStderr() as cap:
                    wall = timed(out.sort_by_query)[0]
                st = cap.stages()
                st["wall"] = round(wall, 3)
                splits.append(st)
                out.close()
            os.environ.pop("BLU_SORT_TRACE", None)
            row["host_sort_ms"] = min(splits, key=lambda s: s["wall"])
            # the writer with and without a prior sort, alternated
            for fmt, ext in ((OutputFormat.Jsonl, "jsonl"), (OutputFormat.Json, "json")):
                plain, with_sort = [], []
                for _ in range(2):
                    out = eng.run_host(hptr, nb)
                    p1 = os.path.join(tmp, "plain." + ext)
                    plain.append(timed(lambda: out.write(p1, fmt, run_id="00000000-0000-4000-8000-000000000000"))[0])
                    out.close()
                    out = eng.run_host(hptr, nb)
                    p2 = os.path.join(tmp, "sorted." + ext)
                    s_ms = timed(out.sort_by_query)[0]
                    w_ms = timed(lambda: out.write(p2, fmt, run_id="00000000-0000-4000-8000-000000000000"))[0]
                    with_sort.append((s_ms, w_ms))
                    out.close()
                    same = hashlib.sha256(open(p1, "rb").read()).digest() == hashlib.sha256(open(p2, "rb").read()).digest()
                    assert same, f"{ext} bytes differ after the sort ({style}, {n})"
                    os.remove(p1)
                    os.remove(p2)
                best = min(with_sort, key=lambda x: x[0] + x[1])
                row[f"write_{ext}_ms"] = round(min(plain), 3)
                row[f"sort_then_write_{ext}_ms"] = {"sort": round(best[0], 3), "write": round(best[1], 3), "total": round(best[0] + best[1], 3)}
            print(json.dumps(row), flush=True)
            del t, host
            torch.cuda.empty_cache()
    os.rmdir(tmp)
    eng.close()


if __name__ == "__main__":
    main()
