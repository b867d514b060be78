"""TEST INFRASTRUCTURE: ctypes binding of tests/csrc/_build/libblu_sim.so, the host simulation of the device-side
logic (see tests/csrc/sim_harness.cpp).  Built on demand with g++; never used by the product."""
from __future__ import annotations

import ctypes as C
import os
import subprocess
from typing import List, Optional, Sequence

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_ROOT = os.path.dirname(_HERE)
_SO = os.path.join(_HERE, "csrc", "_build", "libblu_sim.so")
_SRCS = [os.path.join(_HERE, "csrc", "sim_harness.cpp"), os.path.join(_ROOT, "blutils_b200", "csrc", "blu_taxonomy.cpp")]
_DEPS = _SRCS + [os.path.join(_ROOT, "blutils_b200", "csrc", f) for f in ("blu_core.cuh", "blu_decode.h", "blu_taxonomy.h", "blu_json.h")]
TAXON = {"fungi": 0, "bacteria": 1, "eukaryotes": 2, "custom": 3}
STRATEGY = {"cautious": 0, "relaxed": 1}
KEYS = ["domain", "kingdom", "phylum", "class", "order", "family", "genus", "species"]
ABSENT = -(2 ** 31)


def build() -> str:
    if not os.path.exists(_SO) or any(os.path.getmtime(_SO) < os.path.getmtime(d) for d in _DEPS):
        os.makedirs(os.path.dirname(_SO), exist_ok=True)
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-pthread", "-I/usr/local/cuda/include", "-shared", "-o", _SO] + _SRCS)
    return _SO


_lib = None


def lib():
    global _lib
    if _lib is None:
        l = C.CDLL(build())
        l.blu_sim_run.restype = C.c_int
        l.blu_sim_run.argtypes = [C.c_void_p, C.c_void_p, C.c_char_p, C.c_uint64, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_char_p, C.c_uint64,
                                  C.c_char_p, C.c_uint64, C.POINTER(C.c_void_p), C.POINTER(C.c_uint64), C.c_char_p, C.c_int]
        l.blu_sim_free.argtypes = [C.c_void_p]
        l.blu_sim_interpolate.restype = C.c_int
        l.blu_sim_interpolate.argtypes = [C.c_char_p, C.c_int, C.c_int, C.c_void_p, C.POINTER(C.c_double), C.c_int]
        l.blu_sim_custom_cutoffs.restype = C.c_int
        l.blu_sim_custom_cutoffs.argtypes = [C.c_char_p, C.c_void_p, C.c_char_p, C.c_int]
        l.blu_sim_read_taxonomy_json.restype = C.c_longlong
        l.blu_sim_read_taxonomy_json.argtypes = [C.c_char_p, C.c_int, C.c_char_p, C.c_int]
        _lib = l
    return _lib


def _c8(custom):
    if custom is None:
        return None
    return (C.c_int32 * 8)(*[(ABSENT if custom.get(k) is None else int(custom[k])) for k in KEYS])


def run(taxids: Sequence[int], lineages: Sequence[str], taxon: str, strategy: str, text: bytes, custom=None,
        headers: Optional[List[str]] = None):
    """Returns (rc, jsonl bytes or None, error message)."""
    enc = [s.encode() for s in lineages]
    off = np.zeros(len(enc) + 1, dtype=np.uint64)
    if enc:
        off[1:] = np.cumsum([len(b) for b in enc], dtype=np.uint64)
    ids = np.asarray(list(taxids), dtype=np.int64)
    c8 = _c8(custom)
    out, ol = C.c_void_p(), C.c_uint64()
    err = C.create_string_buffer(512)
    hb = "\n".join(headers).encode() if headers else None
    rc = lib().blu_sim_run(ids.ctypes.data, off.ctypes.data, b"".join(enc), len(enc), TAXON[taxon], 1 if c8 is not None else 0,
                           C.cast(c8, C.c_void_p) if c8 is not None else None, STRATEGY[strategy], text, len(text), hb, len(hb) if hb else 0,
                           C.byref(out), C.byref(ol), err, 512)
    if rc != 0:
        return rc, None, err.value.decode()
    try:
        return 0, C.string_at(out, ol.value), ""
    finally:
        lib().blu_sim_free(out)


def run_write(taxids: Sequence[int], lineages: Sequence[str], taxon: str, strategy: str, text: bytes, out_path: Optional[str], fmt: str, run_id: str,
              custom=None, headers: Optional[List[str]] = None, sorted_records: bool = False, two_parts: bool = False) -> int:
    """The same run, written by the product's writers: fmt json (pretty to a file, compact to stdout) / jsonl / yaml / tsv;
    out_path None = stdout.  sorted_records: records in query-id order (a sorted result); two_parts: the records as two parts (a
    multi-device result).  Returns rc."""
    enc = [s.encode() for s in lineages]
    off = np.zeros(len(enc) + 1, dtype=np.uint64)
    if enc:
        off[1:] = np.cumsum([len(b) for b in enc], dtype=np.uint64)
    ids = np.asarray(list(taxids), dtype=np.int64)
    c8 = _c8(custom)
    err = C.create_string_buffer(512)
    hb = "\n".join(headers).encode() if headers else None
    f = lib().blu_sim_run_write
    f.restype = C.c_int
    f.argtypes = [C.c_void_p, C.c_void_p, C.c_char_p, C.c_uint64, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_char_p, C.c_uint64, C.c_char_p, C.c_uint64,
                  C.c_int, C.c_int, C.c_char_p, C.c_int, C.c_char_p, C.c_char_p, C.c_int]
    return f(ids.ctypes.data, off.ctypes.data, b"".join(enc), len(enc), TAXON[taxon], 1 if c8 is not None else 0,
             C.cast(c8, C.c_void_p) if c8 is not None else None, STRATEGY[strategy], text, len(text), hb, len(hb) if hb else 0, int(sorted_records),
             int(two_parts), None if out_path is None else out_path.encode(), {"json": 0, "jsonl": 1, "yaml": 2, "tsv": 3}[fmt], run_id.encode(), err, 512)


def interpolate(ranks: Sequence[str], taxon: str, custom=None) -> List[float]:
    out = (C.c_double * 128)()
    c8 = _c8(custom)
    n = lib().blu_sim_interpolate("\n".join(ranks).encode(), TAXON[taxon], 1 if c8 is not None else 0,
                                  C.cast(c8, C.c_void_p) if c8 is not None else None, out, 128)
    if n < 0:
        raise RuntimeError("interpolate failed")
    return [out[i] for i in range(n)]


def dump_taxonomy_json(path: str, use_taxid: bool = False):
    """[(taxid, lineage)] as the product's `.blutils.json` reader sees the file; IOError with its message when it rejects it."""
    out, ol = C.c_void_p(), C.c_uint64()
    err = C.create_string_buffer(512)
    f = lib().blu_sim_dump_taxonomy_json
    f.restype = C.c_int
    f.argtypes = [C.c_char_p, C.c_int, C.POINTER(C.c_void_p), C.POINTER(C.c_uint64), C.c_char_p, C.c_int]
    if f(path.encode(), 1 if use_taxid else 0, C.byref(out), C.byref(ol), err, 512) != 0:
        raise IOError(err.value.decode(errors="replace"))
    try:
        raw = C.string_at(out, ol.value)
    finally:
        lib().blu_sim_free(out)
    parts = raw.split(b"\0")[:-1]
    return [(int(parts[i]), parts[i + 1].decode("utf-8")) for i in range(0, len(parts), 2)]


def custom_cutoffs(path: str):
    out = (C.c_int32 * 8)()
    err = C.create_string_buffer(512)
    rc = lib().blu_sim_custom_cutoffs(path.encode(), out, err, 512)
    if rc:
        raise ValueError(err.value.decode())
    return {k: (None if out[i] == ABSENT else out[i]) for i, k in enumerate(KEYS)}


def read_taxonomy_json(path: str, use_taxid: bool = False) -> int:
    err = C.create_string_buffer(512)
    n = lib().blu_sim_read_taxonomy_json(path.encode(), int(use_taxid), err, 512)
    if n < 0:
        raise IOError(err.value.decode())
    return n


def taxonomy_cached(json_path: str, cache_path: str, use_taxid: bool = False, taxon: str = "bacteria", custom=None):
    """Product's side-car cache sequence on the host.  Returns (state, checksum of the resulting tables)."""
    l = lib()
    l.blu_sim_taxonomy_cached.restype = C.c_int
    l.blu_sim_taxonomy_cached.argtypes = [C.c_char_p, C.c_char_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.POINTER(C.c_int), C.POINTER(C.c_uint64),
                                          C.c_char_p, C.c_int]
    c8 = _c8(custom)
    state, ck = C.c_int(0), C.c_uint64(0)
    err = C.create_string_buffer(512)
    rc = l.blu_sim_taxonomy_cached(json_path.encode(), cache_path.encode(), int(use_taxid), TAXON[taxon], 1 if c8 is not None else 0,
                                   C.cast(c8, C.c_void_p) if c8 is not None else None, C.byref(state), C.byref(ck), err, 512)
    if rc == 1:
        raise IOError(err.value.decode())
    if rc:
        raise ValueError(err.value.decode())
    return state.value, ck.value


def yaml_str(s: str) -> str:
    """The product's serde_yaml string-scalar emitter (blu_decode.h yaml_str)."""
    l = lib()
    l.blu_sim_yaml_str.restype = C.c_int
    l.blu_sim_yaml_str.argtypes = [C.c_char_p, C.c_uint64, C.c_char_p, C.c_int]
    b = s.encode("utf-8")
    out = C.create_string_buffer(8 * len(b) + 16)
    n = l.blu_sim_yaml_str(b, len(b), out, len(out))
    assert n >= 0
    return out.raw[:n].decode("utf-8")
