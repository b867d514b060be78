"""Host-side mirror of the reference's interface for the consensus-identity path.

Same names, argument meaning and error behaviour as blutils 8.3.1 (paths relative to the reference repo):

* ``build_consensus_identities(blast_output, taxonomies_file, taxon, strategy, use_taxid, custom_taxon_values)``
  -- core/src/use_cases/build_consensus_identities/mod.rs:40-47
* ``ParallelBlastOutput`` -- core/src/domain/dtos/parallel_blast_output.rs:3-7
* ``Taxon`` / ``CustomTaxon.from_file`` -- core/src/domain/dtos/taxon.rs:14-88
* ``ConsensusStrategy`` -- core/src/domain/dtos/consensus_strategy.rs:3-10
* ``write_blutils_output`` / ``OutputFormat`` -- core/src/use_cases/write_blutils_output.rs:20-38

All computation happens in libblu_consensus.so on the GPU; this file only marshals arguments."""
from __future__ import annotations

import ctypes as C
import enum
import json
import os
from dataclasses import dataclass, field
from typing import Dict, List, Optional, Sequence, Union

from . import _ffi
from ._ffi import blu_opts, blu_timings


class MappedErrors(Exception):
    """I/O-class failure: the reference returns Err(MappedErrors) (mod.rs:250-265,357-364)."""


class ConsensusPanic(Exception):
    """Data-dependent failure on which the reference panics (SURVEY.md section 5); fatal to the run."""


class Unsupported(Exception):
    """Valid for the reference but outside this implementation's documented limits (never a silent answer)."""


class CudaUnavailable(RuntimeError):
    pass


def _raise(rc: int, msg: str):
    if rc == _ffi.BLU_ERR_IO:
        raise MappedErrors(msg)
    if rc == _ffi.BLU_ERR_DATA:
        raise ConsensusPanic(msg)
    if rc == _ffi.BLU_ERR_UNSUPPORTED:
        raise Unsupported(msg)
    if rc == _ffi.BLU_ERR_CUDA:
        raise CudaUnavailable(msg)
    raise RuntimeError(f"blu error {rc}: {msg}")


class Taxon(enum.Enum):
    Fungi = 0
    Bacteria = 1
    Eukaryotes = 2
    Custom = 3

    @classmethod
    def from_str(cls, s: str) -> "Taxon":  # taxon.rs:91-103
        m = {"f": cls.Fungi, "fungi": cls.Fungi, "Fungi": cls.Fungi, "b": cls.Bacteria, "bacteria": cls.Bacteria, "Bacteria": cls.Bacteria,
             "e": cls.Eukaryotes, "eukaryotes": cls.Eukaryotes, "Eukaryotes": cls.Eukaryotes, "c": cls.Custom, "custom": cls.Custom,
             "Custom": cls.Custom}
        if s not in m:
            raise ValueError(s)
        return m[s]


class ConsensusStrategy(enum.Enum):
    Cautious = 0
    Relaxed = 1


class OutputFormat(enum.Enum):
    Json = 0
    Jsonl = 1
    Yaml = 2


_CUSTOM_KEYS = ["domain", "kingdom", "phylum", "class", "order", "family", "genus", "species"]


@dataclass
class CustomTaxon:
    domain: int
    species: int
    kingdom: Optional[int] = None
    phylum: Optional[int] = None
    class_: Optional[int] = None
    order: Optional[int] = None
    family: Optional[int] = None
    genus: Optional[int] = None

    def as_array(self) -> List[int]:
        vals = [self.domain, self.kingdom, self.phylum, self.class_, self.order, self.family, self.genus, self.species]
        return [_ffi.BLU_CUTOFF_ABSENT if v is None else int(v) for v in vals]

    @classmethod
    def from_array(cls, a: Sequence[int]) -> "CustomTaxon":
        v = [None if x == _ffi.BLU_CUTOFF_ABSENT else int(x) for x in a]
        return cls(domain=v[0], kingdom=v[1], phylum=v[2], class_=v[3], order=v[4], family=v[5], genus=v[6], species=v[7])

    @classmethod
    def from_file(cls, path: str) -> "CustomTaxon":
        """CustomTaxon::from_file (taxon.rs:28-65); every failure is a panic in the reference."""
        o = blu_opts()
        err = C.create_string_buffer(512)
        rc = _ffi.lib().blu_custom_cutoffs_from_file(os.fspath(path).encode(), C.byref(o), err, 512)
        if rc != 0:
            raise ConsensusPanic(err.value.decode())
        return cls.from_array(list(o.custom))


@dataclass
class ParallelBlastOutput:
    output_file: str
    headers: Optional[List[str]] = None


@dataclass
class ConsensusBean:  # consensus_result.rs:37-45
    rank: str
    identifier: str
    occurrences: int
    taxonomy: Optional[str]
    accessions: List[str]


@dataclass
class TaxonomyBean:  # taxonomy_bean.rs:5-17
    reached_rank: str
    max_allowed_rank: Optional[str]
    identifier: str
    perc_identity: float
    bit_score: float
    taxonomy: Optional[str]
    mutated: bool
    single_match: bool
    consensus_beans: Optional[List[ConsensusBean]]


@dataclass
class QueryWithConsensus:  # consensus_result.rs:7-13  (ConsensusResult::ConsensusFound)
    query: str
    taxon: Optional[TaxonomyBean]
    run_id: Optional[str] = None


@dataclass
class QueryWithoutConsensus:  # consensus_result.rs:15-19 (ConsensusResult::NoConsensusFound)
    query: str


ConsensusResult = Union[QueryWithConsensus, QueryWithoutConsensus]


class ConsensusOutput:
    """Owns a blu_result (binary records in pinned host memory); decodes lazily."""

    def __init__(self, engine: "ConsensusEngine", handle: int):
        self._engine = engine
        self._h = C.c_void_p(handle)
        self._keep = None

    def __len__(self) -> int:
        return _ffi.lib().blu_result_num_queries(self._h)

    @property
    def n_rows(self) -> int:
        return _ffi.lib().blu_result_num_rows(self._h)

    def add_headers(self, headers: Sequence[str]) -> None:
        b = "\n".join(headers).encode()
        _ffi.lib().blu_result_add_headers(self._h, b, len(b))

    def checksum(self) -> int:
        return _ffi.lib().blu_result_checksum(self._h)

    def jsonl(self, head: Optional[int] = None) -> bytes:
        """Canonical JSONL: one {"query":..,"taxon":..} per line, sorted by query, no runId.  `head`: only the first lines."""
        out = C.c_void_p()
        n = C.c_uint64()
        if head is None:
            rc = _ffi.lib().blu_result_to_jsonl(self._h, C.byref(out), C.byref(n))
        else:
            rc = _ffi.lib().blu_result_to_jsonl_head(self._h, int(head), C.byref(out), C.byref(n))
        if rc != 0:
            raise RuntimeError("blu_result_to_jsonl failed")
        try:
            return bytes((C.c_char * n.value).from_address(out.value)) if n.value else b""  # (string_at takes an int: 2 GB limit)
        finally:
            _ffi.lib().blu_free(out)

    def dicts(self) -> List[dict]:
        return [json.loads(l) for l in self.jsonl().decode("utf-8").splitlines()]

    def results(self) -> List[ConsensusResult]:
        out: List[ConsensusResult] = []
        for d in self.dicts():
            t = d["taxon"]
            if t is None:
                out.append(QueryWithoutConsensus(d["query"]))
                continue
            beans = [ConsensusBean(b["rank"], b["identifier"], b["occurrences"], b["taxonomy"], b["accessions"]) for b in t["consensusBeans"]]
            out.append(QueryWithConsensus(d["query"], TaxonomyBean(t["reachedRank"], t["maxAllowedRank"], t["identifier"], t["percIdentity"],
                                                                   t["bitScore"], t["taxonomy"], t["mutated"], t["singleMatch"], beans)))
        return out

    def write(self, blutils_out_file: Optional[str], out_format: OutputFormat = OutputFormat.Json, run_id: Optional[str] = None) -> None:
        rc = _ffi.lib().blu_result_write(self._h, None if blutils_out_file is None else os.fspath(blutils_out_file).encode(), out_format.value,
                                         None if run_id is None else run_id.encode())
        if rc != 0:
            raise MappedErrors("could not write the blutils output")

    def write_tabular(self, output_file: Optional[str], run_id: Optional[str] = None) -> None:
        """parse_consensus_as_tabular (parse_consensus_as_tabular/mod.rs:15-173) from the binary records."""
        rc = _ffi.lib().blu_result_write_tabular(self._h, None if output_file is None else os.fspath(output_file).encode(),
                                                 None if run_id is None else run_id.encode())
        if rc != 0:
            raise MappedErrors("could not write the tabular output")

    def download(self) -> "ConsensusOutput":
        """Device-resident result (run_device_resident) -> host; afterwards every accessor / writer works."""
        if _ffi.lib().blu_result_download(self._h) != 0:
            raise RuntimeError("blu_result_download failed")
        return self

    def sort_by_query(self) -> "ConsensusOutput":
        """Orders the records by query id on the GPU of the engine that produced the result (blu_result_sort_by_query): a
        stable, bytewise sort, the writer's order.  Works on device-resident results before `.download()` too."""
        self._engine._check(_ffi.lib().blu_result_sort_by_query(self._engine._h, self._h))
        return self

    def device_arrays(self):
        """(records_ptr, beans_ptr, n_beans, accessions_ptr, n_accessions) of a device-resident result."""
        nb, na = C.c_uint64(), C.c_uint64()
        l = _ffi.lib()
        return (l.blu_result_device_records(self._h), l.blu_result_device_beans(self._h, C.byref(nb)), nb.value,
                l.blu_result_device_accessions(self._h, C.byref(na)), na.value)

    def device_text(self):
        """(ptr, n_bytes) of the device text the references of a device-resident result point into: the caller's text, or the
        regrouped copy the library made of a non-contiguous table (owned by the result)."""
        n = C.c_uint64()
        return _ffi.lib().blu_result_device_text(self._h, C.byref(n)), n.value

    def records(self):
        """The binary records as a ctypes array (host results); hit-less headers are not records."""
        n = _ffi.lib().blu_result_num_records(self._h)
        p = _ffi.lib().blu_result_records(self._h)
        return C.cast(p, C.POINTER(_ffi.blu_record * n)).contents if p else None

    def query_ids(self) -> List[bytes]:
        """The query id of every binary record, read through the string base (pool, or the caller's text with text_refs)."""
        n = C.c_uint64()
        base = _ffi.lib().blu_result_pool(self._h, C.byref(n))
        recs = self.records()
        return [] if recs is None else [C.string_at(base + r.query_off, r.query_len) for r in recs]

    def close(self) -> None:
        if self._h:
            _ffi.lib().blu_result_free(self._h)
            self._h = None
        self._keep = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class ConsensusEngine:
    """One blu_ctx: (taxon, strategy, use_taxid, custom cutoffs) + a taxonomy resident on one GPU, or -- with
    `devices=[...]` -- on several GPUs of one box: the hit table is then sharded by query range over them
    (blu_ctx_create_multi; no collective) and the shards' results come back as one result."""

    def __init__(self, taxon: Taxon, strategy: ConsensusStrategy, use_taxid: Optional[bool] = None,
                 custom_taxon_values: Optional[CustomTaxon] = None, device: int = 0, chunk_bytes: int = 0,
                 devices: Optional[Sequence[int]] = None, text_refs: bool = False):
        o = blu_opts()
        o.device = device
        o.flags = _ffi.BLU_OPT_TEXT_REFS if text_refs else 0
        o.taxon = taxon.value
        o.strategy = strategy.value
        o.use_taxid = 1 if use_taxid else 0
        o.has_custom = 1 if custom_taxon_values is not None else 0
        arr = custom_taxon_values.as_array() if custom_taxon_values is not None else [0] * 8
        for i in range(8):
            o.custom[i] = arr[i]
        o.chunk_bytes = chunk_bytes
        h = C.c_void_p()
        if devices is not None:
            arr_d = (C.c_int * len(devices))(*[int(d) for d in devices])
            rc = _ffi.lib().blu_ctx_create_multi(C.byref(o), arr_d, len(devices), C.byref(h))
        else:
            rc = _ffi.lib().blu_ctx_create(C.byref(o), C.byref(h))
        if rc != 0:
            _raise(rc, (_ffi.lib().blu_last_error(None) or b"").decode())
        self._h = h
        self.device = device
        self.devices = list(devices) if devices is not None else [device]
        self.text_refs = text_refs

    def _check(self, rc: int):
        if rc != 0:
            _raise(rc, (_ffi.lib().blu_last_error(self._h) or b"").decode())

    def load_taxonomy(self, taxonomies_file: str, cache: Union[None, bool, str] = None) -> Optional[int]:
        """get_taxonomies_dataframe (mod.rs:246-327).  `cache`: None/False = parse the JSON (what the reference does on every
        run); True = side-car cache `<taxonomies_file>.blucache`; a path = that cache file.  With a cache the return
        value is 1 (loaded from the cache), 0 (built, cache written) or -1 (built, cache not writable)."""
        path = os.fspath(taxonomies_file).encode()
        if not cache:
            self._check(_ffi.lib().blu_taxonomy_load_json(self._h, path))
            return None
        state = C.c_int(0)
        cpath = None if cache is True else os.fspath(cache).encode()
        self._check(_ffi.lib().blu_taxonomy_load_json_cached(self._h, path, cpath, C.byref(state)))
        return state.value

    def load_taxonomy_arrays(self, taxids, lineages: Sequence[Union[str, bytes]]) -> None:
        import numpy as np

        enc = [s.encode("utf-8") if isinstance(s, str) else s for s in lineages]
        off = np.zeros(len(enc) + 1, dtype=np.uint64)
        if enc:
            off[1:] = np.cumsum([len(b) for b in enc], dtype=np.uint64)
        blob = b"".join(enc)
        ids = np.ascontiguousarray(np.asarray(taxids, dtype=np.int64))
        self._check(_ffi.lib().blu_taxonomy_load_arrays(self._h, ids.ctypes.data, off.ctypes.data, blob, len(enc)))

    def load_taxonomy_raw(self, taxids_ptr: int, off_ptr: int, blob_ptr: int, n: int) -> None:
        self._check(_ffi.lib().blu_taxonomy_load_arrays(self._h, taxids_ptr, off_ptr, blob_ptr, n))

    def run_file(self, blast_out: str) -> ConsensusOutput:
        r = C.c_void_p()
        self._check(_ffi.lib().blu_consensus_run_file(self._h, os.fspath(blast_out).encode(), C.byref(r)))
        return ConsensusOutput(self, r.value)

    def run_host(self, text: Union[bytes, int], nbytes: Optional[int] = None) -> ConsensusOutput:
        r = C.c_void_p()
        keep = None
        if isinstance(text, (bytes, bytearray)):
            buf = C.create_string_buffer(bytes(text), len(text)) if len(text) else C.create_string_buffer(1)
            keep = buf  # with text_refs the result's strings point into this buffer
            self._check(_ffi.lib().blu_consensus_run_host(self._h, C.addressof(buf), len(text), C.byref(r)))
        else:
            self._check(_ffi.lib().blu_consensus_run_host(self._h, int(text), int(nbytes), C.byref(r)))
        out = ConsensusOutput(self, r.value)
        out._keep = keep
        return out

    def run_device(self, dptr: int, nbytes: int, stream: int = 0) -> ConsensusOutput:
        r = C.c_void_p()
        self._check(_ffi.lib().blu_consensus_run_device(self._h, int(dptr), int(nbytes), int(stream) or None, C.byref(r)))
        return ConsensusOutput(self, r.value)

    def run_device_resident(self, dptr: int, nbytes: int, stream: int = 0) -> ConsensusOutput:
        """Text in HBM -> records in HBM (SURVEY 8d(i)); `.download()` brings the result to the host."""
        r = C.c_void_p()
        self._check(_ffi.lib().blu_consensus_run_device_resident(self._h, int(dptr), int(nbytes), int(stream) or None, C.byref(r)))
        return ConsensusOutput(self, r.value)

    def timings(self) -> Dict[str, float]:
        t = blu_timings()
        _ffi.lib().blu_ctx_last_timings(self._h, C.byref(t))
        return {k: getattr(t, k) for k, _ in t._fields_ if k != "reserved"}

    def measure_h2d(self, nbytes: int = 1 << 30) -> float:
        g = C.c_double()
        self._check(_ffi.lib().blu_ctx_measure_h2d(self._h, nbytes, C.byref(g)))
        return g.value

    def measure_d2h(self, nbytes: int = 1 << 30) -> float:
        g = C.c_double()
        self._check(_ffi.lib().blu_ctx_measure_d2h(self._h, nbytes, C.byref(g)))
        return g.value

    def close(self) -> None:
        if self._h:
            _ffi.lib().blu_ctx_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def _run_configs(engines: Sequence[ConsensusEngine], call, keep=None) -> List[ConsensusOutput]:
    n = len(engines)
    ctxs = (C.c_void_p * max(n, 1))(*[e._h for e in engines])
    outs = (C.c_void_p * max(n, 1))()
    rc = call(ctxs, n, outs)
    if rc != 0:
        _raise(rc, (_ffi.lib().blu_last_error(engines[0]._h if n else None) or b"").decode())
    res = [ConsensusOutput(e, outs[k]) for k, e in enumerate(engines)]
    for r in res:
        r._keep = keep
    return res


def run_host_configs(engines: Sequence[ConsensusEngine], text: Union[bytes, int], nbytes: Optional[int] = None) -> List[ConsensusOutput]:
    """One pass over a hit table in host memory for several configurations (blu_consensus_run_host_configs): the text is
    parsed and copied to the GPU once; result k is what engines[k].run_host(text) returns and belongs to engines[k]."""
    if isinstance(text, (bytes, bytearray)):
        buf = C.create_string_buffer(bytes(text), len(text)) if len(text) else C.create_string_buffer(1)
        return _run_configs(engines, lambda c, n, o: _ffi.lib().blu_consensus_run_host_configs(c, n, C.addressof(buf), len(text), o), buf)
    return _run_configs(engines, lambda c, n, o: _ffi.lib().blu_consensus_run_host_configs(c, n, int(text), int(nbytes), o))


def run_file_configs(engines: Sequence[ConsensusEngine], blast_out: str) -> List[ConsensusOutput]:
    """One pass over a hit table file for several configurations (blu_consensus_run_file_configs): the file is read once."""
    path = os.fspath(blast_out).encode()
    return _run_configs(engines, lambda c, n, o: _ffi.lib().blu_consensus_run_file_configs(c, n, path, o))


def run_device_resident_configs(engines: Sequence[ConsensusEngine], dptr: int, nbytes: int, stream: int = 0) -> List[ConsensusOutput]:
    """One pass over a hit table in HBM for several configurations (blu_consensus_run_device_resident_configs): the results
    stay on the device; `.download()` each of them."""
    return _run_configs(engines, lambda c, n, o: _ffi.lib().blu_consensus_run_device_resident_configs(c, n, int(dptr), int(nbytes),
                                                                                                        int(stream) or None, o))


def shard_cuts(text: Union[bytes, int], n_shards: int, nbytes: Optional[int] = None) -> List[int]:
    """Byte offsets that split a (contiguous) hit table into n_shards query-aligned ranges (SURVEY 8e).  Host-only."""
    cuts = (C.c_uint64 * (n_shards + 1))()
    if isinstance(text, (bytes, bytearray)):
        buf = C.create_string_buffer(bytes(text), len(text)) if len(text) else C.create_string_buffer(1)
        rc = _ffi.lib().blu_shard_cuts(C.addressof(buf), len(text), n_shards, cuts)
    else:
        rc = _ffi.lib().blu_shard_cuts(int(text), int(nbytes), n_shards, cuts)
    if rc != 0:
        raise ValueError("blu_shard_cuts failed")
    return list(cuts)


def shard_cuts_file(path: str, n_shards: int) -> List[int]:
    """shard_cuts for a table in a file: only the rows around every cut are read.  Host-only."""
    cuts = (C.c_uint64 * (n_shards + 1))()
    rc = _ffi.lib().blu_shard_cuts_file(os.fspath(path).encode(), n_shards, cuts)
    if rc != 0:
        raise MappedErrors("Unexpected error occurred on load table.")
    return list(cuts)


def build_consensus_identities(blast_output: ParallelBlastOutput, taxonomies_file: str, taxon: Taxon, strategy: ConsensusStrategy,
                               use_taxid: Optional[bool] = None, custom_taxon_values: Optional[CustomTaxon] = None, *,
                               device: int = 0, devices: Optional[Sequence[int]] = None) -> ConsensusOutput:
    """Drop-in for mod.rs:40-47.  Returns the results container (len() == number of ConsensusResult values);
    `.results()` gives the reference's result types, `.write()` is write_blutils_output."""
    eng = ConsensusEngine(taxon, strategy, use_taxid, custom_taxon_values, device=device, devices=devices)
    eng.load_taxonomy(taxonomies_file)
    out = eng.run_file(blast_output.output_file)
    if blast_output.headers is not None:
        out.add_headers(blast_output.headers)
    return out


def write_blutils_output(results: ConsensusOutput, config=None, blutils_out_file: Optional[str] = None,
                         out_format: OutputFormat = OutputFormat.Json) -> None:
    """write_blutils_output.rs:33-38; `config` is always None on this path (cmds/blast/mod.rs:139)."""
    if config is not None:
        raise Unsupported("BlastBuilder config echo belongs to run-with-consensus, which is out of scope")
    results.write(blutils_out_file, out_format)


def parse_consensus_as_tabular(blutils_result: str = "-", output_file: Optional[str] = None, result_format: OutputFormat = OutputFormat.Json,
                               run_id: Optional[str] = None) -> None:
    """parse_consensus_as_tabular/mod.rs:15-19 (`blu blastn build-tabular`): blutils result file (or "-" = stdin) -> TSV.
    Needs no GPU.  `run_id` replaces the reference's random UUID where the input carries none."""
    err = C.create_string_buffer(1024)
    rc = _ffi.lib().blu_result_file_to_tabular(os.fspath(blutils_result).encode(), None if output_file is None else os.fspath(output_file).encode(),
                                               result_format.value, None if run_id is None else run_id.encode(), err, 1024)
    if rc != 0:
        _raise(rc, err.value.decode())
