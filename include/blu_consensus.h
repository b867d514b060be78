/* blu_consensus.h -- C ABI of the B200-native consensus-identity stage of blutils.
 *
 * This is the drop-in boundary for ONE path of the reference: `build_consensus_identities`
 * (core/src/use_cases/build_consensus_identities/mod.rs:40-47 of blutils 8.3.1) and its consumer
 * `write_blutils_output` (core/src/use_cases/write_blutils_output.rs:33-38).  The reference has no FFI
 * of its own (no `extern "C"` anywhere); these entry points are what a thin Rust `-sys` crate binds
 * (see INTEGRATION.md and rust/blu-consensus-sys/).  Plain pointers and sizes only; no C++/torch types.
 *
 * The library has NO CPU fallback: every entry point that computes requires a CUDA device (sm_100a) and
 * fails with BLU_ERR_CUDA otherwise.
 *
 * Threading: a blu_ctx is not thread-safe; use one per calling thread / per GPU.  Calls are synchronous.
 */
#ifndef BLU_CONSENSUS_H
#define BLU_CONSENSUS_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define BLU_ABI_VERSION 2

/* Status codes.  The reference distinguishes `Err(MappedErrors)` (I/O-class: mod.rs:250-265,357-364) from
 * panics (every data-dependent failure: mod.rs:123,174-184,371; find_single_query_consensus.rs:59,115;
 * find_multi_taxa_consensus.rs:181; build_blast_consensus_identity.rs:97).  Both are fatal to the run. */
enum {
    BLU_OK = 0,
    BLU_ERR_IO = 1,          /* maps to Err(MappedErrors): file missing / unreadable / not JSON */
    BLU_ERR_DATA = 2,        /* maps to the reference's panics: malformed row, unmapped taxid in a top group,
                                root-level disagreement, empty adjusted taxonomy, ... */
    BLU_ERR_CUDA = 3,        /* no device, launch or allocation failure */
    BLU_ERR_ARG = 4,         /* bad argument to this API */
    BLU_ERR_UNSUPPORTED = 5, /* valid for the reference but outside this implementation's documented limits
                                (never a silent wrong answer) */
    BLU_ERR_INTERNAL = 6
};

/* Taxon (core/src/domain/dtos/taxon.rs:68-88) */
enum { BLU_TAXON_FUNGI = 0, BLU_TAXON_BACTERIA = 1, BLU_TAXON_EUKARYOTES = 2, BLU_TAXON_CUSTOM = 3 };
/* ConsensusStrategy (core/src/domain/dtos/consensus_strategy.rs:3-10) */
enum { BLU_STRATEGY_CAUTIOUS = 0, BLU_STRATEGY_RELAXED = 1 };
/* OutputFormat (core/src/use_cases/write_blutils_output.rs:20-31) */
enum { BLU_FORMAT_JSON = 0, BLU_FORMAT_JSONL = 1, BLU_FORMAT_YAML = 2 };

#define BLU_CUTOFF_ABSENT ((int32_t)-2147483647 - 1) /* Option::None of CustomTaxon's optional i16 fields */

/* blu_opts.flags */
#define BLU_OPT_TEXT_REFS 1u /* blu_consensus_run_host: query ids / accessions of the result stay (offset, length) references into
                                the CALLER's text instead of being copied into a string pool (SURVEY 8b "Ownership"): nothing but
                                records, beans and 8-byte accession references is downloaded.  The text must outlive the result. */

/* The by-value arguments of build_consensus_identities (mod.rs:40-47) other than the two paths. */
typedef struct blu_opts {
    int32_t device;     /* CUDA device ordinal this context runs on (blu_ctx_create_multi: ignored) */
    int32_t taxon;      /* BLU_TAXON_* */
    int32_t strategy;   /* BLU_STRATEGY_* */
    int32_t use_taxid;  /* Option<bool>: 1 -> numericLineage, 0 -> textLineage (mod.rs:287-291) */
    int32_t has_custom; /* Option<CustomTaxon> present */
    int32_t custom[8];  /* domain,kingdom,phylum,class,order,family,genus,species (taxon.rs:14-25); i16 range or
                           BLU_CUTOFF_ABSENT for the six optional ones */
    uint64_t chunk_bytes; /* streaming chunk for host input; 0 = default (256 MiB) */
    uint64_t flags;       /* BLU_OPT_* */
    uint64_t reserved[3];
} blu_opts;

typedef struct blu_ctx blu_ctx;
typedef struct blu_result blu_result;

/* Fixed-size consensus record, one per query, as produced on the device (SURVEY.md section 8 a13).
 * Strings are (offset, length) references into the result's string base (blu_result_pool: the string pool, or the
 * caller's text with BLU_OPT_TEXT_REFS / device-resident results); lineage-derived strings are resolved through the
 * context's taxonomy.  Beans and accession references are stored compactly (no holes): the beans of a record are
 * beans[bean_base .. bean_base + n_beans), its accession references accessions[acc_base ..), bean by bean. */
typedef struct blu_record {
    uint64_t query_off;     /* offset of the query id in the string base */
    uint32_t query_len;
    uint32_t n_rows;        /* hit rows of this query */
    uint64_t keep_mask;     /* bit j set: reference-lineage position j is part of the output `taxonomy` */
    double perc_identity;   /* TaxonomyBean.perc_identity, bit-for-bit the reference row's pident */
    int64_t bit_score;      /* truncated bit score (mod.rs:162,184); serialised as f64 */
    uint32_t ref_lineage;   /* index of the reference lineage in the loaded taxonomy */
    uint32_t bean_base;     /* first bean of this query */
    uint32_t n_beans;
    uint32_t acc_base;      /* first accession reference of this query */
    uint8_t status;         /* 1 = ConsensusFound; 0 = NoConsensusFound (hit-less header) */
    uint8_t single_match;
    uint8_t mutated;
    int8_t reached_pos;     /* lineage position of reachedRank/identifier */
    int8_t allowed_pos;     /* lineage position of maxAllowedRank, -1 = null */
    int8_t bean_level;      /* lineage position the consensus beans were taken at */
    uint8_t pad[2];
} blu_record; /* 64 bytes */

typedef struct blu_bean {
    uint32_t first_lineage; /* lineage of the first (sorted) row carrying this bean: its `taxonomy` string */
    uint32_t occurrences;
    uint32_t acc_begin;     /* relative to the record's acc_base */
    uint32_t n_acc;
} blu_bean;

/* accession reference: offset << 16 | length (an accession is at most 65535 bytes) */
typedef struct blu_acc {
    uint64_t ref;
} blu_acc;
#define BLU_ACC_OFF(a) ((a).ref >> 16)
#define BLU_ACC_LEN(a) ((uint32_t)((a).ref & 0xFFFFu))

/* Stage timings of the last run (CUDA events, milliseconds) and byte counts, for bench.py's roofline. */
typedef struct blu_timings {
    double ms_total_device;  /* first kernel start -> last kernel end, on the run's stream */
    double ms_tile_kernel;   /* the dominant fused tokenise/join/group/consensus kernel */
    double ms_longrun_kernel;
    double ms_gather_kernel;
    double ms_other;
    uint64_t text_bytes, result_bytes, taxonomy_bytes;
    uint64_t h2d_bytes, d2h_bytes;
    uint64_t n_queries, n_rows, n_deferred_runs, n_kernel_launches;
    uint64_t n_regrouped; /* non-zero when the table was non-contiguous and was regrouped by query first: 2 = on the GPU, 1 = on the host */
    uint64_t n_tile_launches; /* tile_kernel launches of the run (ranges / streamed chunks); ms_tile_kernel is their sum */
    uint64_t reserved[2];
} blu_timings;

/* ---- context ------------------------------------------------------------------------------------------- */
int blu_ctx_create(const blu_opts* opts, blu_ctx** out);
/* One context over several GPUs of one box -- the reference's entry point consumes ONE hit table (mod.rs:40-47) and
 * fans its queries out (mod.rs:104-128); here the table is sharded by query range over `n_devices` GPUs (SURVEY 8e):
 * blu_shard_cuts, one host worker thread + its own streams per GPU, lineage tables replicated, every GPU's result
 * downloaded into its own part of ONE blu_result; no collective, no NCCL.  Every entry point that takes a blu_ctx
 * accepts such a context (blu_consensus_run_device / _resident need a single-device one); opts->device is ignored.
 * A table whose queries are not contiguous is detected across the shards (the 64-bit query-id hashes of all shards
 * are merged on the first device) and regrouped like on one GPU. */
int blu_ctx_create_multi(const blu_opts* opts, const int* devices, int n_devices, blu_ctx** out);
int blu_ctx_num_devices(const blu_ctx* ctx);
void blu_ctx_destroy(blu_ctx* ctx);
/* Message of the last failing call on this context (or of the failing blu_ctx_create when ctx == NULL). */
const char* blu_last_error(const blu_ctx* ctx);

/* CustomTaxon::from_file (taxon.rs:28-65): `.yaml` or `.json` by extension; fills opts->custom / has_custom. */
int blu_custom_cutoffs_from_file(const char* path, blu_opts* opts, char* err, size_t errlen);

/* ---- taxonomy (get_taxonomies_dataframe, mod.rs:246-327; TaxonomiesMap, taxonomies_map.rs:6-32) ---------- */
int blu_taxonomy_load_json(blu_ctx* ctx, const char* path);
/* Same, through a binary side-car cache (SURVEY section 8 f2; the reference re-parses the JSON on every run,
 * mod.rs:254-265).  The cache holds the encoded lineage tables and is keyed by the content hash of the JSON file,
 * use_taxid and the cutoff options of `ctx`; a missing, stale or damaged cache is rebuilt from the JSON.
 * cache_path == NULL means `<path>.blucache`.  *cache_state (may be NULL): 1 = loaded from the cache, 0 = built from
 * the JSON and cache written, -1 = built from the JSON, cache could not be written (the call still succeeds). */
int blu_taxonomy_load_json_cached(blu_ctx* ctx, const char* path, const char* cache_path, int* cache_state);
/* Same, from memory: n lineage strings concatenated in blob, string i = blob[off[i]..off[i+1]). */
int blu_taxonomy_load_arrays(blu_ctx* ctx, const int64_t* taxids, const uint64_t* off, const char* blob, uint64_t n);

/* ---- the hot path (build_consensus_identities, mod.rs:40-129) ------------------------------------------- */
/* outfmt-6 text in host memory (pinned or pageable); streamed to the device in chunks. */
int blu_consensus_run_host(blu_ctx* ctx, const char* text, uint64_t n_bytes, blu_result** out);
/* Text already resident in device memory of ctx's device.  `dtext` must be 16-byte aligned and readable up to
 * n_bytes rounded up to 128.  `stream` is a cudaStream_t (NULL = the context's own stream). */
int blu_consensus_run_device(blu_ctx* ctx, const void* dtext, uint64_t n_bytes, void* stream, blu_result** out);
/* Same, but the result stays in device memory (SURVEY 8d(i): "text already in HBM -> records in HBM"): nothing but the
 * counters crosses PCIe, strings stay (offset, length) references into `dtext`, no host round trip inside the call.
 * blu_result_device_* give the device arrays; blu_result_download() brings them (and the referenced strings) to the
 * host, after which every host-side accessor / writer works on the result.  `dtext` must stay valid until then.
 * blu_result_device_text() is the text the references point into: `dtext` itself, or -- when the table's queries were not
 * contiguous (timings.n_regrouped) -- the regrouped copy the library made in device memory, owned by the result. */
int blu_consensus_run_device_resident(blu_ctx* ctx, const void* dtext, uint64_t n_bytes, void* stream, blu_result** out);
const void* blu_result_device_text(const blu_result* res, uint64_t* n_bytes);
const blu_record* blu_result_device_records(const blu_result* res);
const blu_bean* blu_result_device_beans(const blu_result* res, uint64_t* n);
const blu_acc* blu_result_device_accessions(const blu_result* res, uint64_t* n);
int blu_result_download(blu_result* res);
/* ParallelBlastOutput.output_file (parallel_blast_output.rs:3-7).  The file is streamed: parallel pread()s fill a ring of
 * three pinned staging buffers (opts.chunk_bytes each, default 64 MiB; BLU_READ_THREADS readers, default 8) while
 * earlier chunks are copied to the device and processed, so it never has to fit in host memory.  Only a table whose
 * queries are not contiguous is read whole (regrouping needs every row). */
int blu_consensus_run_file(blu_ctx* ctx, const char* blast_out_path, blu_result** out);
/* ParallelBlastOutput.headers: '\n'-separated query ids; ids without hits become NoConsensusFound
 * (mod.rs:84-102).  Call before serialising. */
int blu_result_add_headers(blu_result* res, const char* headers_nl, uint64_t len);

/* ---- several configurations in one pass ---------------------------------------------------------------------------
 * One pass over the table, one result per context: outs[k] is what blu_consensus_run_*(ctxs[k], ...) returns on its own --
 * the same blu_result_checksum, canonical JSONL, counts and writer bytes (record order is unspecified, as it is there).
 * The text is parsed once (and, from host memory or a file, copied to the device once); only the consensus and what
 * follows it runs per context.  outs[k] belongs to ctxs[k]: blu_result_sort_by_query(ctxs[k], outs[k]),
 * blu_result_download, blu_result_add_headers and the writers work on it as on any result.
 *   - 1 <= n_ctx <= 8.  n_ctx == 1 is blu_consensus_run_*(ctxs[0], ...) itself.
 *   - Otherwise all contexts are distinct single-device contexts of one device, each with a taxonomy loaded (the
 *     taxonomies may differ: a textLineage and a numericLineage context can be grouped), and opts.chunk_bytes and
 *     opts.flags are equal across the group.  Anything else returns BLU_ERR_ARG; the message names the context.
 *   - All or nothing: on an error no result is returned and every context of the group carries the message.  A
 *     grammar-class error of the table is the same for every configuration; a consensus-class one (e.g. an empty adjusted
 *     taxonomy, which depends on the cutoffs) fails the call with the error of the lowest-index context that has one, and
 *     the message starts with "ctxs[k]: ".  BLU_ERR_UNSUPPORTED limits are those of a single run.
 *   - A table whose queries are not contiguous is regrouped once, and every configuration runs over the regrouped text;
 *     the device-resident results share the regrouped copy (blu_result_device_text), which lives until the last of them
 *     is freed.
 *   - blu_ctx_last_timings of every context reports the shared pass: n_tile_launches, h2d_bytes and text_bytes are those
 *     of one single-context run, n_kernel_launches counts every launch of the pass, d2h_bytes everything the pass
 *     downloaded; result_bytes and taxonomy_bytes are the context's own. */
int blu_consensus_run_host_configs(blu_ctx* const* ctxs, int n_ctx, const char* text, uint64_t n_bytes, blu_result** outs);
int blu_consensus_run_file_configs(blu_ctx* const* ctxs, int n_ctx, const char* path, blu_result** outs);
int blu_consensus_run_device_resident_configs(blu_ctx* const* ctxs, int n_ctx, const void* dtext, uint64_t n_bytes, void* stream,
                                              blu_result** outs);

/* ---- results -------------------------------------------------------------------------------------------- */
uint64_t blu_result_num_queries(const blu_result* res);
/* Records with hits only (blu_result_num_queries also counts hit-less headers). */
uint64_t blu_result_num_records(const blu_result* res);
/* Orders the records of `res` by query id, bytewise -- the order write_blutils_output writes them in
 * (write_blutils_output.rs:111) -- on the GPU of `ctx` (its first device for a multi-device context).
 * Device-resident result (not yet downloaded): sorted in device memory; `ctx` must be the context that produced it
 * (else BLU_ERR_ARG); blu_result_device_records() may return a new pointer afterwards.
 * Host result: its query ids are copied to the device and sorted there, and its records are permuted on the host.  The
 * parts of a multi-device result are concatenated first; the result is one part afterwards.
 * Only records move: beans and accession references stay where they are, and each record still points at its own.
 * Hit-less headers (blu_result_add_headers) are not records and are not touched, before or after this call.
 * Order afterwards = std::stable_sort of the records by their id bytes (unsigned), applied to the order before the call.
 * The checksum, every count and every writer's output are the same before and after; the writers then only merge the
 * hit-less headers in instead of sorting every entry.  0 records: nothing to do.  Ids plus the sort's scratch that do not
 * fit the device: BLU_ERR_UNSUPPORTED. */
int blu_result_sort_by_query(blu_ctx* ctx, blu_result* res);
uint64_t blu_result_num_rows(const blu_result* res);
/* Host arrays of the result (the parts of a multi-device result are concatenated on the first call; the string
 * references of such a result are relative to blu_result_pool of that same concatenation). */
const blu_record* blu_result_records(const blu_result* res);
const blu_bean* blu_result_beans(const blu_result* res);
const blu_acc* blu_result_accessions(const blu_result* res);
const char* blu_result_pool(const blu_result* res, uint64_t* len);
uint64_t blu_result_num_beans(const blu_result* res);
uint64_t blu_result_num_accessions(const blu_result* res);
/* Order-independent 64-bit checksum of the canonical (runId-less) JSONL lines: sum of FNV-1a per line. */
uint64_t blu_result_checksum(const blu_result* res);
/* Canonical JSONL (one `{"query":..,"taxon":..}` object per line, sorted by query, no runId); caller frees
 * with blu_free. */
int blu_result_to_jsonl(const blu_result* res, char** out, uint64_t* len);
/* The first `max_entries` lines of the same (the entries with the smallest query ids): a check of a prefix of a large result
 * need not format all of it. */
int blu_result_to_jsonl_head(const blu_result* res, uint64_t max_entries, char** out, uint64_t* len);
/* write_blutils_output (write_blutils_output.rs:33-250): path NULL -> stdout; run_id NULL -> fresh UUIDv4;
 * config is always `null` on this path (ports/cli/src/cmds/blast/mod.rs:139). */
int blu_result_write(const blu_result* res, const char* path, int format, const char* run_id);
/* parse_consensus_as_tabular (parse_consensus_as_tabular/mod.rs:15-173) straight from the binary records: the
 * 12-column TSV of `blu blastn build-tabular` (one `consensus` row + one `blast-match` row per bean); path NULL ->
 * stdout, else the extension is forced to `.tsv`.  Reproduces the reference byte for byte, including its quirk of
 * not writing line breaks between pieces in file mode. */
int blu_result_write_tabular(const blu_result* res, const char* path, const char* run_id);
/* `blu blastn build-tabular` proper (parse_consensus_as_tabular/mod.rs:15-173 + file_or_stdin.rs:96-176): reads a blutils
 * result file (BLU_FORMAT_JSON, BLU_FORMAT_JSONL or BLU_FORMAT_YAML; path NULL or "-" = stdin) and writes the same TSV (output_file NULL =
 * stdout, else extension forced to `.tsv`).  Needs no context and no GPU.  `run_id` is used where neither the result nor
 * the config carries one (NULL = a fresh UUIDv4, as the reference).  BLU_ERR_IO with the message in `err` mirrors the
 * reference's Err(MappedErrors); YAML input is read in the block style
 * the writer produces (comments, any quoting, either sequence indentation); other YAML constructs return BLU_ERR_UNSUPPORTED. */
int blu_result_file_to_tabular(const char* blu_result_path, const char* output_file, int input_format, const char* run_id, char* err,
                               size_t errlen);
void blu_result_free(blu_result* res);
void blu_free(void* p);

int blu_ctx_last_timings(const blu_ctx* ctx, blu_timings* out);
/* Measured pinned host->device copy bandwidth (GB/s) on ctx's device, for the end-to-end ceiling: sustained over ~6 GB of
 * back-to-back copies of `bytes` each (call it on every GPU at once to see what the box gives them together). */
int blu_ctx_measure_h2d(blu_ctx* ctx, uint64_t bytes, double* gbps);
/* ... and device->host. */
int blu_ctx_measure_d2h(blu_ctx* ctx, uint64_t bytes, double* gbps);

/* Multi-GPU sharding (SURVEY 8e): byte offsets cuts[0..n_shards] that split the table into n_shards ranges of
 * roughly equal size without ever splitting a query (cuts move forward to the next query boundary).  Valid for
 * contiguous tables (every query's rows adjacent), which is what BLAST and blutils' chunked appends
 * (run_parallel_blast.rs:97,146-151) produce.  Host-only; needs no GPU. */
int blu_shard_cuts(const char* text, uint64_t n_bytes, int n_shards, uint64_t* cuts);
/* The same for a file (what blu_consensus_run_file does on a multi-device context): only a few rows around every cut are
 * read.  BLU_ERR_IO if the file cannot be opened / read. */
int blu_shard_cuts_file(const char* path, int n_shards, uint64_t* cuts);

/* Pinned host buffers (cudaHostAlloc) so callers can stage text for blu_consensus_run_host. */
void* blu_host_alloc(uint64_t bytes);
void blu_host_free(void* p);

int blu_abi_version(void);

#ifdef __cplusplus
}
#endif
#endif /* BLU_CONSENSUS_H */
