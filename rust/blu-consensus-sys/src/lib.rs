//! Raw bindings to `include/blu_consensus.h` plus the safe wrapper that keeps the reference signature of
//! `build_consensus_identities` (blutils-core, core/src/use_cases/build_consensus_identities/mod.rs:40-47).
//! SOURCE ONLY: not compiled in the build image (no cargo/rustc there).
#![allow(non_camel_case_types)]
use libc::{c_char, c_int, c_void, size_t};
use std::{ffi::{CStr, CString}, path::Path, ptr};

pub const BLU_OK: c_int = 0;
pub const BLU_ERR_IO: c_int = 1;
pub const BLU_ERR_DATA: c_int = 2;
pub const BLU_CUTOFF_ABSENT: i32 = i32::MIN;

#[repr(C)]
#[derive(Clone, Copy, Default)]
pub struct blu_opts {
    pub device: i32,
    pub taxon: i32,      // 0 fungi, 1 bacteria, 2 eukaryotes, 3 custom   (Taxon, taxon.rs:68-88)
    pub strategy: i32,   // 0 cautious, 1 relaxed                          (ConsensusStrategy)
    pub use_taxid: i32,
    pub has_custom: i32,
    pub custom: [i32; 8], // domain..species (CustomTaxon, taxon.rs:14-25)
    pub chunk_bytes: u64,
    pub flags: u64,       // BLU_OPT_*
    pub reserved: [u64; 3],
}
pub enum blu_ctx {}
pub enum blu_result {}

extern "C" {
    pub fn blu_abi_version() -> c_int;
    pub fn blu_ctx_create(opts: *const blu_opts, out: *mut *mut blu_ctx) -> c_int;
    pub fn blu_ctx_create_multi(opts: *const blu_opts, devices: *const c_int, n_devices: c_int, out: *mut *mut blu_ctx) -> c_int;
    pub fn blu_ctx_destroy(ctx: *mut blu_ctx);
    pub fn blu_last_error(ctx: *const blu_ctx) -> *const c_char;
    pub fn blu_custom_cutoffs_from_file(path: *const c_char, opts: *mut blu_opts, err: *mut c_char, errlen: size_t) -> c_int;
    pub fn blu_taxonomy_load_json(ctx: *mut blu_ctx, path: *const c_char) -> c_int;
    pub fn blu_taxonomy_load_json_cached(ctx: *mut blu_ctx, path: *const c_char, cache_path: *const c_char, cache_state: *mut c_int) -> c_int;
    pub fn blu_consensus_run_file(ctx: *mut blu_ctx, blast_out: *const c_char, out: *mut *mut blu_result) -> c_int;
    pub fn blu_consensus_run_host(ctx: *mut blu_ctx, text: *const c_char, n: u64, out: *mut *mut blu_result) -> c_int;
    pub fn blu_consensus_run_host_configs(ctxs: *const *mut blu_ctx, n_ctx: c_int, text: *const c_char, n: u64, outs: *mut *mut blu_result) -> c_int;
    pub fn blu_consensus_run_file_configs(ctxs: *const *mut blu_ctx, n_ctx: c_int, blast_out: *const c_char, outs: *mut *mut blu_result) -> c_int;
    pub fn blu_consensus_run_device_resident_configs(ctxs: *const *mut blu_ctx, n_ctx: c_int, dtext: *const c_void, n: u64, stream: *mut c_void,
                                                     outs: *mut *mut blu_result) -> c_int;
    pub fn blu_result_add_headers(res: *mut blu_result, headers_nl: *const c_char, len: u64) -> c_int;
    pub fn blu_result_num_queries(res: *const blu_result) -> u64;
    pub fn blu_result_num_records(res: *const blu_result) -> u64;
    pub fn blu_result_sort_by_query(ctx: *mut blu_ctx, res: *mut blu_result) -> c_int;
    pub fn blu_result_to_jsonl(res: *const blu_result, out: *mut *mut c_char, len: *mut u64) -> c_int;
    pub fn blu_result_write(res: *const blu_result, path: *const c_char, format: c_int, run_id: *const c_char) -> c_int;
    pub fn blu_result_file_to_tabular(blu_result_path: *const c_char, output_file: *const c_char, input_format: c_int, run_id: *const c_char, err: *mut c_char, errlen: size_t) -> c_int;
    pub fn blu_result_free(res: *mut blu_result);
    pub fn blu_free(p: *mut c_void);
}

/// Mirrors of the reference's by-value arguments (the real crate re-uses blul_core's own types).
#[derive(Clone, Copy)] pub enum Taxon { Fungi = 0, Bacteria = 1, Eukaryotes = 2, Custom = 3 }
#[derive(Clone, Copy)] pub enum ConsensusStrategy { Cautious = 0, Relaxed = 1 }
pub struct CustomTaxon { pub values: [Option<i16>; 8] }
pub struct ParallelBlastOutput { pub output_file: std::path::PathBuf, pub headers: Option<Vec<String>> }

#[derive(Debug)]
pub enum ConsensusError { Mapped(String) /* Err(MappedErrors) */, Panic(String) /* the reference panics */ }

/// Owns the binary result; `jsonl()` yields one `{"query":..,"taxon":..}` object per query (sorted by query), which
/// deserialises into blul_core's `QueryWithConsensus` with serde (`taxon: null` = `NoConsensusFound`).
pub struct ConsensusOutput { res: *mut blu_result, ctx: *mut blu_ctx }
impl ConsensusOutput {
    pub fn len(&self) -> usize { unsafe { blu_result_num_queries(self.res) as usize } }
    pub fn jsonl(&self) -> String {
        let (mut p, mut n) = (ptr::null_mut(), 0u64);
        unsafe {
            assert_eq!(blu_result_to_jsonl(self.res, &mut p, &mut n), BLU_OK);
            let s = String::from_utf8_lossy(std::slice::from_raw_parts(p as *const u8, n as usize)).into_owned();
            blu_free(p as *mut c_void);
            s
        }
    }
    /// write_blutils_output (write_blutils_output.rs:33-38): format 0 json, 1 jsonl, 2 yaml; None = stdout
    pub fn write(&self, out_file: Option<&str>, format: i32) -> Result<(), ConsensusError> {
        let c = out_file.map(|s| CString::new(s).unwrap());
        let rc = unsafe { blu_result_write(self.res, c.as_ref().map_or(ptr::null(), |c| c.as_ptr()), format, ptr::null()) };
        if rc == BLU_OK { Ok(()) } else { Err(ConsensusError::Mapped("could not write output".into())) }
    }
}
impl Drop for ConsensusOutput { fn drop(&mut self) { unsafe { blu_result_free(self.res); blu_ctx_destroy(self.ctx); } } }

fn err_of(ctx: *const blu_ctx, rc: c_int) -> ConsensusError {
    let msg = unsafe { CStr::from_ptr(blu_last_error(ctx)).to_string_lossy().into_owned() };
    if rc == BLU_ERR_IO { ConsensusError::Mapped(msg) } else { ConsensusError::Panic(msg) }
}

/// The reference entry point's signature, `Result<Vec<ConsensusResult>, MappedErrors>` included (mod.rs:40-47), without this
/// crate depending on blul_core (which would be circular): the caller passes how one result object is decoded (serde, from
/// the same JSON shape `QueryWithConsensus` serialises to; `taxon: null` = `NoConsensusFound`) and how an I/O-class failure
/// becomes its error type.  Data-class failures panic, as the reference does (mod.rs:123).
///
/// ```ignore
/// // blul_core::use_cases::build_consensus_identities, feature "b200"
/// blu_consensus_sys::build_consensus_identities_as(blast_output.into(), taxonomies_file, taxon.into(), strategy.into(), use_taxid,
///     custom_taxon_values.map(Into::into),
///     |line| { let q: QueryWithConsensus = serde_json::from_str(line).unwrap();
///              match q.taxon { Some(_) => ConsensusResult::ConsensusFound(q),
///                              None => ConsensusResult::NoConsensusFound(QueryWithoutConsensus { query: q.query }) } },
///     |msg| execution_err(msg))
/// ```
pub fn build_consensus_identities_as<R, E>(
    blast_output: ParallelBlastOutput, taxonomies_file: &Path, taxon: Taxon, strategy: ConsensusStrategy,
    use_taxid: Option<bool>, custom_taxon_values: Option<CustomTaxon>, decode: impl Fn(&str) -> R, io_err: impl Fn(String) -> E,
) -> Result<Vec<R>, E> {
    match build_consensus_identities(blast_output, taxonomies_file, taxon, strategy, use_taxid, custom_taxon_values) {
        Ok(out) => Ok(out.jsonl().lines().map(|l| decode(l)).collect()),
        Err(ConsensusError::Mapped(m)) => Err(io_err(m)),
        Err(ConsensusError::Panic(m)) => panic!("Unexpected error on parse blast results: {m}"),
    }
}

/// The GPUs the table is sharded over: `BLU_DEVICES=0,1,2,3` (one result either way); unset = device 0.
fn devices_from_env() -> Vec<c_int> {
    std::env::var("BLU_DEVICES").ok().map(|v| v.split(',').filter_map(|t| t.trim().parse().ok()).collect()).unwrap_or_default()
}

/// Same arguments as the reference entry point (mod.rs:40-47); returns the binary result container.
pub fn build_consensus_identities(
    blast_output: ParallelBlastOutput, taxonomies_file: &Path, taxon: Taxon, strategy: ConsensusStrategy,
    use_taxid: Option<bool>, custom_taxon_values: Option<CustomTaxon>,
) -> Result<ConsensusOutput, ConsensusError> {
    let mut o = blu_opts { taxon: taxon as i32, strategy: strategy as i32, use_taxid: use_taxid.unwrap_or(false) as i32, ..Default::default() };
    if let Some(c) = custom_taxon_values {
        o.has_custom = 1;
        for i in 0..8 { o.custom[i] = c.values[i].map_or(BLU_CUTOFF_ABSENT, |v| v as i32); }
    }
    unsafe {
        let mut ctx = ptr::null_mut();
        let devs = devices_from_env();
        let rc = if devs.len() > 1 { blu_ctx_create_multi(&o, devs.as_ptr(), devs.len() as c_int, &mut ctx) } else {
            if let Some(d) = devs.first() { o.device = *d; }
            blu_ctx_create(&o, &mut ctx)
        };
        if rc != BLU_OK { return Err(err_of(ptr::null(), rc)); }
        let tax = CString::new(taxonomies_file.to_str().unwrap()).unwrap();
        let rc = blu_taxonomy_load_json(ctx, tax.as_ptr());
        if rc != BLU_OK { let e = err_of(ctx, rc); blu_ctx_destroy(ctx); return Err(e); }
        let path = CString::new(blast_output.output_file.to_str().unwrap()).unwrap();
        let mut res = ptr::null_mut();
        let rc = blu_consensus_run_file(ctx, path.as_ptr(), &mut res);
        if rc != BLU_OK { let e = err_of(ctx, rc); blu_ctx_destroy(ctx); return Err(e); }
        if let Some(h) = blast_output.headers {
            let joined = h.join("\n");
            blu_result_add_headers(res, joined.as_ptr() as *const c_char, joined.len() as u64);
        }
        Ok(ConsensusOutput { res, ctx })
    }
}
