// blu_kernels.h -- launch interface between the host runtime (blu_api.cpp) and the sm_100a kernels.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "blu_core.cuh"

namespace blu {

// Device-side counters of one run (zeroed by the host before the first chunk).  Every cursor is its own 64-bit word:
// a reservation that overflows its capacity can never carry into a neighbouring count.
struct Counters {
    unsigned long long rec_count;   // record headers reserved by the tile / long-run kernels (dense)
    unsigned long long slot_count;  // top-row slots reserved (CTA slabs: holes are allowed, the array is never downloaded)
    unsigned long long bean_used;   // compact output cursors of the post-pass: beans, accession references, string pool
    unsigned long long acc_used;
    unsigned long long pool_used;
    unsigned long long post_done;   // records [0, post_done) have been through the post-pass (consensus / gather)
    unsigned long long next_begin;  // resident tables processed in ranges: where the next range starts
    unsigned long long err_off;     // byte offset (in the current device buffer) of the first fatal error
    unsigned long long soft_off;    // ... of the first consensus-class error
    unsigned long long tail_start;  // !final chunks: start of the last (unfinished) run
    unsigned long long n_rows;      // hit rows of the finished queries
    unsigned int n_defer;       // deferred runs of the current chunk
    unsigned int work_ticket;   // dynamic work distribution of the long-run kernel
    unsigned int err_code;      // first grammar-class DevErr: the reference fails on such a row wherever it sits
    unsigned int soft_code;     // first consensus-class DevErr (join / lineage / root disagreement / empty adjusted taxonomy):
                                // fatal only once the table is known to be contiguous -- a fragment of a scattered query may
                                // hit it although the merged query would not (the reference only parses the top group's rows)
    unsigned int dup_found;     // a query id occurs in two separate runs
    unsigned int cap_overflow;  // some output capacity was exceeded (host grows and retries)
    unsigned int pad0;
    unsigned int pad;
};

constexpr uint64_t kBeginFromCounters = ~0ull;  // RunParams.begin: take the start of the range from Counters.next_begin

struct RunParams {
    const uint8_t* text;   // device buffer (16-byte aligned, padded to a multiple of 128 bytes)
    uint64_t begin, end;   // valid text is [begin, end)
    int final_chunk;       // 1: `end` is the end of the input; 0: the run touching `end` is carried over
    int strategy;
    LinTables T;
    blu_record* records;
    uint64_t rec_cap;
    TopRowRaw* toprows;    // top bit-score rows of every query (fields 1..4 folded to integers, or unparsed references;
                           // lineage not joined yet), slot-indexed
    uint64_t slot_cap;
    blu_bean* beans;       // compact outputs (the long-run kernel finishes its queries itself)
    uint64_t bean_cap;
    blu_acc* accs;
    uint64_t acc_cap;
    uint64_t* defer;       // (offset << 1) | check_prev
    uint32_t defer_cap;
    TopRow* big_rows;      // scratch of the long-run kernel: kLongTopCap joined top rows per CTA
    unsigned long long* big_cand;  // ... and as many candidate references (offset << 16 | length)
    Counters* ctr;
};

// Post-pass over the records the tile kernel produced since the last post-pass: [ctr->post_done, ctr->rec_count).
struct PostParams {
    blu_record* records;
    uint64_t rec_cap;
    const TopRowRaw* toprows;
    uint64_t slot_cap;
    blu_bean* beans;
    uint64_t bean_cap;
    blu_acc* accs;
    uint64_t acc_cap;
    const uint8_t* text;
    uint64_t text_end;     // valid text is [0, text_end) of `text` (references beyond it are an internal error)
    uint8_t* pool;         // string pool (gather kernel); nullptr: strings stay references into `text`
    uint64_t pool_cap;
    LinTables T;
    int strategy;
    Counters* ctr;
};

// Duplicate-id check of the records produced since the last post-pass, [ctr->post_done, ctr->rec_count): their 64-bit id
// hashes go into one open-addressing table that lives for the whole run.  The same pass relocates string references
// that have to leave the device as offsets into the caller's host text (ref_delta != 0).
struct DupParams {
    blu_record* records;
    uint64_t rec_cap;
    const blu_bean* beans;
    blu_acc* accs;
    const uint8_t* strings;     // what blu_record.query_off refers to: the string pool, or the text when nothing was gathered
    uint64_t strings_len;
    unsigned long long* table;  // open addressing, 0 = empty; nullptr: no check, only the relocation below (the other
                                // configurations of a pass: their ids are the first configuration's)
    uint32_t mask;
    unsigned long long* hashes; // optional: the 64-bit id hash of every record (multi-device runs merge them), or nullptr
    long long ref_delta;        // added to every string offset after hashing (device-buffer -> caller's text coordinates)
    Counters* ctr;
};

// Configurations of one pass over a table (blu_consensus_run_*_configs): the tile kernel runs once, into the first one's
// records and counters; everything after it runs once per configuration.
constexpr int kMaxConfigs = 8;

// Behind the tile kernel of a pass with several configurations: the record headers it wrote, [src->post_done,
// src->rec_count), and the cursors that depend on the text only (record / slot / deferred-run counts, the open tail, the
// first grammar error, a capacity overflow) are copied from the first configuration to the others.  Every configuration
// of a pass has the same record capacity, so the headers keep their indices.
struct FanoutParams {
    const Counters* src;
    const blu_record* src_records;
    Counters* dst[kMaxConfigs - 1];
    blu_record* dst_records[kMaxConfigs - 1];
    int n_dst;
    uint64_t rec_cap;
};

// End of a range / chunk: post_done <- rec_count, the per-range counters are reset (next_begin <- tail_start or range_end)
// and the counters are copied to `snapshot` (mapped pinned host memory or device memory; may be nullptr).
struct AdvanceParams {
    Counters* ctr;
    uint64_t rec_cap;
    uint64_t range_end;
    Counters* snapshot;
};

// Geometry of the streaming tile kernel (see DESIGN.md): every CTA walks one contiguous segment of the text in
// kTile-byte steps (double-buffered TMA), carrying the unfinished query from one step to the next.
#ifndef BLU_TILE_BYTES
#define BLU_TILE_BYTES 32768
#endif
#ifndef BLU_TILE_CTAS
#define BLU_TILE_CTAS 2
#endif
#ifndef BLU_TILE_THREADS
#define BLU_TILE_THREADS 512
#endif
constexpr int kTile = BLU_TILE_BYTES;   // bytes staged per step
constexpr int kBack = 1024;             // look-behind of a segment's first window (predecessor of its first row)
constexpr int kTileThreads = BLU_TILE_THREADS;
constexpr int kTileCtasPerSm = BLU_TILE_CTAS;
constexpr int kWin = 60416;             // window of the block path (long-run kernel)

int tile_kernel_grid(int device);
cudaError_t launch_tile_kernel(const RunParams& p, int grid, cudaStream_t s);
cudaError_t launch_longrun_kernel(const RunParams& p, int grid, cudaStream_t s);
cudaError_t launch_consensus_kernel(const PostParams& p, int sms, cudaStream_t s);
cudaError_t launch_gather_kernel(const PostParams& p, int sms, cudaStream_t s);
cudaError_t launch_dup_kernel(const DupParams& p, int sms, cudaStream_t s);
cudaError_t launch_fanout_kernel(const FanoutParams& p, int sms, cudaStream_t s);
cudaError_t launch_advance_kernel(const AdvanceParams& p, cudaStream_t s);
cudaError_t launch_dup_merge_kernel(const unsigned long long* hashes, unsigned long long n, unsigned long long* table, uint32_t mask,
                                    unsigned int* dup_found, int sms, cudaStream_t s);
constexpr int kLongTopCap = 8192;       // largest top bit-score group the block path handles (beyond: BLU_ERR_UNSUPPORTED)
cudaError_t kernels_set_attributes();

// blu_regroup.cu: rewrites a non-contiguous hit table (device memory) with every query's rows adjacent -- queries in order of
// first appearance, rows of a query in file order (the reference's HashMap grouping, mod.rs:145,192).  0: *d_out is the
// cudaMalloc'ed regrouped text (the caller frees it); 1: not possible on the device (memory, >= 2^31 rows, two ids with one
// hash): regroup on the host; < 0: -cudaError_t.
int regroup_device(const uint8_t* d_text, uint64_t n, cudaStream_t s, uint8_t** d_out, uint64_t* out_n, uint64_t* n_rows_out);

}  // namespace blu
